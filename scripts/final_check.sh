#!/bin/bash
# verification on one B200: GPU tests, smoke, bench (both arms); logs and bench lines go to $O
set -u
O=gpurun_out
python -m pytest tests -m gpu -x -q > $O/final_pytest.log 2>&1; echo "pytest rc=$?" | tee -a $O/final_pytest.log
python __graft_entry__.py smoke > $O/final_smoke.log 2>&1; echo "smoke rc=$?" | tee -a $O/final_smoke.log
python bench.py --impl reference > $O/final_ref.json 2> $O/final_ref.err; echo "reference arm rc=$?"
python bench.py > $O/final_n1.json 2> $O/final_n1.err; echo "bench rc=$?"
