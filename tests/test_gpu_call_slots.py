"""GPU tests of the per-call lanes and result slots of a handle: calls of different kinds sharing one bank's three result
slots, the handle operations that must wait for outstanding calls, and the sharded-round phases that need an open round."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

D, FM = 768, 28
P = FM * FM


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import Bank, synth
    from cmdiad_b200 import _lib as L
    from cmdiad_b200.fusion import LateFusion
    assert torch.cuda.is_available()
    cent = synth.centroids(D, 128)
    return dict(Bank=Bank, LateFusion=LateFusion, L=L, synth=synth, cent=cent)


def _bank(env, rows):
    b = env["Bank"](D, rows.shape[0])
    b.append(rows)
    b.finalize()
    return b


def _batch(env, seed, n=3, p=P):
    sy = env["synth"]
    return np.stack([sy.patches(p, D, seed=seed + i, anomalous_frac=0.01, cent=env["cent"]) for i in range(n)])


def _fusion(env, banks):
    return env["LateFusion"](banks, [1.0, 0.5], [1.0, 2.0], [0.3, -0.2], 0.1, [0.5, 0.25], -0.05)


_FIELDS = ("min_idx", "min_val", "s", "s_star", "s_idx", "nn_idx", "m_star_knn", "w", "s_map")


def _same(a, b, tag):
    assert len(a) == len(b), tag
    for i in range(len(a)):
        for name in _FIELDS:
            assert (getattr(a[i], name) == getattr(b[i], name)).all(), (tag, i, name)


def _same_fused(a, b, tag):
    assert (a.s == b.s).all() and (a.s_map == b.s_map).all() and (a.s_modal == b.s_modal).all(), tag
    for m in range(len(a.min_val)):
        assert (a.min_val[m] == b.min_val[m]).all() and (a.min_idx[m] == b.min_idx[m]).all(), (tag, m)


def test_three_slots_of_one_bank_held_by_different_calls(env):
    """Two batches and one fused call (bank A is its modality 0) fill all three result slots of A; waited for in
    different orders they give the synchronous results, and a later call with another out_hw still does."""
    sy = env["synth"]
    A = _bank(env, sy.patches(8000, D, seed=11, cent=env["cent"]))
    Bm = _bank(env, sy.patches(5000, D, seed=12, cent=env["cent"]))
    fusion = _fusion(env, [A, Bm])
    x0, x1, xa = _batch(env, 100), _batch(env, 200), _batch(env, 300)
    xb = _batch(env, 400, p=196)
    dims = [(FM, FM), (14, 14)]
    ref112 = A.score_batch(x0, (FM, FM), 112, full=True)
    ref0, ref1 = A.score_batch(x0, (FM, FM), 224, full=True), A.score_batch(x1, (FM, FM), 224, full=True)
    ref_f = fusion.score_batch([xa, xb], dims, 224, want_patch=True)
    for order in ((2, 0, 1), (1, 2, 0), (0, 1, 2)):
        t = [A.score_batch_async(x0, (FM, FM), 224, full=True), A.score_batch_async(x1, (FM, FM), 224, full=True),
             fusion.score_batch_async([xa, xb], dims, 224, want_patch=True)]
        with pytest.raises(env["L"].CmdbError) as e:   # every slot of A is taken
            A.score_batch_async(x0, (FM, FM), 224)
        assert e.value.status == env["L"].CMDB_ERR_STATE
        got = {k: t[k].wait() for k in order}
        _same(ref0, got[0], f"batch 0, order {order}")
        _same(ref1, got[1], f"batch 1, order {order}")
        _same_fused(ref_f, got[2], f"fused, order {order}")
    _same(ref112, A.score_batch(x0, (FM, FM), 112, full=True), "out_hw 112 after the pipelined calls")
    A.close()
    Bm.close()


def test_bank_mutations_wait_for_outstanding_batches(env):
    """normalize, gather and finalize rewrite the rows or the scoring layout that an outstanding batch still reads: they
    are refused until the batch has been waited for, then they work and the bank scores like a fresh one."""
    sy = env["synth"]
    L = env["L"]
    rows = sy.patches(6000, D, seed=21, cent=env["cent"])
    A = _bank(env, rows)
    x = _batch(env, 500)
    ref = A.score_batch(x, (FM, FM), 224, full=True)
    t = A.score_batch_async(x, (FM, FM), 224, full=True)
    idx = np.arange(0, rows.shape[0], 2)
    for op in (lambda: A.normalize(0.5, 2.0), lambda: A.gather(idx), A.finalize):
        with pytest.raises(L.CmdbError) as e:
            op()
        assert e.value.status == L.CMDB_ERR_STATE
    _same(ref, t.wait(), "batch outstanding during the refused calls")
    A.normalize(0.5, 2.0)
    A.gather(idx)
    A.finalize()
    fresh = _bank(env, A.read().numpy())
    assert (A.read().numpy() == ((rows[idx] - np.float32(0.5)) / np.float32(2.0))).all()
    _same(fresh.score_batch(x, (FM, FM), 224, full=True), A.score_batch(x, (FM, FM), 224, full=True), "after the mutations")
    A.close()
    fresh.close()


def test_finalize_refused_during_a_fused_call(env):
    """The second modality of an outstanding fused batch cannot be finalized; the fused wait still returns the results."""
    sy = env["synth"]
    L = env["L"]
    A = _bank(env, sy.patches(6000, D, seed=31, cent=env["cent"]))
    Bm = _bank(env, sy.patches(4000, D, seed=32, cent=env["cent"]))
    fusion = _fusion(env, [A, Bm])
    xa, xb = _batch(env, 600), _batch(env, 700, p=196)
    dims = [(FM, FM), (14, 14)]
    ref = fusion.score_batch([xa, xb], dims, 224, want_patch=True)
    t = fusion.score_batch_async([xa, xb], dims, 224, want_patch=True)
    with pytest.raises(L.CmdbError) as e:
        Bm.finalize()
    assert e.value.status == L.CMDB_ERR_STATE
    _same_fused(ref, t.wait(), "fused wait after the refused finalize")
    Bm.finalize()
    _same_fused(ref, fusion.score_batch([xa, xb], dims, 224, want_patch=True), "after the finalize")
    A.close()
    Bm.close()


def test_shard_phases_need_an_open_round(env):
    """Once the finish call has closed a round, cmdb_score_shard_lookup and _finish_submit are refused until
    cmdb_score_shard_min opens the next one, even when given the buffers of the completed round; later rounds still work."""
    from cmdiad_b200.bank import Bank, _ptr
    sy = env["synth"]
    L = env["L"]
    lib = L.load()
    A = _bank(env, sy.patches(6000, D, seed=41, cent=env["cent"]))
    A.build_knn()
    h = A._h
    B = 2
    x = torch.from_numpy(_batch(env, 800, n=B))
    keys = torch.empty(B * P, dtype=torch.int64, device="cuda")
    d2 = torch.empty(B * 2, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    def refused():
        t = ctypes.c_int64()
        assert lib.cmdb_score_shard_lookup(h, _ptr(keys), B, P, _ptr(d2)) == L.CMDB_ERR_STATE
        assert lib.cmdb_score_shard_finish_submit(h, _ptr(d2), B, P, FM, FM, 224, 0, 1, 0, ctypes.byref(t)) == L.CMDB_ERR_STATE

    def one_round():   # one rank: the keys and distance sums need no collective between the phases
        L.check(lib.cmdb_score_shard_min(h, _ptr(x), B, P, 0, 224, _ptr(keys)))
        L.check(lib.cmdb_score_shard_lookup(h, _ptr(keys), B, P, _ptr(d2)))
        t = ctypes.c_int64()
        L.check(lib.cmdb_score_shard_finish_submit(h, _ptr(d2), B, P, FM, FM, 224, 0, 1, 0, ctypes.byref(t)))
        res, outs, _ = Bank._alloc_out(B, P, 224, False)
        L.check(lib.cmdb_score_shard_wait(h, t.value, outs))
        return res

    first = one_round()
    refused()
    _same(first, one_round(), "round after the refused phases")
    A.close()
