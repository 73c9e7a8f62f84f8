"""GPU tests of the host-side mirror classes (cmdiad_b200/methods.py) and of the sharded entry points with one rank."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import synth
    from oracle import restate as O
    assert torch.cuda.is_available()
    return dict(O=O, synth=synth)


def _train(env, n, P, D, seed):
    return env["synth"].image_bank(n, P, D, seed, k=64)


def test_rgb_features_fp16_pipeline_vs_oracle(env):
    """RGBFeatures (multiple_features.py:28-121) in the default FP16 coreset mode: device statistics, normalisation,
    projection drawn from numpy's global RNG (random_state=None + seed 0 in the ctor), greedy loop, scoring"""
    from cmdiad_b200 import RGBFeatures, default_args
    O = env["O"]
    train = _train(env, 4, 784, 768, 31)
    m = RGBFeatures(default_args(coreset_dtype="FP16", random_state=None), bank_capacity_rows=4 * 784)
    for x in train:
        m.add_sample_to_mem_bank({"rgb": x}, class_name="synthetic")
    m.run_coreset()
    cat = np.concatenate(train, 0)
    assert abs(float(m.rgb_mean) - cat.mean(dtype=np.float64)) < 1e-6 and abs(float(m.rgb_std) - cat.std(ddof=1, dtype=np.float64)) < 1e-5
    lib = ((torch.from_numpy(cat) - m.rgb_mean) / m.rgb_std).numpy()
    # the reference's transformer: random_state=None -> numpy global RNG, seeded 0 by the constructor (features.py:48)
    np.random.seed(0)
    csr = O.sparse_components(lib.shape[0], 768, 0.9, None)
    n = int(0.1 * lib.shape[0])
    ref_idx = O.coreset_restated(O.project_restated(lib, *csr), n, "FP16")
    assert (m.coreset_idx.numpy() == ref_idx).all()
    assert tuple(m.patch_rgb_lib.shape) == (n, 768) and (m.patch_rgb_lib[:].numpy() == lib[ref_idx]).all()
    for x in train:
        m.add_sample_to_late_fusion_mem_bank({"rgb": x})
    m.run_late_fusion()
    test = env["synth"].patches(784, 768, 999, anomalous_frac=0.02, k=64)
    m.predict({"rgb": test}, torch.zeros(1, 224, 224), 1, ["x.png"])
    patch = ((torch.from_numpy(test) - m.rgb_mean) / m.rgb_std).numpy()
    ref = O.score_restated(patch, lib[ref_idx], (28, 28), 224)
    # predict() runs the late-fusion head on the device: last_fused.s_modal = lambda * s per modality
    np.testing.assert_allclose(m.last_fused.s_modal[0, 0], np.float32(m.args.rgb_s_lambda) * ref["s"], rtol=1e-4)
    assert m.predictions[0].shape == (224, 224) and sum(len(a) for a in m.pixel_preds) == 224 * 224
    s_ref = m.detect_fuser.score_samples(np.array([[m.args.rgb_s_lambda * ref["s"]]]))
    np.testing.assert_allclose(m.image_preds[0], s_ref, rtol=1e-4)
    # persistence: a fresh object restored from disk predicts identically without re-running the coreset
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        m.save_state(tmp)
        m2 = RGBFeatures(default_args(coreset_dtype="FP16", random_state=None))
        m2.load_state(tmp)
        m2.predict({"rgb": test}, torch.zeros(1, 224, 224), 1, ["x.png"])
        assert (m2.image_preds[0] == m.image_preds[0]).all() and (m2.predictions[0] == m.predictions[0]).all()
        assert (m2.patch_rgb_lib[:] == m.patch_rgb_lib[:]).all() and float(m2.rgb_std) == float(m.rgb_std)
        m2.close()
    m.close()


@pytest.mark.parametrize("main", ["rgb", "xyz"])
def test_hallucination_class_wiring(env, main):
    """RGBorXYZWithOneHallucination (multiple_features.py:312-573): three banks filled, only main + fusion normalised,
    subsampled and scored; statistics cross-wired (mean of the xyz lib, std of the rgb lib)"""
    from cmdiad_b200 import RGBorXYZWithOneHallucination, default_args
    D = 768
    rgb = _train(env, 2, 196, D, 41)
    xyz = [x * 2 + 0.5 for x in _train(env, 2, 196, D, 42)]
    fus = _train(env, 2, 196, D, 43)
    m = RGBorXYZWithOneHallucination(default_args(coreset_dtype="TF32", random_state=0, main_modality=main, f_coreset=0.25),
                                     bank_capacity_rows=2 * 196)
    for r, x, f in zip(rgb, xyz, fus):
        m.add_sample_to_mem_bank({"rgb": r, "xyz": x, "fusion": f})
    m.run_coreset()
    xyz_cat, rgb_cat = np.concatenate(xyz, 0), np.concatenate(rgb, 0)
    for k in ("xyz", "rgb", "fusion"):
        assert abs(float(getattr(m, f"{k}_mean")) - xyz_cat.mean(dtype=np.float64)) < 1e-5
        assert abs(float(getattr(m, f"{k}_std")) - rgb_cat.std(ddof=1, dtype=np.float64)) < 1e-5
    other = "xyz" if main == "rgb" else "rgb"
    assert m._lib(main).shape[0] == 98 and m.patch_fusion_lib.shape[0] == 98
    assert m._lib(other).shape[0] == 392  # the non-main bank is neither normalised nor subsampled (:379-402)
    raw = (xyz_cat if other == "xyz" else rgb_cat)
    assert (m._lib(other)[:].numpy() == raw).all()
    m.add_sample_to_late_fusion_mem_bank({"rgb": rgb[0], "xyz": xyz[0], "fusion": fus[0]})
    m.add_sample_to_late_fusion_mem_bank({"rgb": rgb[1], "xyz": xyz[1], "fusion": fus[1]})
    assert m.s_lib[0].shape == (1, 2) and m.s_map_lib[0].shape == (224 * 224, 2)
    m.run_late_fusion()
    m.predict({"rgb": rgb[0], "xyz": xyz[0], "fusion": fus[0]}, torch.zeros(1, 224, 224), 0, ["y.png"])
    m.predict({"rgb": rgb[1] + 3, "xyz": xyz[1], "fusion": fus[1] + 3}, torch.ones(1, 224, 224), 1, ["z.png"])
    # batch forms give the per-image results of the one-by-one calls
    n_before = len(m.image_preds)
    samples = [{"rgb": rgb[0], "xyz": xyz[0], "fusion": fus[0]}, {"rgb": rgb[1] + 3, "xyz": xyz[1], "fusion": fus[1] + 3}]
    m.predict_batch(samples, [torch.zeros(1, 224, 224), torch.ones(1, 224, 224)], [0, 1], [["y.png"], ["z.png"]])
    for i in range(2):
        assert (m.image_preds[n_before + i] == m.image_preds[i]).all()
        assert (m.predictions[n_before + i] == m.predictions[i]).all()
    m.calculate_metrics()
    assert 0.0 <= m.image_rocauc <= 1.0 and 0.0 <= m.pixel_rocauc <= 1.0
    assert 0.0 <= m.au_pro <= 1.0 and 0.0 <= m.au_pro_001 <= 1.0 and m.pixel_preds.shape == m.pixel_labels.shape
    with pytest.raises(NotImplementedError):
        m.args.dist_method_s = "l1"
        m.calculate_dist(torch.zeros(2, 2), torch.zeros(2, 2))
    m.close()


def test_projection_error_branch_keeps_unprojected_bank(env, capsys):
    """features.py:364-370: when sklearn raises ValueError (d' > D) the reference prints and continues without
    the projection"""
    from cmdiad_b200 import PointFeatures, default_args
    O = env["O"]
    D = 128
    xyz = _train(env, 2, 400, D, 51)
    m = PointFeatures(default_args(coreset_dtype="TF32", random_state=0, f_coreset=0.1), bank_capacity_rows=800)
    for x in xyz:
        m.add_sample_to_mem_bank({"xyz": x})
    m.run_coreset()
    assert "could not project" in capsys.readouterr().out
    cat = np.concatenate(xyz, 0)
    lib = ((torch.from_numpy(cat) - m.xyz_mean) / m.xyz_std).numpy()
    assert (m.coreset_idx.numpy() == O.coreset_restated(lib.astype(np.float64), 80, "TF32")).all()
    m.close()


def test_sharded_entry_points_with_one_rank(env):
    """the sharded scoring and the sharded coreset entry points on a 1-rank NCCL group must reproduce the plain
    single-GPU calls (several shards of one round: tests/test_gpu_shards.py on one GPU, scripts/shard_check.py and
    scripts/coreset_shard_check.py under torchrun, tests/test_sharding_gloo.py on the host side)"""
    import torch.distributed as dist
    from cmdiad_b200 import Bank, Comm
    O = env["O"]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        lib = env["synth"].patches(4000, 768, 61, k=64)
        b = Bank(768, 4000)
        b.append(lib)
        csr = O.sparse_components(4000, 768, 0.9, 0)
        comm = Comm(0, d_proj_max=512)
        assert (b.coreset_select_sharded(comm, 4000, 300, csr) == b.coreset_select(300, csr)).all()
        comm.close()
        b.finalize()
        patches = np.stack([env["synth"].patches(784, 768, 70 + i, anomalous_frac=0.01, k=64) for i in range(3)])
        # no neighbour table yet: score_batch sweeps the bank, and the first sharded call builds the replicated table
        c = b.score_batch(patches, (28, 28), 224, full=True)
        a = b.score_sharded_batch(patches, (28, 28), 224, full=True)
        for i in range(3):
            for name in ("s", "s_idx", "min_val", "min_idx", "nn_idx", "m_star_knn", "w", "s_map"):
                assert (getattr(a[i], name) == getattr(c[i], name)).all(), (i, name)
        # finalize frees the table: the next sharded call has to build it again
        b.finalize()
        c = b.score_batch(patches, (28, 28), 224, full=True)
        a = b.score_sharded_batch(patches, (28, 28), 224, full=True)
        for i in range(3):
            for name in ("s", "s_idx", "min_val", "min_idx", "nn_idx", "m_star_knn", "w", "s_map"):
                assert (getattr(a[i], name) == getattr(c[i], name)).all(), (i, name)
        # explicit build + pipelined rounds (three phases, two collectives per round); 40 images = 2 rounds
        b.build_knn_sharded()
        many = np.stack([env["synth"].patches(784, 768, 170 + i, anomalous_frac=0.01, k=64) for i in range(40)])
        a = b.score_sharded_batch(many, (28, 28), 224, full=True)
        c = b.score_batch(many, (28, 28), 224, full=True)
        d = b.score_sharded_batch(torch.from_numpy(many).cuda(), (28, 28), 224, full=True, distribute=True)
        for i in range(40):
            for name in ("s", "s_idx", "min_val", "min_idx", "nn_idx", "m_star_knn", "w", "s_map", "s_map_pre"):
                assert (getattr(a[i], name) == getattr(c[i], name)).all(), (i, name)
                assert (getattr(d[i], name) == getattr(c[i], name)).all(), (i, name)
        # the same rounds with the exchanges over peer-mapped memory instead of NCCL (cmdb_score_shard_round_submit)
        comm2 = Comm(0)
        b.attach_comm(comm2)
        e = b.score_sharded_batch(many, (28, 28), 224, full=True, distribute=True)
        for i in range(40):
            for name in ("s", "s_idx", "min_val", "min_idx", "nn_idx", "m_star_knn", "w", "s_map", "s_map_pre"):
                assert (getattr(e[i], name) == getattr(c[i], name)).all(), (i, name)
        b.attach_comm(None)
        comm2.close()
        b.close()
    finally:
        dist.destroy_process_group()
