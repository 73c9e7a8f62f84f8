"""GPU tests of row-sharded scoring with several shards on one GPU.

Row-offset handles on one device play the ranks of one round, all in one process.  The helper below drives the three
phases of the NCCL protocol (include/cmdiad_b200.h) through the C API and stands in for the collectives with torch:
the MIN all-reduce of the packed keys is torch.stack(keys).amin(0), the SUM all-reduce of the neighbour distances is
torch.stack(contribs).sum(0) (one owner contributes x, the others 0: exact in any order).  Every round must equal
cmdb_score_batch on the un-sharded bank bit for bit, in every field, and the un-sharded result must equal the exact
float32 scan of the whole bank (cmdb_debug_exact_min)."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

PER_IMAGE = ("min_idx", "min_val", "s", "s_star", "s_idx", "nn_idx", "m_star_knn", "w")
MAPS = ("s_map", "s_map_pre", "s_map_u8")
SENTINEL = 0x5A   # byte pattern of the map buffers a distributed finish must leave untouched
MODES = ("certified", "simt")


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import Bank, sharding, synth
    from cmdiad_b200 import _lib as L
    from cmdiad_b200.bank import _ptr
    assert torch.cuda.is_available()
    return SimpleNamespace(Bank=Bank, sharding=sharding, synth=synth, L=L, lib=L.load(), ptr=_ptr)


def _bank(env, rows, lo=0):
    b = env.Bank(rows.shape[1], rows.shape[0], row_offset=lo)
    b.append(rows)
    b.finalize()
    return b


def _set_mode(env, banks, mode):
    for b in banks:
        b.set_score_impl(env.L.SCORE_SIMT if mode == "simt" else env.L.SCORE_TCGEN05)


class Sharded:
    """an un-sharded handle with its neighbour table, and k row-offset handles (sharding.shard_range) holding the same
    rows with the replicated table installed"""

    def __init__(self, env, lib, k, full=None):
        self.R, self.k = lib.shape[0], k
        self.full = full
        if self.full is None:
            self.full = _bank(env, lib)
            self.full.build_knn()
        self.table = self.full.read_knn(0, self.R)
        self.ranges = [env.sharding.shard_range(self.R, r, k) for r in range(k)]
        self.shards = []
        for lo, hi in self.ranges:
            b = _bank(env, lib[lo:hi], lo)
            b.set_knn_table(self.table, self.R)
            self.shards.append(b)

    def layout(self):
        return f"R={self.R} in {self.k} shards " + " ".join(f"[{lo},{hi})" for lo, hi in self.ranges)

    def set_mode(self, env, mode):
        _set_mode(env, [self.full] + self.shards, mode)

    def close(self, full=True):
        for b in self.shards + ([self.full] if full else []):
            b.close()


def _report(capsys, line):
    with capsys.disabled():
        print(f"\n    {line}", end="")


def _submit(env, shards, x, dims, out_hw, distribute=False):
    """one round on every shard: the three phases with torch in place of the collectives.  Returns the tickets, the
    per-shard contributions of the lookup and the tensors the round reads until it is waited for."""
    L, lib, ptr = env.L, env.lib, env.ptr
    if not isinstance(x, torch.Tensor):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    B, P = x.shape[0], x.shape[1]
    fh, fw = dims
    k = len(shards)
    keys = [torch.empty(B * P, dtype=torch.int64, device="cuda") for _ in shards]
    torch.cuda.synchronize()
    for b, kk in zip(shards, keys):
        L.check(lib.cmdb_score_shard_min(b._h, ptr(x), B, P, int(x.is_cuda), int(out_hw), ptr(kk)))
    torch.cuda.synchronize()
    red = torch.stack(keys).amin(0)
    contribs = [torch.empty(B * 2, dtype=torch.float32, device="cuda") for _ in shards]
    torch.cuda.synchronize()
    for b, c in zip(shards, contribs):
        L.check(lib.cmdb_score_shard_lookup(b._h, ptr(red), B, P, ptr(c)))
    torch.cuda.synchronize()
    total = torch.stack(contribs).sum(0)
    torch.cuda.synchronize()
    tickets = []
    for r, b in enumerate(shards):
        first, step = (r, k) if distribute else (0, 1)
        t = ctypes.c_int64()
        L.check(lib.cmdb_score_shard_finish_submit(b._h, ptr(total), B, P, int(fh), int(fw), int(out_hw), first, step, 3,
                                                   ctypes.byref(t)))
        tickets.append(t.value)
    return SimpleNamespace(tickets=tickets, contribs=[c.cpu().numpy() for c in contribs], B=B, P=P, out_hw=out_hw,
                           keep=(x, keys, red, contribs, total))


def _wait(env, bank, ticket, B, P, out_hw):
    _, outs, arr = env.Bank._alloc_out(B, P, out_hw, True)
    for name in MAPS:
        arr[name].view(np.uint8)[...] = SENTINEL
    env.L.check(env.lib.cmdb_score_shard_wait(bank._h, ticket, outs))
    return arr


def _round(env, sh, x, dims, out_hw, distribute=False):
    rd = _submit(env, sh.shards, x, dims, out_hw, distribute)
    return [_wait(env, b, t, rd.B, rd.P, out_hw) for b, t in zip(sh.shards, rd.tickets)], rd


def _exact_min(b, q):
    q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, b.dim)
    v, i = np.empty(q.shape[0], np.float32), np.empty(q.shape[0], np.int64)
    assert b._lib.cmdb_debug_exact_min(b._h, q.ctypes.data, q.shape[0], v.ctypes.data, i.ctypes.data) == 0
    return v, i


def _host(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _reference(full, x, dims, out_hw, exact_q=None):
    """the un-sharded handle's score_batch, checked against the exact scan of the whole bank"""
    want = full.score_batch(x, dims, out_hw, full=True).arrays
    v, i = _exact_min(full, _host(x) if exact_q is None else exact_q)
    _same({"min_val": v, "min_idx": i}, {"min_val": want["min_val"].ravel(), "min_idx": want["min_idx"].ravel()},
          ("min_idx", "min_val"), slice(None), "un-sharded result vs exact scan")
    return want


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int32) if a.dtype == np.float32 else a


def _same(got, want, names, imgs, tag):
    for n in names:
        a, b = _bits(got[n][imgs]), _bits(want[n][imgs])
        assert a.shape == b.shape, (tag, n)
        bad = np.argwhere(a != b)
        if len(bad):
            at = tuple(bad[0])
            raise AssertionError(f"{tag}: {n} differs in {len(bad)} entries, first at {bad[:4].tolist()}: "
                                 f"got {got[n][imgs][at]!r}, want {want[n][imgs][at]!r}")


def _check_replicated(got, want, tag):
    for r, g in enumerate(got):
        _same(g, want, PER_IMAGE + MAPS, slice(None), f"{tag} shard {r}")


def _check_distributed(got, want, tag):
    k, B = len(got), want["s"].shape[0]
    for r, g in enumerate(got):
        mine = [i for i in range(B) if i % k == r]
        other = [i for i in range(B) if i % k != r]
        _same(g, want, PER_IMAGE, slice(None), f"{tag} shard {r} (scalars, per-patch arrays)")
        _same(g, want, MAPS, mine, f"{tag} shard {r} (maps of its images {mine})")
        for n in MAPS:
            assert (g[n][other].view(np.uint8) == SENTINEL).all(), f"{tag} shard {r}: {n} of images {other} was written"


# ---- shapes ------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def bank30k(env):
    sy = env.synth
    cent = sy.centroids(768)
    lib = sy.patches(30_011, 768, seed=5, cent=cent)
    full = _bank(env, lib)
    full.build_knn()
    x = np.stack([sy.patches(784, 768, seed=300 + i, anomalous_frac=0.01, cent=cent) for i in range(5)])
    yield SimpleNamespace(lib=lib, full=full, x=x, cent=cent)
    full.close()


@pytest.mark.parametrize("k", [2, 3, 8], ids=lambda k: f"R30011-D768-P784-k{k}")
def test_rounds_of_several_shards_equal_one_bank(env, bank30k, k, capsys):
    """B = 5 images (not a multiple of k): replicated finish with host and device queries, distributed finish (shard r
    finishes images r, r + k, ...; with k = 8 three shards finish none) -- in the certified and the CUDA-core mode"""
    sh = Sharded(env, bank30k.lib, k, full=bank30k.full)
    _report(capsys, sh.layout())
    x = bank30k.x
    xd = torch.from_numpy(x).cuda()
    try:
        for mode in MODES:
            sh.set_mode(env, mode)
            want = _reference(sh.full, x, (28, 28), 224)
            got, _ = _round(env, sh, x, (28, 28), 224)
            _check_replicated(got, want, f"{mode}/host")
            got, _ = _round(env, sh, xd, (28, 28), 224)
            _check_replicated(got, want, f"{mode}/device")
            got, _ = _round(env, sh, x, (28, 28), 224, distribute=True)
            _check_distributed(got, want, f"{mode}/host/distributed")
    finally:
        sh.set_mode(env, "certified")
        sh.close(full=False)


def test_rounds_of_two_200k_row_shards(env, capsys):
    """200 000 x 768 in two shards of 100 000 rows: each shard's GEMM runs the multi-tile-run schedule"""
    sy = env.synth
    cent = sy.centroids(768)
    lib = sy.patches(200_000, 768, seed=6, cent=cent)
    sh = Sharded(env, lib, 2)
    _report(capsys, sh.layout())
    x = np.stack([sy.patches(784, 768, seed=400 + i, anomalous_frac=0.01, cent=cent) for i in range(3)])
    try:
        for mode in MODES:
            sh.set_mode(env, mode)
            want = _reference(sh.full, x, (28, 28), 224)
            got, _ = _round(env, sh, x, (28, 28), 224)
            _check_replicated(got, want, f"{mode}/host")
            got, _ = _round(env, sh, torch.from_numpy(x).cuda(), (28, 28), 224, distribute=True)
            _check_distributed(got, want, f"{mode}/device/distributed")
    finally:
        sh.close()


@pytest.mark.parametrize("R", [3, 4, 5, 6, 7], ids=lambda R: f"R{R}-D64-7x7")
def test_rounds_of_tiny_shards(env, R, capsys):
    """D = 64, 7 x 7 maps, banks of 3 to 7 rows split into 2 .. R shards: one-row shards, shards far below a GEMM tile"""
    sy = env.synth
    lib = sy.patches(R, 64, seed=700 + R, dist="G")
    x = np.stack([sy.patches(49, 64, seed=710 + R * 10 + i, dist="G") for i in range(3)])
    full = _bank(env, lib)
    full.build_knn()
    try:
        for k in range(2, R + 1):
            sh = Sharded(env, lib, k, full=full)
            _report(capsys, sh.layout())
            try:
                for mode in MODES:
                    sh.set_mode(env, mode)
                    want = _reference(full, x, (7, 7), 16)
                    got, _ = _round(env, sh, x, (7, 7), 16)
                    _check_replicated(got, want, f"k={k} {mode}/host")
                    got, _ = _round(env, sh, torch.from_numpy(x).cuda(), (7, 7), 16, distribute=True)
                    _check_distributed(got, want, f"k={k} {mode}/device/distributed")
            finally:
                sh.close(full=False)
                _set_mode(env, [full], "certified")
    finally:
        full.close()


# ---- cross-shard near-ties ---------------------------------------------------------------------------------------

N_PAIRS, NEAR = 24, 128


def _near_tie_bank(env, k):
    """R = 4099 x 64 Gaussian rows; rows J[t] (on the last shard) are copies of rows I[t] (on shard 0) nudged by 2 ulps
    in two coordinates, so that a query near the pair sees d^2 that differ by about one ulp"""
    g = np.random.Generator(np.random.PCG64(77))
    R, D = 4099, 64
    lib = g.standard_normal((R, D), dtype=np.float32)
    I = 100 + np.arange(N_PAIRS)
    J = env.sharding.shard_range(R, k - 1, k)[0] + 300 + np.arange(N_PAIRS)
    for i, j in zip(I, J):
        lib[j] = lib[i]
        for c in g.choice(D, 2, replace=False):
            step = np.float32(np.inf) if g.random() < 0.5 else np.float32(-np.inf)
            lib[j, c] = np.nextafter(np.nextafter(lib[j, c], step), step)
    # candidate queries: near (|q - row| ~ 1.6) and far (~ 4, the farthest patch of an image) around every pair
    near = np.concatenate([lib[i] + 0.2 * g.standard_normal((NEAR, D), dtype=np.float32) for i in I]).astype(np.float32)
    far = np.concatenate([lib[i] + 0.5 * g.standard_normal((NEAR, D), dtype=np.float32) for i in I]).astype(np.float32)
    pair = np.repeat(np.arange(N_PAIRS), NEAR)   # pair of every near and every far candidate
    return lib, I, J, near, far, pair


def _classify(sh, q, I, J, pair):
    """on the device: witness = equal min_val on the shards of I[t] and J[t] (with those rows), the un-sharded bank
    returns J[t]; control = the same, the un-sharded bank returns I[t]"""
    lo_j = sh.ranges[-1][0]
    vi, ii = _exact_min(sh.shards[0], q)
    vj, ij = _exact_min(sh.shards[-1], q)
    vf, jf = _exact_min(sh.full, q)
    tie = (ii == I[pair]) & (ij == J[pair]) & (vi == vj) & (I[pair] < lo_j)
    return tie & (jf == J[pair]), tie & (jf == I[pair])


@pytest.mark.parametrize("k", [2, 3])
def test_cross_shard_near_ties_pick_the_nearer_row(env, k, capsys):
    """Pairs of rows on the first and the last shard whose float32 d^2 to a query differ by an ulp while sqrtf makes
    their distances equal: one bank returns the nearer (higher) row, so the sharded round must too -- the exchange keys
    carry d^2, not the distance.  Image 0's farthest patch is such a witness, so its m_star and nn_idx depend on it."""
    lib, I, J, near, far, pair = _near_tie_bank(env, k)
    sh = Sharded(env, lib, k)
    try:
        wit, ctl = _classify(sh, near, I, J, pair)
        fwit, _ = _classify(sh, far, I, J, pair)
        assert fwit.any(), "no far witness: the farthest patch of image 0 cannot be planted"
        # 4 images of 16 x 16 patches: witnesses and controls first, then the other near queries
        B, P = 4, 256
        order = np.concatenate([np.flatnonzero(wit), np.flatnonzero(ctl), np.flatnonzero(~wit & ~ctl)])[:B * P]
        q = near[order].copy()
        f = int(np.flatnonzero(fwit)[0])
        s_pos = 37
        q[s_pos] = far[f]
        x = q.reshape(B, P, 64)
        n_wit = int(wit[order].sum()) - int(wit[order][s_pos]) + 1
        n_ctl = int(ctl[order].sum()) - int(ctl[order][s_pos])
        _report(capsys, f"{sh.layout()}: {n_wit} witnesses (image 0's farthest patch one of them), {n_ctl} controls "
                        f"among {B * P} queries")
        assert n_wit >= 20, f"only {n_wit} witnesses: the test would not exercise the near-tie"
        assert n_ctl >= 5, f"only {n_ctl} controls"
        for mode in MODES:
            sh.set_mode(env, mode)
            want = _reference(sh.full, x, (16, 16), 64)
            assert want["s_idx"][0, 0] == s_pos and want["min_idx"][0, s_pos] == J[pair[f]]
            assert want["nn_idx"][0, 0] == J[pair[f]]   # m_star is the nearer row J, not I
            got, _ = _round(env, sh, x, (16, 16), 64)
            _check_replicated(got, want, f"{mode}/host")
            got, _ = _round(env, sh, torch.from_numpy(x).cuda(), (16, 16), 64)
            _check_replicated(got, want, f"{mode}/device")
    finally:
        sh.close()


# ---- ownership at shard edges ------------------------------------------------------------------------------------

def test_neighbour_rows_owned_by_different_shards(env, capsys):
    """An image's farthest patch sits next to a row at a shard boundary whose two nearest other rows live on two other
    shards: each shard's lookup contributes only the distances of the rows it owns, zero for the others"""
    g = np.random.Generator(np.random.PCG64(91))
    R, D, k = 3001, 64, 3
    lib = g.standard_normal((R, D), dtype=np.float32)
    ranges = [env.sharding.shard_range(R, r, k) for r in range(k)]
    (lo0, hi0), (lo1, hi1), (lo2, hi2) = ranges
    plant = [(lo1, hi0 - 1, lo2), (hi1 - 1, lo0, hi2 - 1)]   # (m_star row, nearest, second nearest) per image
    B, P, s_pos = 3, 49, 5
    free = np.setdiff1d(np.arange(R), np.array(plant).ravel())   # the other patches sit near rows that stay as drawn
    x = np.stack([lib[g.choice(free, P)] + 0.2 * g.standard_normal((P, D), dtype=np.float32) for _ in range(B)])
    for img, (m, n1, n2) in enumerate(plant):
        v = 0.5 * g.standard_normal(D).astype(np.float32)
        lib[n1] = lib[m] - 0.02 * v + 0.01 * g.standard_normal(D, dtype=np.float32)
        lib[n2] = lib[m] - 0.04 * v + 0.01 * g.standard_normal(D, dtype=np.float32)
        x[img, s_pos] = lib[m] + v
    x = x.astype(np.float32)
    sh = Sharded(env, lib, k)
    _report(capsys, sh.layout())
    owner = lambda row: [r for r, (lo, hi) in enumerate(ranges) if lo <= row < hi][0]   # noqa: E731
    try:
        for mode in MODES:
            sh.set_mode(env, mode)
            want = _reference(sh.full, x, (7, 7), 16)
            got, rd = _round(env, sh, x, (7, 7), 16)
            _check_replicated(got, want, mode)
            for img, rows in enumerate(plant):
                assert want["s_idx"][img, 0] == s_pos and tuple(want["nn_idx"][img]) == rows, (img, want["nn_idx"][img])
                assert len({owner(r) for r in rows[1:]}) == 2
            for img in range(B):
                for kk in range(2):
                    o = owner(int(want["nn_idx"][img, 1 + kk]))
                    vals = [float(c[img * 2 + kk]) for c in rd.contribs]
                    assert vals[o] > 0 and all(v == 0.0 for r, v in enumerate(vals) if r != o), (mode, img, kk, o, vals)
    finally:
        sh.close()


# ---- pipelining ----------------------------------------------------------------------------------------------------

def test_three_outstanding_rounds_waited_out_of_order(env, bank30k, capsys):
    """three rounds opened and closed on every shard before any wait, waited for in a different order on each shard"""
    sy = env.synth
    sh = Sharded(env, bank30k.lib, 3, full=bank30k.full)
    _report(capsys, sh.layout())
    xs = [np.stack([sy.patches(784, 768, seed=500 + 10 * t + i, anomalous_frac=0.01, cent=bank30k.cent) for i in range(3)])
          for t in range(3)]
    try:
        for mode in MODES:
            sh.set_mode(env, mode)
            wants = [_reference(sh.full, x, (28, 28), 224) for x in xs]
            rounds = [_submit(env, sh.shards, torch.from_numpy(x).cuda() if t == 1 else x, (28, 28), 224, distribute=t == 2)
                      for t, x in enumerate(xs)]
            got = [[None] * 3 for _ in range(3)]
            for r, b in enumerate(sh.shards):
                for t in ((2, 0, 1), (1, 2, 0), (0, 2, 1))[r]:
                    got[t][r] = _wait(env, b, rounds[t].tickets[r], 3, 784, 224)
            _check_replicated(got[0], wants[0], f"{mode} round 0")
            _check_replicated(got[1], wants[1], f"{mode} round 1")
            _check_distributed(got[2], wants[2], f"{mode} round 2")
    finally:
        sh.set_mode(env, "certified")
        sh.close(full=False)


# ---- query normalisation on the device ----------------------------------------------------------------------------

def test_device_query_normalisation_equals_torch_on_the_host(env, bank30k, capsys):
    """set_query_norm(mean, std): raw patches scored with (x - mean) / std on the device give the bits of the rounds and
    batches on patches normalised by torch on the CPU in float32"""
    sy = env.synth
    mean, std = float(np.float32(0.3172)), float(np.float32(1.7431))
    raw = np.stack([sy.patches(784, 768, seed=600 + i, anomalous_frac=0.01, cent=bank30k.cent) for i in range(3)])
    raw = (raw * np.float32(1.7) + np.float32(0.3)).astype(np.float32)
    rt = torch.from_numpy(raw)
    normed = ((rt - torch.full_like(rt, mean)) / torch.full_like(rt, std)).numpy()
    assert (normed == ((raw - np.float32(mean)) / np.float32(std)).astype(np.float32)).all()
    sh = Sharded(env, bank30k.lib, 3, full=bank30k.full)
    _report(capsys, sh.layout())
    handles = [sh.full] + sh.shards
    try:
        for mode in MODES:
            sh.set_mode(env, mode)
            want = _reference(sh.full, normed, (28, 28), 224)
            for b in handles:
                b.set_query_norm(mean, std)
            try:
                for src, xs in (("host", raw), ("device", rt.cuda())):
                    got, _ = _round(env, sh, xs, (28, 28), 224)
                    _check_replicated(got, want, f"{mode}/{src} sharded")
                    one = sh.full.score_batch(xs, (28, 28), 224, full=True).arrays
                    _same(one, want, PER_IMAGE + MAPS, slice(None), f"{mode}/{src} score_batch")
                    one = sh.full.score_batch_async(xs, (28, 28), 224, full=True).wait().arrays
                    _same(one, want, PER_IMAGE + MAPS, slice(None), f"{mode}/{src} score_batch_async")
            finally:
                for b in handles:
                    b.set_query_norm(0.0, 1.0, enabled=False)
    finally:
        sh.set_mode(env, "certified")
        sh.close(full=False)
