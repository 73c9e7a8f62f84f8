"""CPU suite: the distance GEMM's tile schedule with runs of N tiles, restated on the host, and the library's one
enumeration of "the rows producer (CTA c, column group g) saw for M tile m", which the exact rescan (rescan_kernel) and
the re-weighting certificate (reweight_cert_kernel) share -- checked against it for the launch shapes of large banks
through the host-only hook cmdb_debug_producer_tiles.  tests/test_gpu_schedule.py checks the same restatement against
the candidate lists the GPU writes."""
import ctypes
from math import gcd

import numpy as np

BM, BN, EG = 128, 256, 2      # query rows per M tile, bank rows per N tile, epilogue column groups (score_gemm.cu)
COLS = BN // EG
G_B200 = 148                  # CTAs of the GEMM launch: one per SM


# ---- restatement of score_gemm.cu / score_tail.cu (host side) ----------------------------------------------------
def tile_stride(mt, G):
    """score_tile_stride: the first s >= mt with gcd(s mod G, G) == 1"""
    s = mt
    while True:
        a = s % G or G
        if gcd(a, G) == 1 or G == 1:
            return s
        s += 1


def gemm_run(nt, mt_units, G):
    """score_gemm_run: N tiles per visit of an M tile"""
    ideal = nt * mt_units / G
    for run in range(min(8, max(1, nt // G)), 1, -1):
        nruns = (nt + run - 1) // run
        makespan = (nruns * mt_units + G - 1) // G * run
        if makespan <= ideal * 1.02:
            return run
    return 1


def stage_chunks(P, device, pending=False):
    """score_local_min's split of a batch of P query rows into GEMM launches: [(first M tile, M tiles)]"""
    mt_total = (P + BM - 1) // BM
    via_copy = not device and (pending or mt_total >= 16)
    n = 1
    if via_copy and not pending:
        n = 4 if mt_total >= 64 else 2
    n = max(1, min(n, mt_total))
    ct = (mt_total + n - 1) // n
    n = (mt_total + ct - 1) // ct
    return [(c * ct, min(ct, mt_total - c * ct)) for c in range(n)]


def table_chunks(row_first, n_rows):
    """score_build_knn_table: launches of <= 8192 rows from row_first on: [(first row, rows)]"""
    return [(r, min(64 * BM, row_first + n_rows - r)) for r in range(row_first, row_first + n_rows, 64 * BM)]


def tile_iter(c, G, mt, stride, nruns):
    """TileIter of score_gemm_kernel, literally: the (run, M tile) pairs unit c processes, in order"""
    smod = stride % G
    n, m, base = -1, mt, (c + smod) % G
    while True:
        m += G
        while m >= mt:
            n += 1
            if n >= nruns:
                return
            base -= smod
            if base < 0:
                base += G
            m = base
        yield n, m


class Launch:
    """one GEMM launch (no CTA pairs: the pre-filter GEMMs behind the rescan and the re-weighting certificate never pair):
    nt N tiles over `rows` bank rows, mt M tiles, G CTAs.  owner[j, m] = CTA that ran (run j, M tile m)."""

    def __init__(self, rows, mt, G=G_B200):
        self.rows, self.mt, self.G = rows, mt, G
        self.nt = (rows + BN - 1) // BN
        self.run = gemm_run(self.nt, mt, G)
        self.stride = tile_stride(mt, G)
        self.nruns = (self.nt + self.run - 1) // self.run
        owner = np.full((self.nruns, mt), -1, np.int64)
        for c in range(G):
            for j, m in tile_iter(c, G, mt, self.stride, self.nruns):
                assert owner[j, m] == -1, ("dealt twice", j, m)
                owner[j, m] = c
        self.owner = owner

    def tiles(self, c, m):
        """N tiles CTA c processed for M tile m"""
        return sorted(n for j in np.nonzero(self.owner[:, m] == c)[0]
                      for n in range(j * self.run, min(self.nt, (j + 1) * self.run)))

    def rows_of(self, c, g, m):
        """bank rows producer (c, g) saw for M tile m"""
        r = np.concatenate([n * BN + g * COLS + np.arange(COLS) for n in self.tiles(c, m)] or [np.zeros(0, np.int64)])
        return r[r < self.rows]

    def row_owner(self, m, r):
        """CTA whose list for M tile m saw bank rows r (array): the owner of the row's run"""
        return self.owner[r // BN // self.run, m]


# ---- the library's enumeration ----------------------------------------------------------------------------------------
class ProducerTiles:
    """cmdb_debug_producer_tiles: the N tiles the exact rescan visits for (query in M tile `mtile` of a batch whose
    first-pass GEMM ran in launches of chunk_tiles out of mt_total M tiles, CTA c), from the schedules the library records
    for the full and the last chunk launch, in slot order -- so a slot bound that misses part of a producer shows as
    missing tiles.  A single chunk (chunk_tiles == mt_total) is reweight_cert_kernel's walk over a launch of that size."""

    def __init__(self, G=G_B200):
        from cmdiad_b200 import _lib as L
        self.L, self.lib, self.G = L, L.load(), G
        self.buf, self.n = (ctypes.c_int32 * 65536)(), ctypes.c_int()

    def __call__(self, c, mtile, nt, chunk_tiles, mt_total):
        self.L.check(self.lib.cmdb_debug_producer_tiles(self.G, nt, chunk_tiles, mt_total, mtile, c, self.buf,
                                                        len(self.buf), ctypes.byref(self.n)))
        return self.buf[:self.n.value]


# ---- shapes -----------------------------------------------------------------------------------------------------------
P_IMG = 784
ROWS = (100_000, 150_000, 200_000, 400_000)


def batch_layouts(rows):
    """(what, chunk launches) of the scoring calls the large-bank tests run"""
    out = []
    for B in (3, 6, 16):
        out.append((f"{B} img host", stage_chunks(B * P_IMG, device=False)))
        out.append((f"{B} img device", stage_chunks(B * P_IMG, device=True)))
        out.append((f"{B} img pending", stage_chunks(B * P_IMG, device=False, pending=True)))
    return out


def test_schedule_restatement_matches_the_library(built):
    from cmdiad_b200 import _lib as L
    lib = L.load()
    for mt in (1, 2, 3, 4, 9, 10, 18, 19, 23, 25, 37, 49, 53, 64, 74, 98, 148, 149, 296):
        for G in (148, 74, 7, 1):
            assert tile_stride(mt, G) == lib.cmdb_debug_tile_stride(mt, G), (mt, G)


def test_run_lengths_of_large_banks():
    """run length (full chunk / last chunk) per bank size and call kind: the shapes the GPU tests claim to exercise"""
    def runs(rows, chunks):
        nt = (rows + BN - 1) // BN
        return tuple(dict.fromkeys(gemm_run(nt, mt, G_B200) for _, mt in (chunks[0], chunks[-1])))
    lay = {rows: dict(batch_layouts(rows)) for rows in ROWS}
    assert [len(lay[200_000][k]) for k in ("16 img host", "16 img device", "16 img pending", "3 img host")] == [4, 1, 1, 2]
    assert runs(200_000, lay[200_000]["16 img host"]) == (2, 3)
    assert runs(200_000, lay[200_000]["16 img device"]) == (5,)
    assert runs(200_000, lay[200_000]["3 img host"]) == (1, 4)
    assert runs(400_000, lay[400_000]["6 img host"]) == (7, 8)
    assert runs(150_000, lay[150_000]["16 img host"]) == (2,)
    assert runs(100_000, lay[100_000]["6 img host"]) == (1, 2)
    tbl = {rows: runs(rows, [(0, (n + BM - 1) // BM) for _, n in table_chunks(0, rows)]) for rows in ROWS}
    assert tbl == {100_000: (2, 1), 150_000: (3, 2), 200_000: (5,), 400_000: (8,)}
    assert table_chunks(0, 200_000)[-1] == (196_608, 3392) and len(table_chunks(0, 200_000)) == 25
    assert [gemm_run((r + BN - 1) // BN, 1, G_B200) for r in ROWS] == [1, 2, 1, 1]   # re-weighting GEMM: one M tile


def _launch_shapes():
    """(bank rows, [launch M tiles]) of every scoring / table launch at the large-bank sizes, plus awkward gcds"""
    out = []
    for rows in ROWS:
        mts = {mt for _, chunks in batch_layouts(rows) for _, mt in chunks}
        mts |= {(n + BM - 1) // BM for _, n in table_chunks(0, rows)} | {1}
        out.append((rows, sorted(mts)))
    # mt sharing factors with 148 = 4 * 37 (stride != mt), nt not a multiple of the run, tiny and huge nt
    out += [(300_001, [2, 37, 74, 111]), (77_000, [4, 148, 150]), (1_000_000, [8, 98]), (40_000, [1, 3])]
    return out


def test_tile_schedule_with_runs_partitions_the_bank():
    """every (run, M tile) pair is dealt to exactly one CTA; for every M tile the 296 producers' row sets partition the
    bank; every window of G runs is dealt evenly"""
    for rows, mts in _launch_shapes():
        for mt in mts:
            la = Launch(rows, mt)
            assert (la.owner >= 0).all(), (rows, mt)          # ... and exactly once (Launch asserts)
            for w in range(0, la.nruns - la.G + 1, la.G):   # every G runs each CTA receives exactly mt pairs
                assert (np.bincount(la.owner[w:w + la.G].ravel(), minlength=la.G) == mt).all(), (rows, mt, w)
            for m in sorted({0, mt // 2, mt - 1}):
                got = np.concatenate([la.rows_of(c, g, m) for c in range(la.G) for g in range(EG)])
                assert got.size == rows and (np.sort(got) == np.arange(rows)).all(), (rows, mt, m)
            if la.nruns >= la.G:   # every producer sees rows of every query tile (what the certificate leans on)
                assert all(len(set(la.owner[:, m])) == la.G for m in sorted({0, mt - 1}))


def test_rescan_enumeration_equals_the_gemm_schedule(built):
    """the rescan's closed form (stride inverse, run_full / run_last, tile slots sized from run_min / run_max) names
    exactly the N tiles the GEMM's iterator gave each producer, each once, for every producer and every M tile of every
    chunk, full and last"""
    rescan_tiles = ProducerTiles()
    n_diff_runs = 0
    for rows in ROWS:
        nt = (rows + BN - 1) // BN
        for what, chunks in batch_layouts(rows):
            ct, mt_total = chunks[0][1], chunks[-1][0] + chunks[-1][1]
            launches = {mt: Launch(rows, mt) for mt in {mt for _, mt in chunks}}
            n_diff_runs += launches[chunks[0][1]].run != launches[chunks[-1][1]].run
            for first, mt in (chunks[0], chunks[-1]):
                la = launches[mt]
                for m in range(mt):
                    for c in range(la.G):
                        assert sorted(rescan_tiles(c, first + m, nt, ct, mt_total)) == la.tiles(c, m), (rows, what, first, m, c)
    assert n_diff_runs >= 6   # run_full != run_last is exercised


def test_reweight_certificate_walk_equals_the_gemm_schedule(built):
    """reweight_cert_kernel's bad-producer walk (first run, then every G runs, `run` tiles each) names exactly the GEMM
    iterator's tiles, in order: table-build launches (full and ragged last chunk, chunks starting anywhere) and the
    one-M-tile re-weighting launch"""
    producer_tiles = ProducerTiles()
    for rows, mts in _launch_shapes():
        for mt in mts:
            la = Launch(rows, mt)
            for m in sorted({0, 1 % mt, mt // 2, mt - 1}):
                for c in range(la.G):
                    assert producer_tiles(c, m, la.nt, mt, mt) == la.tiles(c, m), (rows, mt, m, c)
