"""Python handle around one device-resident memory bank (cmdb_bank) -- thin marshalling only, all compute is in the
CUDA library.  torch is used for host/device buffers and streams, never for the arithmetic of the path."""
import ctypes

import numpy as np
import torch

from . import _lib as L


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        return ctypes.c_void_p(t.data_ptr())
    return ctypes.c_void_p(t.ctypes.data)


def _as_f32(x):
    """contiguous float32 torch tensor (host or device) without copying when already so"""
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    if x.dtype != torch.float32:
        x = x.float()
    return x.contiguous()


class ScoreResult:
    """Outputs of one scoring call; field names follow compute_single_s_s_map (features.py:225-297)."""
    __slots__ = ("s", "s_star", "s_idx", "min_val", "min_idx", "nn_idx", "m_star_knn", "w", "s_map", "s_map_pre",
                 "s_map_u8")


class Comm:
    """Peer-mapped buffer of this rank for the row-sharded coreset loop (CUDA IPC over NVLink, one process per GPU): key
    slots for the per-pick exchange + a replica of the whole projected bank.  Collective constructor: every rank of
    `group` must create it together; coreset_select_sharded grows it (collectively) when a bank needs more room."""

    def __init__(self, device, d_proj_max=512, group=None, rows_max=0, dtype_mode=L.CORESET_FP16):
        import torch.distributed as dist
        self._lib = L.load()
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = int(device)
        self.d_proj_max = int(d_proj_max)
        self._h = ctypes.c_void_p()
        self.bytes = 0
        self._create(self._lib.cmdb_coreset_comm_bytes(self.world, int(d_proj_max), int(rows_max), int(dtype_mode)))

    def _create(self, nbytes):
        import torch.distributed as dist
        self.close()
        L.check(self._lib.cmdb_comm_create(self.device, self.rank, self.world, int(nbytes), ctypes.byref(self._h)))
        hb = self._lib.cmdb_comm_handle_bytes()
        mine = np.zeros(hb, np.uint8)
        L.check(self._lib.cmdb_comm_export(self._h, _ptr(mine)))
        dev = torch.device("cuda", self.device)
        gathered = torch.empty(self.world * hb, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(gathered, torch.from_numpy(mine).to(dev), group=self.group)
        handles = np.ascontiguousarray(gathered.cpu().numpy())
        L.check(self._lib.cmdb_comm_import(self._h, _ptr(handles)))
        self.bytes = int(nbytes)
        for b in list(self.__dict__.get("_attached", ())):   # banks that exchange through this buffer follow it
            if b._h:
                L.check(self._lib.cmdb_bank_attach_comm(b._h, self._h))

    def ensure(self, nbytes):
        """collective: every rank passes the same size"""
        import torch.distributed as dist
        if self.bytes < nbytes:
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)   # nobody still uses the old mapping
            self._create(nbytes)

    def reset_and_barrier(self):
        import torch.distributed as dist
        L.check(self._lib.cmdb_comm_reset(self._h))
        dist.barrier(group=self.group)

    def close(self):
        if getattr(self, "_h", None):
            for b in list(self.__dict__.get("_attached", ())):
                if b._h:
                    self._lib.cmdb_bank_attach_comm(b._h, None)
            self._lib.cmdb_comm_destroy(self._h)
            self._h = ctypes.c_void_p()
            self.bytes = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchResult:
    """Results of a batch: r[i] is a ScoreResult viewing image i of the batch arrays (created on demand)."""

    def __init__(self, arrays, owned=None):
        self.arrays = arrays
        self.owned = owned  # None = all images; otherwise a set of image indices that were finished on this rank

    def __len__(self):
        return self.arrays["s"].shape[0]

    def __getitem__(self, i):
        if i < 0:
            i += len(self)
        if self.owned is not None and i not in self.owned:
            return None
        r = ScoreResult()
        for name, a in self.arrays.items():
            setattr(r, name, a[i] if a is not None else None)
        return r

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class Bank:
    """One memory bank (patch_rgb_lib / patch_xyz_lib / patch_fusion_lib) resident in HBM on one GPU."""

    def __init__(self, dim, capacity_rows, device=0, row_offset=0):
        self._lib = L.load()
        self._h = ctypes.c_void_p()
        L.check(self._lib.cmdb_bank_create(int(device), int(dim), int(capacity_rows), ctypes.byref(self._h)))
        self.dim = int(dim)
        self.device = int(device)
        self.capacity = int(capacity_rows)
        if row_offset:
            self.set_row_offset(row_offset)

    # ---- lifecycle -------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.cmdb_bank_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def rows(self):
        n = ctypes.c_int64()
        L.check(self._lib.cmdb_bank_rows(self._h, ctypes.byref(n)))
        return n.value

    def set_row_offset(self, off):
        L.check(self._lib.cmdb_bank_set_row_offset(self._h, int(off)))
        self._row_off = int(off)

    def set_score_impl(self, impl):
        L.check(self._lib.cmdb_bank_set_option(self._h, L.OPT_SCORE_IMPL, int(impl)))

    def set_prefilter_terms(self, terms):
        """Distance-GEMM mode.  0 (default): certified hi.hi pre-filter, uncertified queries redone with the
        FP32-equivalent GEMM; 3: FP32-equivalent GEMM for every query; 1: uncertified pre-filter (diagnostics)."""
        L.check(self._lib.cmdb_bank_set_option(self._h, L.OPT_PREFILTER_TERMS, int(terms)))

    def attach_comm(self, comm):
        """Row-sharded scoring without NCCL: rounds exchange through `comm`'s peer-mapped buffers (the ones the sharded
        coreset loop uses), fused into the kernels (cmdb_score_shard_round_submit).  None detaches."""
        old = getattr(self, "_comm", None)
        if old is not None and self in old.__dict__.get("_attached", []):
            old._attached.remove(self)
        L.check(self._lib.cmdb_bank_attach_comm(self._h, comm._h if comm is not None else None))
        self._comm = comm
        if comm is not None:
            comm.__dict__.setdefault("_attached", []).append(self)

    def set_query_norm(self, mean, std, enabled=True):
        """enabled: scoring calls take RAW patches and compute (patch - mean) / std on the device (float32, bit-identical
        to the reference's host expression, multiple_features.py:90)"""
        L.check(self._lib.cmdb_bank_set_query_norm(self._h, float(mean), float(std), int(bool(enabled))))

    def build_knn(self):
        """Precompute the three nearest bank rows of every bank row (exact; the bank against itself through the
        certified pre-filter GEMM).  The re-weighting step of score / score_batch then becomes a table lookup with
        identical results.  Un-sharded banks only; call after finalize()."""
        L.check(self._lib.cmdb_bank_build_knn(self._h))

    def build_knn_rows(self, row_first, n_rows):
        """neighbour-table entries of rows [row_first, row_first + n_rows) only (the others stay empty)"""
        L.check(self._lib.cmdb_bank_build_knn_rows(self._h, int(row_first), int(n_rows)))

    def read_knn(self, row_first, n_rows, out=None):
        """packed (d^2 bits << 32 | global row) keys [n_rows, 3] of the neighbour table; out: int64 tensor (host or device)"""
        if out is None:
            out = torch.empty((n_rows, 3), dtype=torch.int64)
        assert out.is_contiguous() and out.numel() >= 3 * n_rows
        L.check(self._lib.cmdb_bank_read_knn(self._h, int(row_first), int(n_rows), _ptr(out), int(out.is_cuda)))
        return out

    def set_knn_table(self, keys, n_rows_total):
        """installs a replicated table covering ALL global rows on this (row-sharded) handle"""
        assert keys.dtype == torch.int64 and keys.is_contiguous() and keys.numel() == 3 * n_rows_total
        self._order_after_producer(keys)
        if keys.is_cuda:
            torch.cuda.current_stream(keys.device).synchronize()
        L.check(self._lib.cmdb_bank_set_knn_table(self._h, _ptr(keys), int(n_rows_total), int(keys.is_cuda)))
        self._knn_replicated = True

    def read_device(self, row0=0, n_rows=None, out=None):
        n_rows = self.rows - row0 if n_rows is None else n_rows
        if out is None:
            out = torch.empty((n_rows, self.dim), dtype=torch.float32, device=torch.device("cuda", self.device))
        L.check(self._lib.cmdb_bank_read_device(self._h, int(row0), int(n_rows), _ptr(out)))
        return out

    def build_knn_sharded(self, group=None):
        """Row-sharded bank: builds the REPLICATED neighbour table (SURVEY 8f-1 for sharded banks).  Collective: the fp32
        shards are all-gathered over NVLink into a temporary un-sharded handle on every rank, each rank computes the table
        entries of the rows it owns (R/world x R distance work per rank, through the same certified GEMM), and the
        24-byte-per-row slices are all-gathered.  score_sharded_batch / score_sharded_async look the neighbours of
        m_star up in this table, so a round needs two small collectives and no re-weighting pass over the bank.
        finalize() drops the table."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        dev = torch.device("cuda", self.device)
        rows = self.rows
        counts = torch.zeros(world, dtype=torch.int64, device=dev)
        counts[rank] = rows
        dist.all_reduce(counts, group=group)
        counts = counts.cpu().tolist()
        offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        n_total, max_rows = int(offs[-1]), int(max(counts))
        assert int(offs[rank]) == self._row_offset(), "shards must be contiguous blocks in rank order"
        mine = torch.zeros((max_rows, self.dim), dtype=torch.float32, device=dev)
        self.read_device(0, rows, out=mine)
        gathered = torch.empty((world * max_rows, self.dim), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(gathered, mine, group=group)
        torch.cuda.current_stream(dev).synchronize()
        del mine
        full = Bank(self.dim, n_total, device=self.device)
        for r in range(world):
            full.append(gathered[r * max_rows:r * max_rows + counts[r]])
        del gathered
        full.finalize()
        full.build_knn_rows(int(offs[rank]), rows)
        keys_mine = torch.full((max_rows, 3), -1, dtype=torch.int64, device=dev)
        full.read_knn(int(offs[rank]), rows, out=keys_mine)
        full.close()
        all_keys = torch.empty((world * max_rows, 3), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(all_keys, keys_mine, group=group)
        table = torch.cat([all_keys[r * max_rows:r * max_rows + counts[r]] for r in range(world)]).contiguous()
        self.set_knn_table(table, n_total)

    def score_stats(self):
        """Counters of the last scoring call on this handle: queries, GEMM mode that ran, and for the certified
        pre-filter how many queries it could not certify, how many (query, producer) pairs were rescanned exactly,
        whether the 3-term GEMM fallback ran instead, and how many calls the adaptive mode still runs in mode 3."""
        arr = (ctypes.c_int64 * 6)()
        L.check(self._lib.cmdb_bank_score_stats(self._h, arr))
        return {"queries": int(arr[0]), "mode": int(arr[1]), "fallback_queries": int(arr[2]),
                "rescan_pairs": int(arr[3]), "gemm_fallback": bool(arr[4]), "direct_calls_left": int(arr[5])}

    def set_timing(self, on=True):
        L.check(self._lib.cmdb_bank_set_option(self._h, L.OPT_TIMING, int(bool(on))))

    def timings(self):
        """{stage: ms} of the last score() call (CUDA events on the handle's stream); needs set_timing(True)"""
        arr = (ctypes.c_float * len(L.T_STAGES))()
        L.check(self._lib.cmdb_bank_get_timings(self._h, arr))
        return dict(zip(L.T_STAGES, [float(x) for x in arr]))

    def lane_streams(self):
        """torch views of the handle's two lane streams (scoring calls alternate between them)"""
        st = getattr(self, "_lanes", None)
        if st is None:
            arr = (ctypes.c_void_p * 2)()
            L.check(self._lib.cmdb_bank_lane_streams(self._h, arr))
            dev = torch.device("cuda", self.device)
            st = self._lanes = {int(arr[i]): torch.cuda.ExternalStream(int(arr[i]), device=dev) for i in range(2)}
        return st

    def stream(self):
        """torch view of the CUDA stream the NEXT scoring call of this handle runs on (event timing, ordering of
        collectives between the phases of a sharded round)"""
        p = ctypes.c_void_p()
        L.check(self._lib.cmdb_bank_stream(self._h, ctypes.byref(p)))
        return self.lane_streams()[int(p.value)]

    def _order_after_producer(self, t):
        """Device inputs: the library reads `t` on the handle's own (non-blocking) lane streams, so those first have to
        wait for whatever torch stream is producing it (ordering contract of `*_is_device = 1`, include/cmdiad_b200.h).
        The tensor is kept alive by the caller / the ticket until the library has consumed it (synchronous calls return
        after that point), so torch's caching allocator cannot recycle the block early; tensor.record_stream is
        deliberately NOT used: it would make the allocator touch the handle's stream when the tensor dies, possibly after
        the bank (and its stream) has been closed."""
        if isinstance(t, torch.Tensor) and t.is_cuda:
            cur = torch.cuda.current_stream(t.device)
            for st in self.lane_streams().values():
                st.wait_stream(cur)
        return t

    # ---- storage ---------------------------------------------------------------------------------------------
    def append(self, rows):
        rows = _as_f32(rows)
        assert rows.dim() == 2 and rows.shape[1] == self.dim, f"expected [n,{self.dim}], got {tuple(rows.shape)}"
        self._order_after_producer(rows)
        L.check(self._lib.cmdb_bank_append(self._h, _ptr(rows), rows.shape[0], int(rows.is_cuda)))

    def stats(self):
        """(mean, unbiased std, sum, sum of squares) over all elements, float64"""
        m, s, sm, sq = (ctypes.c_double() for _ in range(4))
        L.check(self._lib.cmdb_bank_stats(self._h, ctypes.byref(m), ctypes.byref(s), ctypes.byref(sm), ctypes.byref(sq)))
        return m.value, s.value, sm.value, sq.value

    def normalize(self, mean, std):
        L.check(self._lib.cmdb_bank_normalize(self._h, float(mean), float(std)))

    def gather(self, idx):
        idx = np.ascontiguousarray(np.asarray(idx, dtype=np.int64))
        L.check(self._lib.cmdb_bank_gather(self._h, _ptr(idx), idx.shape[0]))

    def read(self, row0=0, n_rows=None):
        n_rows = self.rows - row0 if n_rows is None else n_rows
        out = torch.empty((n_rows, self.dim), dtype=torch.float32)
        L.check(self._lib.cmdb_bank_read(self._h, int(row0), int(n_rows), _ptr(out)))
        return out

    def finalize(self):
        L.check(self._lib.cmdb_bank_finalize(self._h))
        self._knn_replicated = False   # cmdb_bank_finalize frees the neighbour table

    # ---- persistence (SURVEY 8f: the reference rebuilds its banks on every run and never saves them) -------------------
    def save(self, path, **meta):
        """rows (float32, exactly as stored: normalised / subsampled) + row_offset + caller metadata -> one .npz"""
        np.savez(path, rows=self.read().numpy(), dim=np.int64(self.dim), row_offset=np.int64(self._row_offset()),
                 **{f"meta_{k}": np.asarray(v) for k, v in meta.items()})

    @classmethod
    def load(cls, path, device=0, finalize=True, capacity_rows=None):
        """returns (bank, meta dict); the scoring layout is rebuilt on the device (finalize=True)"""
        with np.load(path) as f:
            rows = f["rows"]
            bank = cls(int(f["dim"]), capacity_rows or max(1, rows.shape[0]), device=device, row_offset=int(f["row_offset"]))
            meta = {k[5:]: f[k] for k in f.files if k.startswith("meta_")}
        if rows.shape[0]:
            bank.append(rows)
            if finalize:
                bank.finalize()
        return bank, meta

    def _row_offset(self):
        return getattr(self, "_row_off", 0)

    # ---- coreset ---------------------------------------------------------------------------------------------
    @staticmethod
    def _csr(csr):
        if csr is None:
            return None, None, None, 0
        indptr, indices, data, d_proj = csr
        return (np.ascontiguousarray(indptr, dtype=np.int32), np.ascontiguousarray(indices, dtype=np.int32),
                np.ascontiguousarray(data, dtype=np.float64), int(d_proj))

    def coreset_select(self, n_select, csr, dtype_mode=L.CORESET_FP16, force_idx=None, return_min=False,
                       _mind_global=False):
        """Greedy k-center selection on the projected bank; csr = (indptr, indices, data, d_proj) or None.
        _mind_global (tests): keep the kernel's min-distance vector in global memory even where it fits shared memory."""
        indptr, indices, data, d_proj = self._csr(csr)
        out = np.zeros(int(n_select), dtype=np.int64)
        if force_idx is None and not return_min and not _mind_global:
            L.check(self._lib.cmdb_coreset_select(self._h, int(n_select), _ptr(indptr), _ptr(indices), _ptr(data), d_proj,
                                                  int(dtype_mode), _ptr(out)))
            return out
        fi = None if force_idx is None else np.ascontiguousarray(force_idx, dtype=np.int64)
        mn = np.zeros(self.rows, dtype=np.float16 if dtype_mode == L.CORESET_FP16 else np.float64)
        L.check(self._lib.cmdb_coreset_select_debug(self._h, int(n_select), _ptr(indptr), _ptr(indices), _ptr(data),
                                                    d_proj, int(dtype_mode), _ptr(out), _ptr(fi), _ptr(mn),
                                                    int(bool(_mind_global))))
        return (out, mn) if return_min else out

    def coreset_select_sharded(self, comm, n_total_rows, n_select, csr, dtype_mode=L.CORESET_FP16):
        """Row-sharded greedy selection: this bank holds global rows [row_offset, row_offset + rows) of an n_total_rows
        bank; every rank calls this together and gets the same GLOBAL indices as the single-GPU coreset_select."""
        import torch.distributed as dist
        indptr, indices, data, d_proj = self._csr(csr)
        comm.ensure(self._lib.cmdb_coreset_comm_bytes(comm.world, d_proj, int(n_total_rows), int(dtype_mode)))
        dev = torch.device("cuda", self.device)
        z0 = torch.zeros(d_proj, dtype=torch.float64, device=dev)
        if comm.rank == 0:  # rank 0 owns global row 0 (contiguous shards in rank order)
            z0.copy_(torch.from_numpy(self.project(csr, 0, 1)[0]))
        dist.broadcast(z0, src=dist.get_global_rank(comm.group, 0) if comm.group is not None else 0, group=comm.group)
        z0_host = np.ascontiguousarray(z0.cpu().numpy())
        comm.reset_and_barrier()
        out = np.zeros(int(n_select), dtype=np.int64)
        L.check(self._lib.cmdb_coreset_select_sharded(self._h, comm._h, int(n_total_rows), int(n_select), _ptr(indptr),
                                                      _ptr(indices), _ptr(data), d_proj, int(dtype_mode), _ptr(z0_host),
                                                      _ptr(out)))
        return out

    def project(self, csr, row0=0, n_rows=None):
        indptr, indices, data, d_proj = self._csr(csr)
        n_rows = self.rows - row0 if n_rows is None else n_rows
        out = np.zeros((n_rows, d_proj), dtype=np.float64)
        L.check(self._lib.cmdb_project(self._h, _ptr(indptr), _ptr(indices), _ptr(data), d_proj, int(row0), int(n_rows),
                                       _ptr(out)))
        return out

    # ---- scoring ---------------------------------------------------------------------------------------------
    @staticmethod
    def _alloc_out(B, P, out_hw, full):
        """batch arrays + the matching array of struct cmdb_score_out (filled by pointer arithmetic, no per-image views)"""
        arr = dict(s=np.empty((B, 1), np.float32), s_star=np.empty((B, 1), np.float32), s_idx=np.empty((B, 1), np.int64),
                   min_val=np.empty((B, P), np.float32), min_idx=np.empty((B, P), np.int64), nn_idx=np.empty((B, 3), np.int64),
                   m_star_knn=np.empty((B, 2), np.float32), w=np.empty((B, 1), np.float32),
                   s_map=np.empty((B, out_hw, out_hw), np.float32),
                   s_map_pre=np.empty((B, out_hw, out_hw), np.float32) if full else None,
                   s_map_u8=np.empty((B, out_hw, out_hw), np.uint8) if full else None)
        outs = (L.ScoreOut * B)()
        base = ctypes.addressof(outs)
        size = ctypes.sizeof(L.ScoreOut)
        ptrs = (ctypes.c_void_p * (11 * B)).from_address(base)  # struct cmdb_score_out is 11 pointers
        assert size == 11 * ctypes.sizeof(ctypes.c_void_p)
        for f, (name, _) in enumerate(L.ScoreOut._fields_):
            a = arr[name]
            if a is None:
                continue
            p0, st = a.ctypes.data, a.strides[0]
            for i in range(B):
                ptrs[i * 11 + f] = p0 + i * st
        return BatchResult(arr), outs, arr

    def score(self, patch, feature_map_dims, out_hw=224, full=False):
        """calculate_dist + compute_single_s_s_map for one image; patch [P,dim] float32, already normalised."""
        patch = _as_f32(patch)
        return self.score_batch(patch.unsqueeze(0), feature_map_dims, out_hw, full)[0]

    def score_batch(self, patches, feature_map_dims, out_hw=224, full=False):
        """B images at once: patches [B,P,dim] float32 (host or device).  Returns a list of B ScoreResult."""
        patches = _as_f32(patches)
        assert patches.dim() == 3 and patches.shape[2] == self.dim, f"expected [B,P,{self.dim}], got {tuple(patches.shape)}"
        B, P = patches.shape[0], patches.shape[1]
        fh, fw = feature_map_dims
        results, outs, _ = self._alloc_out(B, P, out_hw, full)
        self._order_after_producer(patches)
        L.check(self._lib.cmdb_score_batch(self._h, _ptr(patches), B, P, int(fh), int(fw), int(out_hw), int(patches.is_cuda),
                                           outs))
        return results

    def score_batch_async(self, patches, feature_map_dims, out_hw=224, full=False):
        """Pipelined score_batch: enqueues the batch (at most max_shard_batch() images) and returns a ticket at once;
        ticket.wait() returns the list of ScoreResult.  Three batches may be outstanding per bank, so the result copy of
        batch k and the staging of batch k+1 overlap the kernels of the other compute lane, and the host's enqueue time
        never delays the next distance GEMM:

            pending = []
            for batch in batches:
                pending.append(bank.score_batch_async(batch, dims))
                if len(pending) == 3: consume(pending.pop(0).wait())
            while pending: consume(pending.pop(0).wait())
        """
        patches = _as_f32(patches)
        assert patches.dim() == 3 and patches.shape[2] == self.dim, f"expected [B,P,{self.dim}], got {tuple(patches.shape)}"
        B, P = patches.shape[0], patches.shape[1]
        fh, fw = feature_map_dims
        ticket = ctypes.c_int64()
        self._order_after_producer(patches)
        L.check(self._lib.cmdb_score_batch_submit(self._h, _ptr(patches), B, P, int(fh), int(fw), int(out_hw),
                                                  int(patches.is_cuda), 3 if full else 0, ctypes.byref(ticket)))
        return _Ticket(self, ticket.value, patches, B, P, out_hw, full)

    def max_shard_batch(self):
        """images per round of the sharded protocol (shared-memory bound of the re-weighting kernel)"""
        return max(1, min(32, (160 * 1024) // (4 * self.dim + 8 * 3 * 8)))

    def score_sharded(self, patch, feature_map_dims, out_hw=224, full=False, group=None):
        patch = _as_f32(patch)
        return self.score_sharded_batch(patch.unsqueeze(0), feature_map_dims, out_hw, full, group)[0]

    def _shard_buf(self, name, slot, shape, dtype):
        """device buffers of the sharded rounds, cached per result slot (no allocator traffic per round)"""
        cache = self.__dict__.setdefault("_shard_bufs", {})
        key = (name, slot, tuple(shape), dtype)
        t = cache.get(key)
        if t is None:
            t = cache[key] = torch.empty(shape, dtype=dtype, device=torch.device("cuda", self.device))
        return t

    def _stage_sharded(self, chunk, slot, world, rank, group, lane):
        """Host queries of a sharded round: every rank copies only its 1/world slice of the rows over PCIe and the slices
        are all-gathered over NVLink -- every rank needs all queries, but NVLink is ~10x the host link.  Copy and
        all-gather run on a staging stream of their own, so that with several rounds outstanding they overlap the kernels
        of the earlier rounds instead of sitting in front of this round's GEMM on its lane; the lane only waits for the
        event behind the all-gather.  One set of buffers per outstanding round (slot = round % 3): a set is rewritten
        three rounds later, after the caller has waited for the round that read it."""
        import torch.distributed as dist
        from .sharding import stage_slice
        B, P, D = chunk.shape
        rows = B * P
        flat = chunk.reshape(rows, D)
        per, lo, hi = stage_slice(rows, world, rank)
        dev = torch.device("cuda", self.device)
        ss = self.__dict__.get("_stage_stream")
        if ss is None:
            ss = self._stage_stream = torch.cuda.Stream(device=dev)
        part = self._shard_buf("part", slot, (per, D), torch.float32)
        full = self._shard_buf("full", slot, (per * world, D), torch.float32)
        with torch.cuda.stream(ss):
            if hi > lo:
                part[:hi - lo].copy_(flat[lo:hi], non_blocking=True)
            if hi - lo < per:
                part[hi - lo:].zero_()
            dist.all_gather_into_tensor(full, part, group=group)
            ev = torch.cuda.Event()
            ev.record(ss)
        lane.wait_event(ev)
        return full[:rows].view(B, P, D)

    def score_sharded_async(self, patches, feature_map_dims, out_hw=224, full=False, group=None, distribute=False,
                            img_base=0, phase_events=None):
        """One pipelined round (<= max_shard_batch() images) of row-sharded scoring with the replicated neighbour table
        (build_knn_sharded): min -> MIN all-reduce -> lookup -> SUM all-reduce -> finish, all enqueued on the handle's
        stream without waiting.  Returns a ticket; ticket.wait() -> BatchResult.  Three rounds may be outstanding, so the
        caller submits rounds k + 1 and k + 2 before waiting for round k.  Collective: every rank calls it with the same images.
        distribute: rank r runs the blur and the device->host copy only for the images i with (img_base + i) % world == r
        (the scalars of all images are replicated)."""
        import torch.distributed as dist
        assert getattr(self, "_knn_replicated", False), "call build_knn_sharded() first"
        patches = _as_f32(patches)
        B, P = patches.shape[0], patches.shape[1]
        assert B <= self.max_shard_batch()
        fh, fw = feature_map_dims
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        slot = self.__dict__.setdefault("_shard_round", 0) % 3   # staging buffers: one set per outstanding round
        self._shard_round += 1
        evs = phase_events
        lane = self.stream()   # the lane this round runs on (the finish call below hands the handle to the other lane)

        def mark():
            if evs is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record(lane)
                evs.append(e)

        self._order_after_producer(patches)
        # host-side allocations first: everything below is enqueued without waiting, and the GPU should not idle between
        # two phases while numpy allocates the result arrays
        res, outs, _ = self._alloc_out(B, P, out_hw, full)
        with torch.cuda.stream(lane):
            mark()
            chunk = patches
            if not chunk.is_cuda and world > 1 and B * P >= 1024:
                chunk = self._stage_sharded(chunk, slot, world, rank, group, lane)
            mark()
            first, stride = ((rank - img_base) % world, world) if distribute else (0, 1)
            if getattr(self, "_comm", None) is not None:
                # one call enqueues the whole round; the two exchanges run over peer-mapped memory inside the kernels
                ticket = ctypes.c_int64()
                L.check(self._lib.cmdb_score_shard_round_submit(self._h, _ptr(chunk), B, P, int(fh), int(fw), int(out_hw),
                                                                int(chunk.is_cuda), int(first), int(stride), 3 if full else 0,
                                                                ctypes.byref(ticket)))
                for _ in range(5):
                    mark()
                return _ShardTicket(self, ticket.value, (patches, chunk), res, outs, first, stride, B)
            keys = self._shard_buf("keys", slot, (B * P,), torch.int64)
            L.check(self._lib.cmdb_score_shard_min(self._h, _ptr(chunk), B, P, int(chunk.is_cuda), int(out_hw), _ptr(keys)))
            mark()
            dist.all_reduce(keys, op=dist.ReduceOp.MIN, group=group)
            mark()
            d2 = self._shard_buf("d2", slot, (B * 2,), torch.float32)
            L.check(self._lib.cmdb_score_shard_lookup(self._h, _ptr(keys), B, P, _ptr(d2)))
            mark()
            dist.all_reduce(d2, op=dist.ReduceOp.SUM, group=group)
            mark()
            ticket = ctypes.c_int64()
            L.check(self._lib.cmdb_score_shard_finish_submit(self._h, _ptr(d2), B, P, int(fh), int(fw), int(out_hw), int(first),
                                                             int(stride), 3 if full else 0, ctypes.byref(ticket)))
            mark()
        return _ShardTicket(self, ticket.value, patches, res, outs, first, stride, B)

    PHASES = ("stage", "local_min", "allreduce_min", "lookup", "allreduce_sum", "finish")

    def score_sharded_batch(self, patches, feature_map_dims, out_hw=224, full=False, group=None, distribute=False,
                            phase_events=None):
        """Row-sharded scoring: one process per GPU, each holding a contiguous block of bank rows; torch.distributed
        (NCCL over NVLink) collectives between the phases of include/cmdiad_b200.h.  Rounds of up to max_shard_batch()
        images go through score_sharded_async with two rounds kept in flight.  Collective: without a replicated
        neighbour table (build_knn_sharded) on this handle, the first call builds it.
        distribute=False: every rank returns all maps.  distribute=True: rank r finishes (blur, device->host) only images
        r, r+world, ... and returns None for the others.
        phase_events: optional list; gets one list of torch events per round, recorded on the handle's stream around the
        phases named in Bank.PHASES."""
        if not getattr(self, "_knn_replicated", False):
            self.build_knn_sharded(group)
        patches = _as_f32(patches)
        results = []
        step = self.max_shard_batch()
        pending = None
        for b0 in range(0, patches.shape[0], step):
            evs = [] if phase_events is not None else None
            t = self.score_sharded_async(patches[b0:b0 + step], feature_map_dims, out_hw, full, group, distribute, b0, evs)
            if phase_events is not None:
                phase_events.append(evs)
            if pending is not None:
                results.extend(pending.wait())
            pending = t
        if pending is not None:
            results.extend(pending.wait())
        return results


class _ShardTicket:
    """An outstanding score_sharded_async round (keeps inputs and result arrays alive until the results are fetched)."""

    def __init__(self, bank, ticket, patches, res, outs, first, stride, B):
        self._bank, self._ticket, self._patches = bank, ticket, patches
        self._res, self._outs, self._sub = res, outs, (first, stride, B)
        self._done = False

    def wait(self):
        if not self._done:
            L.check(self._bank._lib.cmdb_score_shard_wait(self._bank._h, self._ticket, self._outs))
            first, stride, B = self._sub
            if stride > 1:
                self._res.owned = set(range(first, B, stride))
            self._done, self._patches, self._outs = True, None, None
        return self._res


class _Ticket:
    """An outstanding score_batch_async call (keeps the input alive until the results are fetched)."""

    def __init__(self, bank, ticket, patches, B, P, out_hw, full):
        self._bank, self._ticket, self._patches = bank, ticket, patches
        self._shape = (B, P, out_hw, full)
        self._results = None

    def wait(self):
        if self._results is None:
            results, outs, _ = Bank._alloc_out(*self._shape)
            L.check(self._bank._lib.cmdb_score_batch_wait(self._bank._h, self._ticket, outs))
            self._results, self._patches = results, None
        return self._results


def upsample_blur(s_map, out_hw=224, device=0):
    """F.interpolate(bilinear) + KNNGaussianBlur(4) of a [fh,fw] float32 map (features.py:293-295)."""
    lib = L.load()
    m = np.ascontiguousarray(np.asarray(s_map, dtype=np.float32))
    fh, fw = m.shape
    out = np.zeros((out_hw, out_hw), np.float32)
    pre = np.zeros((out_hw, out_hw), np.float32)
    u8 = np.zeros((out_hw, out_hw), np.uint8)
    L.check(lib.cmdb_upsample_blur(int(device), _ptr(m), fh, fw, int(out_hw), _ptr(out), _ptr(pre), _ptr(u8)))
    return out, pre, u8


def coreset_rownorms(z, last, device=0):
    """One canonical-order distance pass ||z - last||_2 (float16 or float64 arrays), for parity pinning."""
    lib = L.load()
    z = np.ascontiguousarray(z)
    mode = L.CORESET_FP16 if z.dtype == np.float16 else L.CORESET_FP64
    last = np.ascontiguousarray(np.asarray(last, dtype=z.dtype).reshape(-1))
    out = np.zeros(z.shape[0], dtype=z.dtype)
    L.check(lib.cmdb_coreset_rownorms(int(device), _ptr(z), _ptr(last), z.shape[0], z.shape[1], mode, _ptr(out)))
    return out
