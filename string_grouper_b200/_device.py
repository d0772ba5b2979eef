"""Device-side plumbing: HBM containers (torch tensors) and the calls into libsg_b200.so.

PyTorch is used for device memory, streams and (in _dist.py) torch.distributed
only; every kernel on the hot path lives in csrc/*.cu behind the C ABI.
"""
import ctypes
from typing import NamedTuple

import numpy as np

from . import _lib

_TORCH = None

# hand-written kernels launched so far (CUB scans / sorts and memsets are not counted); bench.py "gpu_launches"
LAUNCH_COUNTS = {"postings": 0, "candidates": 0, "rescore": 0, "select": 0, "symmetrize": 0, "tfidf": 0,
                 "rowdot": 0, "order": 0, "tiles": 0, "groups": 0, "gather": 0, "prune": 0}
# "tiles": the tile-centric K2 (csrc/sg_tiles.cu): build, pack_left, filter, candidates

TRANSFER_BYTES = {"d2h": 0, "h2d": 0}      # bytes moved by the bulk copies (bench.py e2e accounting)

DEFAULT_WARPS = 8        # 8 warps x 5 CTAs at 48 registers (no spills)
GROUP_BYTES = 12 << 20   # posting bytes one column-tile group may hold
CAND_MARGIN = 1.5e-3   # candidates: fp16 posting weights (<= 4.9e-4) + fp32 accumulation; all are re-scored exactly
U16_MARGIN_PER_FEATURE = 2e-5   # 1/32768 fixed-point accumulator tile: one rounding of <= 2^-16 per added product
# Exact threshold pruning (csrc/sg_prune.cu): the most expensive heavy features of a left row are skipped while
# their norm times the largest right-row norm stays below PRUNE_FRAC * min_similarity.  0 switches it off.
PRUNE_FRAC = 0.9
ACC_DTYPE = "u16"               # accumulator tile: u16 | f32
MAX_CAND_DENSITY = 1.5e-3       # candidates per (row, column) pair
MAX_BUCKETS = 400_000_000       # directory entries (22 B each)
CAND_CHUNK = 1 << 28            # candidates per chunk of left rows
# up to this many (left row, right row) pairs the candidates kernel is launched without a sizing pass (see cossim_topn)
OPTIMISTIC_PAIRS = 5e11
REFINE = True                   # grouped per-candidate bound before the exact re-score
# K2 formulation: "row" (the default) = one warp per left row over L2-resident posting buckets (csrc/sg_cossim.cu; also
# the general path: negative values, norms above 1, near-zero thresholds); "tiles" = right tiles staged through TMA into
# shared memory (csrc/sg_tiles.cu), for L2-normalised non-negative operands.  Measured on B200 at 663k rows the row kernel
# is the faster one (DESIGN.md §4: both are bound by instruction issue at ~340 warp instructions per (row, tile) pair).
K2_KERNEL = "row"
TILE_MARGIN = 2e-5               # fp32 arithmetic of thresholds / norms and the f64 -> f32 copy of the values
TILE_MARGIN_PER_FEATURE = 3.1e-5  # a_q * w_q / 2^30 vs a * w: both weights rounded to nearest 2^-15 (<= 2^-15 + 2^-32)
SELECT_MODE = "rows"            # "rows" (per-row ranking) | "sort" (global sorts)


def torch():
    global _TORCH
    if _TORCH is None:
        import torch as _t
        _TORCH = _t
    return _TORCH


def require_cuda():
    t = torch()
    if not t.cuda.is_available():
        raise _lib.SgB200Error("string_grouper_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback "
                               "for the hot path")
    _lib.load()
    return t


def _ptr(x):
    return ctypes.c_void_p(0 if x is None else x.data_ptr())


def _stream():
    return ctypes.c_void_p(torch().cuda.current_stream().cuda_stream)


def _empty(n, dtype, device):
    return torch().empty(max(int(n), 1), dtype=dtype, device=device)


TIME_KERNELS = False      # bench.py: record CUDA events for the phases of every product (also through the public API)


def _timed(stats):
    return stats is not None and (stats.get("time_kernels") or TIME_KERNELS)


def mark(stats, name):
    """Phase boundary for bench.py `phases_ms`: a CUDA event on the current stream when stats["time_kernels"] is set."""
    if _timed(stats):
        ev = torch().cuda.Event(enable_timing=True)
        ev.record()
        stats.setdefault("marks", []).append((name, ev))


def phases_ms(stats):
    """{phase: milliseconds} from the marks of one step (the time between a mark and its predecessor is charged to
    the mark's name; the first mark only starts the clock)."""
    out = {}
    marks = stats.get("marks", [])
    for (_, e0), (name, e1) in zip(marks[:-1], marks[1:]):
        out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
    return out


def to_host(*tensors):
    """Device tensors -> numpy arrays through page-locked staging buffers (torch's caching host allocator
    re-uses them from call to call): all copies are queued on the current stream, one synchronisation.
    Pageable `.cpu()` copies run at a fraction of the PCIe rate and were the largest end-to-end cost."""
    t = torch()
    tensors = [x.contiguous() for x in tensors]
    TRANSFER_BYTES["d2h"] += sum(x.numel() * x.element_size() for x in tensors)
    try:
        outs = [t.empty(x.shape, dtype=x.dtype, pin_memory=bool(x.numel())) for x in tensors]
    except RuntimeError:          # page-locking refused (memlock limit): plain copies
        return [x.cpu().numpy() for x in tensors]
    for h, x in zip(outs, tensors):
        if x.numel():
            h.copy_(x, non_blocking=True)
    t.cuda.current_stream().synchronize()
    return [h.numpy() for h in outs]


class DeviceCSR:
    """CSR matrix resident in HBM: indptr int64, indices int32, val (matrix dtype), val32 (fp32 copy).

    Quacks like the scipy matrices StringGrouper._get_tf_idf_matrices returns
    (/root/reference/string_grouper/string_grouper.py:685-697): `.shape`,
    `.toarray()`, `.indptr` ... are served from a lazily materialised scipy
    copy, so reference-style tests and user code keep working.
    """

    def __init__(self, shape, indptr, indices, val, val32, nnz, dtype, norm_bound=1.0, base=0):
        self.shape = (int(shape[0]), int(shape[1]))
        # indptr holds ABSOLUTE positions into indices/val (a row-range view of a bigger matrix keeps
        # the parent's arrays and starts at `base`); the kernels never assume indptr[0] == 0.
        self.d_indptr, self.d_indices, self.d_val, self.d_val32 = indptr, indices, val, val32
        self.base = int(base)
        self.nnz = int(nnz)
        self.nnz_parent = int(nnz)     # stored values of the whole array a row-range view points into
        self.dtype = np.dtype(dtype)
        self.norm_bound = float(norm_bound)
        self._host = None
        self._order = None          # (hrank, perm, rank): rows ordered by (quantised heavy norm, heavy-feature signature)
        self._postings2 = {}
        self._tiles = None          # tile blobs of the tile-centric K2 (right_tiles)
        self.row_offset = None      # set when this matrix is one rank's block of rows of a sharded matrix
        self.global_rows = None
        self._df = None             # document frequency of every feature (sg_feature_df)
        self._heavy_norm = None     # per-row norm over the heavy features (sg_heavy_norms)
        self._heavy_groups = None   # the same per group of heavy ranks, fp16[16] (sg_rescore_refined)
        self.nonneg = True          # no negative stored value (K1 output; checked for uploaded matrices)

    @property
    def device(self):
        return self.d_indptr.device

    @classmethod
    def from_scipy(cls, m, device=None):
        t = require_cuda()
        from scipy.sparse import issparse
        if not issparse(m):
            raise TypeError("expected a scipy sparse matrix, got %r" % type(m))
        m = m.tocsr()
        if not m.has_sorted_indices:
            m = m.sorted_indices()
        if m.nnz >= 2**31 - 1:
            raise OverflowError("matrix has %d stored values; int32 indices overflow" % m.nnz)
        dtype = np.float32 if m.dtype == np.float32 else np.float64
        device = device or t.device("cuda", t.cuda.current_device())
        data = np.ascontiguousarray(m.data, dtype=dtype)
        indptr = t.from_numpy(np.ascontiguousarray(m.indptr, dtype=np.int64)).to(device)
        indices = t.from_numpy(np.ascontiguousarray(m.indices, dtype=np.int32)).to(device)
        val = t.from_numpy(data).to(device)
        val32 = val if dtype == np.float32 else val.to(t.float32)
        bound = float(np.sqrt(m.multiply(m).sum(axis=1).max())) if m.nnz else 1.0
        out = cls(m.shape, indptr, indices, val, val32, m.nnz, dtype, max(bound, 1e-30))
        out._host = m
        out.nonneg = bool(m.nnz == 0 or data.min() >= 0)
        return out

    def to_scipy(self):
        if self._host is None:
            from scipy.sparse import csr_matrix
            lo, hi = self.base, self.base + self.nnz
            indptr = self.d_indptr[:self.shape[0] + 1].cpu().numpy() - lo
            idx_dtype = np.int32 if max(self.shape) < 2**31 and self.nnz < 2**31 else np.int64
            self._host = csr_matrix((self.d_val[lo:hi].cpu().numpy(),
                                     self.d_indices[lo:hi].cpu().numpy().astype(idx_dtype),
                                     indptr.astype(idx_dtype)), shape=self.shape)
        return self._host

    def get_shape(self):
        return self.shape

    def toarray(self):
        return self.to_scipy().toarray()

    def __getitem__(self, key):
        return self.to_scipy()[key]

    def __matmul__(self, other):
        return self.to_scipy() @ (other.to_scipy() if hasattr(other, "to_scipy") else other)

    def __getattr__(self, name):
        # the scipy face: only the attributes below materialise the host copy (a typo or a probing hasattr() must not
        # trigger a device-to-host copy of the whole matrix)
        if name in _SCIPY_CSR_ATTRS:
            return getattr(self.to_scipy(), name)
        raise AttributeError("%s has no attribute %r" % (type(self).__name__, name))


# what callers of StringGrouper._get_tf_idf_matrices / _build_matches use on the returned scipy matrices
_SCIPY_CSR_ATTRS = frozenset([
    "indptr", "indices", "data", "T", "transpose", "multiply", "dot", "tocsr", "tocsc", "tocoo", "tolil", "todense",
    "nonzero", "sum", "max", "min", "mean", "getrow", "getcol", "diagonal", "astype", "copy", "getnnz", "has_sorted_indices",
    "sort_indices", "sorted_indices", "format", "ndim", "count_nonzero", "power", "maximum", "minimum", "A", "todok",
    "eliminate_zeros", "sum_duplicates", "asformat", "conj", "conjugate", "getH", "setdiag", "trace", "tobsr", "todia"])


def as_device_csr(m):
    return m if isinstance(m, DeviceCSR) else DeviceCSR.from_scipy(m)


def heavy_features(B):
    """int8 rank of every feature among the 64 most frequent ones of B (-1 otherwise)."""
    t = require_cuda()
    L = _lib.load()
    n_rows, n_cols = B.shape
    hrank = _empty(n_cols, t.int8, B.device)
    ws_bytes = int(L.sg_order_workspace_bytes(n_rows, n_cols))
    ws = _empty(ws_bytes, t.uint8, B.device)
    _lib.check(L.sg_heavy_features(n_rows, n_cols, _ptr(B.d_indptr), _ptr(B.d_indices), _ptr(feature_df(B)), 64,
                                   _ptr(hrank), _ptr(ws), ws_bytes, _stream()))
    LAUNCH_COUNTS["order"] += 3
    return hrank


def heavy_norms(M, hrank, row_begin=0, row_end=None, groups=False):
    """fp32 norm of rows [row_begin,row_end) of M over the heavy features, rounded up (sg_heavy_norms); with
    `groups` also the fp16 norms per group of heavy ranks (16 per row, csrc/sg_prune.cu): (norm, group_norms)."""
    t = require_cuda()
    L = _lib.load()
    row_end = M.shape[0] if row_end is None else row_end
    n = max(row_end - row_begin, 0)
    out = _empty(n, t.float32, M.device)
    grp = _empty(16 * n, t.float16, M.device) if groups else None
    _lib.check(L.sg_heavy_norms(row_begin, row_end, _ptr(M.d_indptr), _ptr(M.d_indices), _ptr(M.d_val32),
                                _ptr(hrank), _ptr(out), _ptr(grp), _stream()))
    LAUNCH_COUNTS["prune"] += 1
    return (out, grp) if groups else out


def row_order(M, hrank, row_begin=0, row_end=None, want_rank=True, row_norm=None, norm_scale=1.0):
    """(perm, rank) of rows [row_begin,row_end) of M sorted by (quantised heavy norm,) heavy-feature signature."""
    t = require_cuda()
    L = _lib.load()
    row_end = M.shape[0] if row_end is None else row_end
    n = max(row_end - row_begin, 0)
    perm = _empty(n, t.int32, M.device)
    rank = _empty(n, t.int32, M.device) if want_rank else None
    ws_bytes = int(L.sg_order_workspace_bytes(max(n, 1), M.shape[1]))
    ws = _empty(ws_bytes, t.uint8, M.device)
    _lib.check(L.sg_row_order(row_begin, row_end, _ptr(M.d_indptr), _ptr(M.d_indices), _ptr(hrank), _ptr(row_norm),
                              float(norm_scale), _ptr(perm), _ptr(rank), _ptr(ws), ws_bytes, _stream()))
    LAUNCH_COUNTS["order"] += 2
    return perm, rank


def right_order(B):
    """(hrank, perm, rank) of the right matrix: heavy features, rows sorted by (quantised heavy norm, signature)."""
    if B._order is None:
        hrank = heavy_features(B)
        B._heavy_norm, B._heavy_groups = heavy_norms(B, hrank, groups=True)
        perm, rank = row_order(B, hrank, row_norm=B._heavy_norm, norm_scale=1.0 / max(B.norm_bound, 1e-30))
        B._order = (hrank, perm, rank)
    return B._order


def _tile_bounds(B, perm, tile_w):
    """Largest heavy norm of B's rows per column tile of `tile_w` rows of the processing order `perm`
    (sg_tile_bounds): the per-tile pruning bound."""
    t = torch()
    L = _lib.load()
    bound = t.zeros(int(L.sg_num_tiles_padded(B.shape[0], tile_w)), dtype=t.float32, device=B.device)
    _lib.check(L.sg_tile_bounds(B.shape[0], _ptr(perm), _ptr(B._heavy_norm), tile_w, _ptr(bound), _stream()))
    LAUNCH_COUNTS["prune"] += 1
    return bound


def right_tiles(B):
    """Tile blobs of the tile-centric K2 (csrc/sg_tiles.cu), cached on B: per 256-row tile of the processing order
    the postings sorted by feature, the bitmap directory and the bucket offsets as one blob (what the candidates
    kernel stages through TMA), the fp16 block maxima of every (feature, tile), the per-tile pruning bound and the
    bytes the kernel stages per tile (read back once)."""
    t = require_cuda()
    L = _lib.load()
    hrank, perm, rank = right_order(B)
    if B._tiles is None:
        n_rows, n_cols = B.shape
        W = int(L.sg_tiles_tile_w())
        T = int(L.sg_num_tiles(n_rows, W))
        Tp = int(L.sg_num_tiles_padded(n_rows, W))
        cap = int(L.sg_tiles_blob_bound(B.nnz, n_rows, n_cols))
        blob = _empty(cap, t.uint8, B.device)
        desc = _empty(2 * T, t.int64, B.device)
        maxw = _empty((n_cols + 1) * Tp, t.float16, B.device)
        maxima = t.zeros(2, dtype=t.int32, device=B.device)
        ws_bytes = int(L.sg_tiles_workspace_bytes(B.nnz, n_rows, n_cols))
        ws = _empty(ws_bytes, t.uint8, B.device)
        _lib.check(L.sg_tiles_build(n_rows, n_cols, B.nnz, _ptr(B.d_indptr), _ptr(B.d_indices), _ptr(B.d_val32),
                                    _ptr(rank), B.base, 1.0 / max(B.norm_bound, 1.0), _ptr(desc), _ptr(blob), cap,
                                    _ptr(maxw), _ptr(maxima), _ptr(ws), ws_bytes, _stream()))
        LAUNCH_COUNTS["tiles"] += 4
        bound = _tile_bounds(B, perm, W)
        B._tiles = {"desc": desc, "blob": blob, "maxw": maxw, "bound": bound, "maxima": maxima, "T": T, "W": W,
                    "stage_bytes": int(maxima[0].item())}
    return B._tiles


def right_side(B, tile_w):
    """Row order (heavy norm, signature), feature-major bucketed postings, bucket directory with block maxima and
    per-tile pruning bounds of the right matrix, cached on B."""
    t = require_cuda()
    L = _lib.load()
    hrank, perm, rank = right_order(B)
    if tile_w not in B._postings2:
        n_rows, n_cols = B.shape
        T = int(L.sg_num_tiles(n_rows, tile_w))
        nb = T * (n_cols + 1) + 1
        if nb >= 2**31 - 1:
            raise OverflowError("posting bucket table too large: %d features x %d tiles" % (n_cols, T))
        Tp = int(L.sg_num_tiles_padded(n_rows, tile_w))
        bucket_ptr = _empty(nb, t.int32, B.device)
        bucket_dir = _empty(2 * nb, t.int32, B.device)
        bucket_maxw = _empty((n_cols + 1) * Tp, t.float16, B.device)
        post = _empty(max(B.nnz, 1), t.int32, B.device)
        ws_bytes = int(L.sg_postings_workspace_bytes(B.nnz, n_cols, T))
        ws = _empty(ws_bytes, t.uint8, B.device)
        _lib.check(L.sg_postings_build(n_rows, n_cols, B.nnz, _ptr(B.d_indptr), _ptr(B.d_indices), _ptr(B.d_val32),
                                       _ptr(rank), tile_w, B.base, 1.0 / max(B.norm_bound, 1.0), _ptr(bucket_ptr),
                                       _ptr(bucket_dir), _ptr(bucket_maxw), _ptr(post),
                                       _ptr(ws), ws_bytes, _stream()))
        LAUNCH_COUNTS["postings"] += 4
        bound = _tile_bounds(B, perm, tile_w)
        B._postings2[tile_w] = (bucket_dir, bucket_maxw, post, T, bound)     # bucket_ptr is only needed for the build
    return (hrank, perm, rank) + B._postings2[tile_w]


class DeviceMatches:
    """Result of the top-n product in HBM: COO triples ordered by (row asc, score desc)
    or, after symmetrize(), by (row asc, col asc).  Lazily materialises the scipy CSR that
    StringGrouper._build_matches returns in the reference (string_grouper.py:709-752)."""

    def __init__(self, shape, row, col, score, nnz, max_row, out_dtype=np.float64, indptr=None):
        self.shape = (int(shape[0]), int(shape[1]))
        self.d_row, self.d_col, self.d_score, self.d_indptr = row, col, score, indptr
        self.nnz = int(nnz)
        self.max_row = int(max_row)
        self.out_dtype = np.dtype(out_dtype)
        self._host = None
        self.pending_fix_diagonal = False
        self.pending_mirror = False

    def with_pending(self, fix_diagonal=False, mirror=False):
        """Record a post-processing step (StringGrouper._fix_diagonal / _symmetrize_matrix); the fused K4
        launch happens in apply_pending()."""
        self.pending_fix_diagonal |= bool(fix_diagonal)
        self.pending_mirror |= bool(mirror)
        return self

    def host_triples(self):
        """(row int64, col int64, score f64) on the host; the widening to the reference's int64 columns
        (string_grouper.py:759-763) happens on the device."""
        n = self.nnz
        t = torch()
        return tuple(to_host(self.d_row[:n].to(t.int64), self.d_col[:n].to(t.int64), self.d_score[:n]))

    def to_scipy(self):
        if self._host is None:
            from scipy.sparse import csr_matrix
            r, c, s = self.host_triples()
            indptr = np.zeros(self.shape[0] + 1, dtype=np.int64)
            np.cumsum(np.bincount(r, minlength=self.shape[0]), out=indptr[1:])
            idx_dtype = np.int32 if max(self.shape) < 2**31 and self.nnz < 2**31 else np.int64
            self._host = csr_matrix((s.astype(self.out_dtype, copy=False), c.astype(idx_dtype),
                                     indptr.astype(idx_dtype)), shape=self.shape)
        return self._host

    def get_shape(self):
        return self.shape

    def toarray(self):
        return self.to_scipy().toarray()

    def __getattr__(self, name):
        if name in _SCIPY_CSR_ATTRS:
            return getattr(self.to_scipy(), name)
        raise AttributeError("%s has no attribute %r" % (type(self).__name__, name))

    # operators scipy matrices answer; they materialise the host copy like the attributes above
    def __getitem__(self, key):
        return self.to_scipy()[key]

    def __matmul__(self, other):
        return self.to_scipy() @ other

    def __sub__(self, other):
        return self.to_scipy() - (other.to_scipy() if hasattr(other, "to_scipy") else other)

    def __ne__(self, other):
        return self.to_scipy() != (other.to_scipy() if hasattr(other, "to_scipy") else other)

    __hash__ = object.__hash__


def pick_tile(n_right, tile_w=None, warps=None, acc_bytes=4, n_left=None):
    """Column-tile width and warps per CTA.  Default: 512-byte accumulator tiles (256 columns of 16-bit fixed
    point): narrow tiles make the block-max test skip most (row, tile) pairs, and the test itself costs a
    fraction of an instruction per pair."""
    warps = int(warps or DEFAULT_WARPS)
    # measured on B200 (profiles/r2_notes.md): 128-column tiles win from a few 10^5 right rows on (the block-max test
    # skips more, 34.5 vs 38.0 ms at 663k), 256-column tiles below (1.4 vs 1.8 ms at 100k: fewer directory entries)
    # (the finer directory costs ~0.6 ms more to build: not worth it for a small block of left rows, e.g. one of 8 shards)
    many_left = n_left is None or int(n_left) >= 150_000
    auto_w = 128 if (acc_bytes == 4 or (int(n_right) >= 400_000 and many_left)) else 256
    tile_w = int(tile_w or auto_w)
    q = 256 // acc_bytes                               # tile bytes must be a multiple of 256
    need = ((max(int(n_right), 1) + q - 1) // q) * q
    tile_w = max(q, min(tile_w, 32768) // q * q)
    return min(tile_w, need), warps


def k2_accumulator(acc, threshold, scale, nonneg):
    """(accumulator tile, candidate threshold) of K2: the tile the caller asked for (default ACC_DTYPE) and
    threshold - CAND_MARGIN * max(scale, 1) clamped at 0.  `scale` bounds every score (the product of the operands'
    largest row norms); `nonneg`: no negative stored value in either operand."""
    thr_c = max(float(threshold) - CAND_MARGIN * max(scale, 1.0), 0.0)
    acc = (acc or ACC_DTYPE).lower()
    if acc not in ("u16", "f32"):
        raise ValueError("accumulator dtype must be 'u16' or 'f32', got %r" % (acc,))
    # fixed-point accumulator tiles need non-negative weights and scores below 2 (K1's L2-normalised rows); also
    # near-zero thresholds take fp32: a tiny positive score must not round to a fixed-point zero
    if not (nonneg and scale <= 1.0 + 1e-6) or thr_c < 0.05:
        acc = "f32"
    return acc, thr_c


class K2Plan(NamedTuple):
    """What cossim_topn decides before its first candidates launch (plan_k2)."""
    kernel: str              # "row" (csrc/sg_cossim.cu) | "tiles" (csrc/sg_tiles.cu)
    acc: str                 # accumulator tile: "u16" | "f32"
    margin: float            # score error of the candidate traversal ...
    margin_pf: float         # ... plus this much per kept feature of the left row (fixed-point products)
    thr_c: float             # candidate threshold
    tile_w: int              # columns per tile
    warps: int               # warps per CTA
    tiles_per_group: int     # column tiles per work group of the row kernel (0: tile formulation)
    refine: bool             # candidates carry their partial score; sg_rescore_refined re-tests them first
    levels: tuple            # pruning levels, in the order they are tried
    whole_range: bool        # one launch over every row at levels[0] before any sizing pass
    sample_stride: int       # every stride-th row of the processing order sizes the buffers (None: no sample)
    cand_limit: float        # a lower pruning level is tried above this many candidates (MAX_CAND_DENSITY)


def plan_k2(n_rows, n_right, n_cols, nnz_right, threshold, scale=1.0, nonneg=True, kernel=None, acc=None, prune=None,
            tile_w=None, warps=None, tile_fit=None):
    """K2's decisions for `n_rows` left rows against a right matrix of n_right x n_cols with nnz_right stored values;
    the arguments after `nonneg` are those of cossim_topn.

    tile_fit: (tile width, shared memory the tile kernel needs at 8 warps, the device's opt-in shared memory per
    block) of the right matrix's tile blobs (right_tiles); cossim_topn builds them only when the tile formulation is
    asked for, the fixed-point accumulator applies and the bitmap directory holds every feature.  Without it, or
    when the stage does not fit shared memory, the row kernel runs."""
    acc, thr_c = k2_accumulator(acc, threshold, scale, nonneg)
    kernel = (kernel or K2_KERNEL).lower()
    if kernel not in ("tiles", "row"):
        raise ValueError("kernel must be 'tiles' or 'row', got %r" % (kernel,))
    if kernel == "tiles" and acc == "u16" and tile_fit is not None and tile_fit[1] <= tile_fit[2]:
        margin, margin_pf = TILE_MARGIN * max(scale, 1.0), TILE_MARGIN_PER_FEATURE
        tile_w, warps, tiles_per_group = tile_fit[0], 8, 0
    else:
        kernel, margin = "row", CAND_MARGIN * max(scale, 1.0)
        margin_pf = U16_MARGIN_PER_FEATURE if acc == "u16" else 0.0
        tile_w, warps = pick_tile(n_right, tile_w, warps, 2 if acc == "u16" else 4, n_left=n_rows)
        # the bucket directory holds one entry per (feature, tile): widen the tiles until it stays below MAX_BUCKETS
        while (-(-n_right // tile_w)) * (n_cols + 1) > MAX_BUCKETS and tile_w < 32768:
            tile_w *= 2
        n_tiles = -(-n_right // tile_w)
        # column tiles per work group (a multiple of 64): the group's posting buckets should stay L2-resident
        tiles_per_group = max(64, int(GROUP_BYTES // max(4 * nnz_right / n_tiles, 1)) // 64 * 64)
    # when the caller left the pruning level open it may be lowered (see _size_candidates)
    level = PRUNE_FRAC if prune is None else float(prune)
    levels = (level,)
    if prune is None and level > 0.0 and thr_c > 0.0:
        levels = (level, 0.75 * level, 0.5 * level, 0.25 * level, 0.0)
    return K2Plan(kernel=kernel, acc=acc, margin=margin, margin_pf=margin_pf, thr_c=thr_c, tile_w=tile_w, warps=warps,
                  tiles_per_group=tiles_per_group, refine=REFINE and kernel == "row" and acc == "u16", levels=levels,
                  whole_range=float(n_rows) * float(n_right) <= OPTIMISTIC_PAIRS,
                  sample_stride=max(64, n_rows // 8192) if n_rows >= 65536 else None,
                  cand_limit=MAX_CAND_DENSITY * n_rows * n_right)


def row_chunks(n_rows, est):
    """(chunks, rows per chunk): slices of the processing order whose candidates, `est` for all rows with 30 %
    headroom, fit CAND_CHUNK entries; one chunk without an estimate."""
    n_chunks = 1 if est is None else max(1, -(-int(1.3 * est) // CAND_CHUNK))
    return n_chunks, -(-n_rows // n_chunks)


def chunk_capacity(n_rows, rows, est):
    """Candidate buffer entries for a chunk of `rows` of the `n_rows` left rows, `est` candidates expected for all of
    them.  Without an estimate a guess: clusters of identical names make the candidates much more than top_n per row
    (37 M for the 663k benchmark corpus); a chunk that overflows is launched again with the exact count."""
    if est is None:
        return min(96 * n_rows + (1 << 22), 1 << 30)
    return min(int(1.3 * est * rows / n_rows) + (1 << 22), 1 << 31)


def select_mode(top_n, max_row_cnt, rows_cap):
    """"rows": survivors bucketed by row, every row ranked on its own (warp shuffle network, or one CTA in shared
    memory for up to `rows_cap` = sg_topn_rows_cap() survivors, longer rows in pieces while top_n <= rows_cap / 2);
    "sort": three global radix sorts.  `max_row_cnt`: survivors of the longest row."""
    if SELECT_MODE != "sort" and (top_n <= 32 or max_row_cnt <= rows_cap or top_n <= rows_cap // 2):
        return "rows"
    return "sort"


def feature_df(B):
    """int32 document frequency of every feature of B (cached): the postings walked per use of the feature."""
    if B._df is None:
        t = require_cuda()
        L = _lib.load()
        df = _empty(B.shape[1], t.int32, B.device)
        _lib.check(L.sg_feature_df(B.shape[0], B.shape[1], _ptr(B.d_indptr), _ptr(B.d_indices), _ptr(df), _stream()))
        LAUNCH_COUNTS["prune"] += 1
        B._df = df
    return B._df


def prune_left(A, B, hrank, row_begin, row_end, threshold, margin, margin_per_feature, frac):
    """Exact threshold pruning of rows [row_begin,row_end) of A against B (sg_prune_rows); only B's heavy
    features (hrank >= 0) are prunable.  Returns (indices, val32, row_len, row_threshold, pruned_norm,
    pruned_group_norms) device arrays indexed like A's own."""
    t = require_cuda()
    L = _lib.load()
    df = feature_df(B)
    p_idx = t.empty_like(A.d_indices)
    p_val = t.empty_like(A.d_val32)
    p_len = _empty(A.shape[0], t.int32, A.device)
    p_thr = _empty(A.shape[0], t.float32, A.device)
    p_xp = _empty(A.shape[0], t.float32, A.device)
    p_xg = _empty(16 * A.shape[0], t.float16, A.device)     # |x_P| per group of heavy ranks
    budget = max(float(frac) * (float(threshold) - margin), 0.0)
    # the kernel works on left weights as stored and right rows of norm <= B.norm_bound
    _lib.check(L.sg_prune_rows(row_begin, row_end, _ptr(A.d_indptr), _ptr(A.d_indices), _ptr(A.d_val32), _ptr(df),
                               _ptr(hrank), float(B.norm_bound), budget, float(threshold), float(margin),
                               float(margin_per_feature), _ptr(p_idx), _ptr(p_val), _ptr(p_len), _ptr(p_thr),
                               _ptr(p_xp), _ptr(p_xg), _stream()))
    LAUNCH_COUNTS["prune"] += 1
    return p_idx, p_val, p_len, p_thr, p_xp, p_xg


def cossim_topn(A, B, top_n, threshold, row_begin=0, row_end=None, tile_w=None, warps=None, stats=None,
                prune=None, acc=None, kernel=None):
    """C[i,:] = top_n{ j : A_i . B_j > threshold } for rows [row_begin,row_end) of A.

    Device counterpart of the whole block loop of StringGrouper._build_matches
    (string_grouper.py:734-750).  Returns DeviceMatches with absolute row ids.
    """
    t = require_cuda()
    if A.shape[1] != B.shape[1]:
        raise ValueError("dimension mismatch: left has %d features, right has %d" % (A.shape[1], B.shape[1]))
    if A.dtype != B.dtype:
        raise TypeError("left and right matrices must have the same dtype")
    n_left, n_right = A.shape[0], B.shape[0]
    row_end = n_left if row_end is None else int(row_end)
    row_begin = int(row_begin)
    n_rows = max(row_end - row_begin, 0)
    top_n = int(min(int(top_n), n_right))
    if n_rows == 0 or n_right == 0 or top_n <= 0 or A.nnz == 0 or B.nnz == 0:
        z32 = _empty(1, t.int32, A.device)
        return DeviceMatches((n_left, n_right), z32, z32, _empty(1, t.float64, A.device), 0, 0)

    mark(stats, "k2_start")
    plan = _plan(A, B, n_rows, threshold, kernel, acc, prune, tile_w, warps)
    k = _K2Call(A, B, row_begin, row_end, threshold, plan)
    mark(stats, "right_side")
    survivors = _candidates_rescored(k, stats)
    if stats is not None:
        stats["tile_w"], stats["warps"], stats["n_tiles"] = plan.tile_w, plan.warps, k.n_tiles
        stats["tiles_per_group"] = plan.tiles_per_group
        if plan.kernel == "tiles":
            stats["stage_bytes"] = k.tiles["stage_bytes"]
    return _select(k, top_n, *survivors, stats)


def _plan(A, B, n_rows, threshold, kernel, acc, prune, tile_w, warps):
    """plan_k2 for one call.  The tile formulation's fit check needs its blobs: they are built here when it may run."""
    t = torch()
    L = _lib.load()
    scale, nonneg = A.norm_bound * B.norm_bound, A.nonneg and B.nonneg
    tile_fit = None
    if ((kernel or K2_KERNEL).lower() == "tiles" and k2_accumulator(acc, threshold, scale, nonneg)[0] == "u16"
            and B.shape[1] <= int(L.sg_tiles_max_cols())):
        tiles = right_tiles(B)
        tile_fit = (tiles["W"], int(L.sg_tiles_smem_bytes(tiles["stage_bytes"], 8)),
                    t.cuda.get_device_properties(A.device).shared_memory_per_block_optin)
    return plan_k2(n_rows, B.shape[0], B.shape[1], B.nnz, threshold, scale, nonneg, kernel=kernel, acc=acc,
                   prune=prune, tile_w=tile_w, warps=warps, tile_fit=tile_fit)


class _K2Call:
    """Device arrays of one cossim_topn call: the right side in the plan's formulation (`tiles`, or the row kernel's
    bucket directory, block maxima and postings), both operands' processing orders and the counters the kernels
    report through ([0] candidates / survivors, [1] work queue / longest row, [2] pairs walked / refined candidates,
    [3] postings walked)."""

    def __init__(self, A, B, row_begin, row_end, threshold, plan):
        t = torch()
        self.A, self.B, self.plan, self.threshold = A, B, plan, float(threshold)
        self.row_begin, self.row_end, self.n_rows = row_begin, row_end, row_end - row_begin
        self.counters = t.zeros(4, dtype=t.int64, device=A.device)
        # both operands in the same processing order (quantised heavy norm, heavy-feature signature): neighbouring left
        # rows stream the same buckets, and the rows of a column tile have similar heavy norms (tight per-tile bound)
        if plan.kernel == "tiles":
            self.tiles = right_tiles(B)
            self.hrank, self.perm_b, _ = right_order(B)
            self.n_tiles, self.tile_bound = self.tiles["T"], self.tiles["bound"]
            self.lpack = _empty(2 * A.d_indices.numel(), t.int32, A.device)
        else:
            (self.hrank, self.perm_b, _, self.bucket_dir, self.bucket_maxw, self.post, self.n_tiles,
             self.tile_bound) = right_side(B, plan.tile_w)
        if A is B and row_begin == 0 and row_end == A.shape[0]:
            self.perm_a = self.perm_b
        else:
            self.perm_a, _ = row_order(A, self.hrank, row_begin, row_end, want_rank=False)

    def counter(self, i):
        return ctypes.c_void_p(self.counters.data_ptr() + 8 * i)


def _prune(k, level):
    """The call's left rows pruned at `level` (prune_left; the fixed-point tile always takes per-row thresholds: its
    margin grows with the number of features added), or A's own arrays when neither applies."""
    p = k.plan
    if (level > 0.0 and p.thr_c > 0.0) or p.margin_pf > 0.0:
        return prune_left(k.A, k.B, k.hrank, k.row_begin, k.row_end, k.threshold, p.margin, p.margin_pf,
                          level if p.thr_c > 0.0 else 0.0)
    return k.A.d_indices, k.A.d_val32, None, None, None, None


def _launch_candidates(k, pruned, perm, n, row_buf, col_buf, capacity, partial_buf=None):
    """Candidates of the left rows perm[:n] into (row_buf, col_buf, partial_buf)[:capacity]; counters[0] = their
    number, which may exceed `capacity`."""
    t = torch()
    L = _lib.load()
    A, B, p = k.A, k.B, k.plan
    l_idx, l_val, l_len, l_thr, l_xp, _ = pruned
    if p.kernel == "tiles":
        # pack the pruned rows of `perm`, block-max filter -> survivor bits, tile kernel
        stride = (n + 31) // 32 * 32
        rowinfo = _empty(4 * stride, t.int32, A.device)
        mask = _empty(int(L.sg_tiles_mask_words(B.shape[0])) * stride, t.int32, A.device)
        k.counters.zero_()
        _lib.check(L.sg_tiles_pack_left(n, _ptr(perm), 0, _ptr(A.d_indptr), _ptr(l_len), _ptr(l_idx), _ptr(l_val),
                                        _ptr(l_thr), _ptr(l_xp), max(B.norm_bound, 1.0), _ptr(k.lpack),
                                        _ptr(rowinfo), _stream()))
        _lib.check(L.sg_tiles_filter(n, _ptr(rowinfo), _ptr(k.lpack), _ptr(k.tiles["maxw"]), B.shape[0],
                                     _ptr(k.tile_bound), _ptr(mask), stride, _stream()))
        _lib.check(L.sg_tiles_candidates(_ptr(perm), n, 0, _ptr(rowinfo), _ptr(k.lpack), _ptr(mask), stride,
                                         _ptr(k.tiles["desc"]), _ptr(k.tiles["blob"]), B.shape[0], B.shape[1],
                                         _ptr(k.tile_bound), _ptr(k.perm_b), k.tiles["stage_bytes"], _ptr(row_buf),
                                         _ptr(col_buf), capacity, k.counter(0), k.counter(1), k.counter(2), p.warps,
                                         _stream()))
        LAUNCH_COUNTS["tiles"] += 3
        return
    k.counters.zero_()
    _lib.check(L.sg_cossim_candidates(
        _ptr(A.d_indptr), _ptr(l_len), _ptr(l_idx), _ptr(l_val), k.row_begin, k.row_begin + n, _ptr(perm),
        B.shape[0], A.shape[1], _ptr(k.bucket_dir), _ptr(k.bucket_maxw), _ptr(k.post), _ptr(k.perm_b), p.tile_w,
        _lib.SG_ACC_U16 if p.acc == "u16" else _lib.SG_ACC_F32, max(B.norm_bound, 1.0),
        p.thr_c, _ptr(l_thr), _ptr(l_xp), _ptr(k.tile_bound), p.tiles_per_group, _ptr(row_buf), _ptr(col_buf),
        _ptr(partial_buf), capacity, k.counter(0), k.counter(1), p.warps, _stream()))
    LAUNCH_COUNTS["candidates"] += 1


def _cand_buffers(k, capacity):
    """(rows, columns, partial scores | None) of `capacity` candidates."""
    t = torch()
    dev = k.A.device
    return (_empty(capacity, t.int32, dev), _empty(capacity, t.int32, dev),
            _empty(capacity, t.float32, dev) if k.plan.refine else None)


def _timed_candidates(k, pruned, perm, n, bufs, capacity, stats):
    """A candidates launch that produces candidates (sizing passes do not): timed for bench.py's kernel time, the
    walk counters of the tile kernel added to stats.  Returns the number of candidates."""
    t = torch()
    if _timed(stats):
        ev0, ev1 = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
        ev0.record()
    _launch_candidates(k, pruned, perm, n, bufs[0], bufs[1], capacity, bufs[2])
    if _timed(stats):
        ev1.record()
        stats.setdefault("candidate_events", []).append((ev0, ev1))
    head = k.counters[:4].cpu().numpy()
    if k.plan.kernel == "tiles" and stats is not None:
        stats["pairs_walked"] = stats.get("pairs_walked", 0) + int(head[2])
        stats["postings_walked"] = stats.get("postings_walked", 0) + int(head[3])
    return int(head[0])


def _size_candidates(k, stats):
    """Pruning level and candidate buffers of the call: (level, pruned rows at that level, candidate estimate | None,
    (rows, columns, partial scores, count) of a whole-range launch that already holds every candidate | None).

    Every candidate costs an exact re-score and every skipped posting saves one update, so with several levels
    (plan.levels) the level is lowered while the candidates exceed plan.cand_limit.  Three strategies:
      1. whole range (plan.whole_range): a sizing pass is latency-bound (a few thousand rows against every column
         tile, cold: 2-3 ms whatever the shard) while a wasted launch over a moderate range costs no more than a few
         tens of ms.  So all rows are launched at the first level into buffers of the density limit.  When their
         candidates fit and are not too many, that is the answer; when they overflow the buffers without exceeding the
         limit, the exact count is the estimate at this level; when they exceed the limit, the sample search below
         goes on from the next level.
      2. sample (plan.sample_stride): a counting pass over every stride-th row of the processing order (clusters of
         identical names are sampled in proportion) per level, down the levels until the estimate is within the limit.
      3. neither: the first level and no estimate; the chunk loop sizes its buffer from the row count."""
    p = k.plan
    levels = p.levels
    sample = k.perm_a[:k.n_rows:p.sample_stride].contiguous() if p.sample_stride else None
    dummy = _empty(1, torch().int32, k.A.device)          # the counting pass stores no candidate
    if p.whole_range:
        pruned = _prune(k, levels[0])
        capacity = int(min(int(p.cand_limit) + (1 << 22), CAND_CHUNK))
        bufs = _cand_buffers(k, capacity)
        mark(stats, "prune_sample")
        n = _timed_candidates(k, pruned, k.perm_a, k.n_rows, bufs, capacity, stats)
        mark(stats, "candidates")
        too_dense = len(levels) > 1 and sample is not None and n > p.cand_limit
        if n <= capacity and not too_dense:
            return levels[0], pruned, None, bufs + (n,)
        del bufs
        if _timed(stats):
            stats["wasted_launch"] = True
        if not too_dense:
            return levels[0], pruned, n, None
        levels = levels[1:]
    est = None
    for level in levels:
        pruned = _prune(k, level)
        if sample is None:
            break
        _launch_candidates(k, pruned, sample, int(sample.numel()), dummy, dummy, 0)
        est = int(k.counters[0].item()) * p.sample_stride
        if est <= p.cand_limit:
            break
    return level, pruned, est, None


def _count_macs(k, pruned):
    """(postings of B the kept features of the pruned left rows walk, kept features): stats["count_macs"]."""
    t = torch()
    A, n_left = k.A, k.A.shape[0]
    l_idx, _, l_len = pruned[:3]
    df = feature_df(k.B).long()
    pos = t.arange(A.d_indices.numel(), device=A.device)
    rid = t.searchsorted(A.d_indptr[:n_left + 1].contiguous(), pos, right=True) - 1
    ok = (rid >= k.row_begin) & (rid < k.row_end)
    rid = rid.clamp(0, n_left - 1)
    live = ok & ((pos - A.d_indptr[rid]) < l_len[rid].long())
    return int(df[l_idx.long().clamp(0, A.shape[1] - 1)][live].sum().item()), int(live.sum().item())


def _chunk_candidates(k, pruned, perm, n, capacity, stats):
    """(rows, columns, partial scores, count) of the candidates of the left rows perm[:n]; buffers that overflow are
    allocated again with the exact count."""
    for attempt in range(3):
        bufs = _cand_buffers(k, capacity)
        n_cand = _timed_candidates(k, pruned, perm, n, bufs, capacity, stats)
        if n_cand <= capacity:
            return bufs + (n_cand,)
        if n_cand * 24 > 96 * 2**30:
            raise OverflowError("%d candidate pairs above the threshold do not fit the candidate buffer; "
                                "raise min_similarity or split the input" % n_cand)
        capacity = n_cand
    raise OverflowError("candidate buffer overflow")


def _rescore(k, pruned, cands, row_cnt, last, stats):
    """Exact scores of one chunk's candidates; only the pairs strictly above the threshold are kept, and counted per
    left row in row_cnt.  Returns (rows, columns, scores, kept count, survivors of the longest row when `last`)."""
    t = torch()
    L = _lib.load()
    A, B, dev = k.A, k.B, k.A.device
    cand_row, cand_col, cand_part, n_cand = cands
    _, _, _, l_thr, _, l_xg = pruned
    dt = _lib.SG_DTYPE_F32 if A.dtype == np.float32 else _lib.SG_DTYPE_F64
    score = _empty(n_cand, t.float64, dev)
    keep_row = _empty(n_cand, t.int32, dev)
    keep_col = _empty(n_cand, t.int32, dev)
    k.counters.zero_()
    if k.plan.refine:
        _lib.check(L.sg_rescore_refined(n_cand, _ptr(cand_row), _ptr(cand_col), _ptr(cand_part), _ptr(l_xg),
                                        _ptr(B._heavy_groups), _ptr(l_thr), _ptr(A.d_indptr), _ptr(A.d_indices),
                                        _ptr(A.d_val), _ptr(B.d_indptr), _ptr(B.d_indices), _ptr(B.d_val), dt,
                                        _ptr(score), k.threshold, _ptr(keep_row), _ptr(keep_col), k.counter(0),
                                        k.counter(2), _ptr(row_cnt), k.row_begin, _stream()))
    else:
        _lib.check(L.sg_rescore(n_cand, _ptr(cand_row), _ptr(cand_col), _ptr(A.d_indptr), _ptr(A.d_indices),
                                _ptr(A.d_val), _ptr(B.d_indptr), _ptr(B.d_indices), _ptr(B.d_val), dt,
                                _ptr(score), k.threshold, _ptr(keep_row), _ptr(keep_col), k.counter(0),
                                _ptr(row_cnt), k.row_begin, _stream()))
    LAUNCH_COUNTS["rescore"] += 1
    if last:      # the largest row rides along with the read-back
        _lib.check(L.sg_row_count_max(k.n_rows, _ptr(row_cnt), k.counter(1), _stream()))
    head = k.counters[:3].cpu().numpy()
    if k.plan.refine and stats is not None:
        stats["n_refined"] = stats.get("n_refined", 0) + int(head[2])
    return keep_row, keep_col, score, int(head[0]), int(head[1])


def _candidates_rescored(k, stats):
    """Pruning level and sizing (_size_candidates), then the candidates of the left rows chunk by chunk (slices of the
    processing order), each chunk re-scored exactly right away.  Returns the survivors (rows, columns, scores, count),
    their count per left row and that of the longest row."""
    t = torch()
    dev, n_rows = k.A.device, k.n_rows
    # sized here so that only the chunk loop holds the whole-range launch's buffers (released after their re-score)
    level, pruned, est, first = _size_candidates(k, stats)
    mark(stats, "prune_sample")
    if stats is not None:
        stats["prune"], stats["acc"] = level, k.plan.acc
        stats["kernel"] = k.plan.kernel
        stats["n_candidates_estimate"] = est
        if stats.get("count_macs") and pruned[2] is not None:
            stats["macs_walked"], stats["features_kept"] = _count_macs(k, pruned)
    n_chunks, rows_per_chunk = row_chunks(n_rows, est)
    kept = []
    n_cand_total = 0
    row_cnt = t.zeros(n_rows + 1, dtype=t.int32, device=dev)      # survivors per left row (sg_rescore)
    for lo in range(0, n_rows, rows_per_chunk):
        hi = min(lo + rows_per_chunk, n_rows)
        if first is not None:        # only without an estimate, i.e. in one chunk
            cands, first = first, None
        else:
            perm = k.perm_a if (lo == 0 and hi == n_rows) else k.perm_a[lo:hi]
            cands = _chunk_candidates(k, pruned, perm, hi - lo, chunk_capacity(n_rows, hi - lo, est), stats)
        n_cand_total += cands[3]
        mark(stats, "candidates")
        keep_row, keep_col, score, n_keep, max_row_cnt = _rescore(k, pruned, cands, row_cnt, hi == n_rows, stats)
        mark(stats, "rescore")
        if n_chunks > 1:      # release the chunk-sized buffers, keep the survivors
            keep_row, keep_col, score = keep_row[:n_keep].clone(), keep_col[:n_keep].clone(), score[:n_keep].clone()
        kept.append((keep_row, keep_col, score, n_keep))
        del cands
    if len(kept) == 1:
        cand_row, cand_col, score, n_cand = kept[0]
    else:
        n_cand = sum(x[3] for x in kept)
        cand_row = t.cat([x[0][:x[3]] for x in kept]) if n_cand else _empty(1, t.int32, dev)
        cand_col = t.cat([x[1][:x[3]] for x in kept]) if n_cand else _empty(1, t.int32, dev)
        score = t.cat([x[2][:x[3]] for x in kept]) if n_cand else _empty(1, t.float64, dev)
    if stats is not None:
        stats["n_candidates"] = n_cand_total
        stats["n_above_threshold"] = n_cand
        stats["n_row_chunks"] = n_chunks
    return cand_row, cand_col, score, n_cand, row_cnt, max_row_cnt


def _select(k, top_n, cand_row, cand_col, score, n_cand, row_cnt, max_row_cnt, stats):
    """The top_n survivors of every left row, by descending score (one read-back: match count and longest row)."""
    t = torch()
    L = _lib.load()
    dev, n_rows, row_begin = k.A.device, k.n_rows, k.row_begin
    out_indptr = _empty(n_rows + 1, t.int64, dev)
    out_row = _empty(n_cand, t.int32, dev)
    out_col = _empty(n_cand, t.int32, dev)
    out_score = _empty(n_cand, t.float64, dev)
    tail = t.zeros(2, dtype=t.int64, device=dev)            # [0] out_nnz, [1] max_row (int32 view)
    c_nnz, c_max = ctypes.c_void_p(tail.data_ptr()), ctypes.c_void_p(tail.data_ptr() + 8)
    mode = select_mode(top_n, max_row_cnt, int(L.sg_topn_rows_cap()))
    if mode == "rows":
        ws_bytes = int(L.sg_topn_select_rows_workspace_bytes(n_cand, n_rows))
        ws = _empty(ws_bytes, t.uint8, dev)
        _lib.check(L.sg_topn_select_rows(n_cand, _ptr(cand_row), _ptr(cand_col), _ptr(score), row_begin, n_rows, top_n,
                                         _ptr(row_cnt), _ptr(out_indptr), _ptr(out_row), _ptr(out_col),
                                         _ptr(out_score), c_nnz, c_max, _ptr(ws), ws_bytes, _stream()))
        LAUNCH_COUNTS["select"] += 6
    else:
        ws_bytes = int(L.sg_topn_select_workspace_bytes(n_cand, n_rows))
        ws = _empty(ws_bytes, t.uint8, dev)
        _lib.check(L.sg_topn_select(n_cand, _ptr(cand_row), _ptr(cand_col), _ptr(score), row_begin, n_rows, top_n,
                                    k.threshold, _ptr(out_indptr), _ptr(out_row), _ptr(out_col), _ptr(out_score),
                                    c_nnz, c_max, _ptr(ws), ws_bytes, _stream()))
        LAUNCH_COUNTS["select"] += 7
    if stats is not None:
        stats["select"] = mode
    th = tail.cpu().numpy()
    mark(stats, "select")
    return DeviceMatches((k.A.shape[0], k.B.shape[0]), out_row, out_col, out_score, int(th[0]),
                         int(th[1:2].view(np.int32)[0]), indptr=out_indptr)


def symmetrize(M, fix_diagonal=True, mirror=True):
    """diag := 1 (fix_diagonal), pattern := pattern U pattern^T (mirror), rows ordered by column
    (string_grouper.py:419-427, :955-964) on the device."""
    t = require_cuda()
    L = _lib.load()
    n = M.shape[0]
    dev = M.d_row.device
    flags = (_lib.SG_SYMM_FIX_DIAGONAL if fix_diagonal else 0) | (_lib.SG_SYMM_MIRROR if mirror else 0)
    cap = 2 * M.nnz + n
    out_row = _empty(cap, t.int32, dev)
    out_col = _empty(cap, t.int32, dev)
    out_score = _empty(cap, t.float64, dev)
    out_nnz = t.zeros(1, dtype=t.int64, device=dev)
    ws_bytes = int(L.sg_symmetrize_workspace_bytes(M.nnz, n))
    ws = _empty(ws_bytes, t.uint8, dev)
    _lib.check(L.sg_symmetrize(n, M.nnz, flags, _ptr(M.d_row), _ptr(M.d_col), _ptr(M.d_score), _ptr(out_row),
                               _ptr(out_col), _ptr(out_score), _ptr(out_nnz), _ptr(ws), ws_bytes, _stream()))
    LAUNCH_COUNTS["symmetrize"] += 3
    nnz = int(out_nnz.item())
    return DeviceMatches(M.shape, out_row, out_col, out_score, nnz, M.max_row, out_dtype=M.out_dtype)


def group_reps(M, n, centroid, keep_device=False):
    """Representative index of every string's group from the (row, col)-sorted device match list
    (StringGrouper._deduplicate, string_grouper.py:851-904).  keep_device: also return the int32 device tensor
    (positions for the device string gather)."""
    t = require_cuda()
    L = _lib.load()
    dev = M.d_row.device
    rep = _empty(n, t.int32, dev)
    ws_bytes = int(L.sg_group_reps_workspace_bytes(n))
    ws = _empty(ws_bytes, t.uint8, dev)
    _lib.check(L.sg_group_reps(n, M.nnz, _ptr(M.d_row), _ptr(M.d_col), _ptr(M.d_score), 1 if centroid else 0,
                               _ptr(rep), _ptr(ws), ws_bytes, _stream()))
    LAUNCH_COUNTS["groups"] += 6
    host = rep[:n].cpu().numpy().astype(np.int64)
    return (host, rep) if keep_device else host


def nearest_master(M, n_right):
    """int64 [n_right]: for every right row the left row of its best match (smallest index among equal scores),
    -1 without a match — the reduction of StringGrouper._get_nearest_matches (string_grouper.py:803-807)."""
    t = require_cuda()
    L = _lib.load()
    dev = M.d_row.device
    best = _empty(n_right, t.int32, dev)
    ws_bytes = int(L.sg_nearest_master_workspace_bytes(n_right))
    ws = _empty(ws_bytes, t.uint8, dev)
    _lib.check(L.sg_nearest_master(M.nnz, _ptr(M.d_row), _ptr(M.d_col), _ptr(M.d_score), n_right, _ptr(best), _ptr(ws),
                                   ws_bytes, _stream()))
    LAUNCH_COUNTS["groups"] += 3
    return best[:n_right].cpu().numpy().astype(np.int64)


class RawStrings:
    """Packed UTF-8 strings of master ++ duplicates as uploaded for K1, kept for the device string gather."""

    def __init__(self, d_bytes, d_off, n_master, n_docs):
        self.d_bytes, self.d_off, self.n_master, self.n_docs = d_bytes, d_off, int(n_master), int(n_docs)


def gather_strings(raw, sides):
    """For every (doc_base, positions, n_sel) in `sides`: (offsets int64 [n_sel+1], bytes uint8) on the host of the
    strings at `positions` (device int32) of the Series starting at document `doc_base` — the
    `Series.iloc[...]` of get_matches (string_grouper.py:462, :467).  Two synchronisations in total: the byte
    counts, then all offsets and bytes."""
    t = require_cuda()
    L = _lib.load()
    dev = raw.d_off.device
    offs = []
    for doc_base, positions, n_sel in sides:
        out_off = _empty(n_sel + 1, t.int64, dev)
        ws_bytes = int(L.sg_gather_workspace_bytes(n_sel))
        ws = _empty(ws_bytes, t.uint8, dev)
        _lib.check(L.sg_gather_offsets(_ptr(raw.d_off), int(doc_base), n_sel, _ptr(positions), _ptr(out_off),
                                       _ptr(ws), ws_bytes, _stream()))
        offs.append(out_off)
    totals = t.stack([o[n_sel] for o, (_, _, n_sel) in zip(offs, sides)]).cpu().numpy()
    datas = []
    for out_off, total, (doc_base, positions, n_sel) in zip(offs, totals, sides):
        out = _empty(int(total), t.uint8, dev)
        _lib.check(L.sg_gather_bytes(_ptr(raw.d_bytes), _ptr(raw.d_off), int(doc_base), n_sel, _ptr(positions),
                                     _ptr(out_off), _ptr(out), _stream()))
        LAUNCH_COUNTS["gather"] += 2
        datas.append(out[:int(total)])
    host = to_host(*([o[:n_sel + 1] for o, (_, _, n_sel) in zip(offs, sides)] + datas))
    k = len(sides)
    return [(host[i], host[k + i]) for i in range(k)]


def matches_from_scipy(m):
    """Upload a host CSR of matches (e.g. returned by a user-supplied _build_matches)."""
    t = require_cuda()
    m = m.tocsr()
    dev = t.device("cuda", t.cuda.current_device())
    # keep CSR storage order (value-descending inside a row for the reference's product)
    r2 = np.repeat(np.arange(m.shape[0], dtype=np.int32), np.diff(m.indptr))
    row = t.from_numpy(r2).to(dev)
    col = t.from_numpy(np.ascontiguousarray(m.indices, dtype=np.int32)).to(dev)
    score = t.from_numpy(np.ascontiguousarray(m.data, dtype=np.float64)).to(dev)
    max_row = int(np.diff(m.indptr).max()) if m.shape[0] else 0
    if row.numel() == 0:
        row = _empty(1, t.int32, dev)
        col = _empty(1, t.int32, dev)
        score = _empty(1, t.float64, dev)
    return DeviceMatches(m.shape, row, col, score, m.nnz, max_row, out_dtype=m.dtype)


def rowwise_dot(A, B):
    """StringGrouper.dot (string_grouper.py:433-440): row-wise similarity of two equal-shape matrices."""
    t = require_cuda()
    L = _lib.load()
    if A.shape != B.shape:
        raise ValueError("shape mismatch")
    out = _empty(A.shape[0], t.float64, A.device)
    dt = _lib.SG_DTYPE_F32 if A.dtype == np.float32 else _lib.SG_DTYPE_F64
    _lib.check(L.sg_rowwise_dot(A.shape[0], _ptr(A.d_indptr), _ptr(A.d_indices), _ptr(A.d_val), _ptr(B.d_indptr),
                                _ptr(B.d_indices), _ptr(B.d_val), dt, _ptr(out), _stream()))
    LAUNCH_COUNTS["rowdot"] += 1
    return out[:A.shape[0]].cpu().numpy().astype(A.dtype, copy=False)


class DeviceVocabulary:
    """df / rank tables of the fitted vectoriser (the device twin of TfidfVectorizer.vocabulary_ / idf_)."""

    def __init__(self, df_table, rank_table, ngram, n_docs, vocab_size):
        self.d_df, self.d_rank = df_table, rank_table
        self.ngram, self.n_docs, self.size = int(ngram), int(n_docs), int(vocab_size)

    def feature_names(self):
        """Sorted n-grams, column order of the TF-IDF matrices (sklearn get_feature_names_out)."""
        from ._ingest import decode_vocab_keys
        t = require_cuda()
        L = _lib.load()
        keys = _empty(self.size, t.int32, self.d_df.device)
        _lib.check(L.sg_tfidf_vocab_keys(_ptr(self.d_df), _ptr(self.d_rank), self.ngram, _ptr(keys), _stream()))
        return decode_vocab_keys(keys[:self.size].cpu().numpy().view(np.uint32), self.ngram)


def upload_strings(data, offsets, device=None):
    """H2D of the packed strings: (uint8 bytes, int64 offsets) -> device tensors."""
    t = require_cuda()
    device = device or t.device("cuda", t.cuda.current_device())
    total = int(offsets[-1])
    d_bytes = (t.from_numpy(np.ascontiguousarray(data)).to(device, non_blocking=True) if total
               else _empty(1, t.uint8, device))
    d_off = t.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64)).to(device, non_blocking=True)
    return d_bytes, d_off, total


class DeviceVocabulary64:
    """Sorted vocabulary of the general vectoriser (csrc/sg_tfidf64.cu): 64-bit keys over a dense alphabet."""

    def __init__(self, keys, df, alphabet, bits, ngram, n_docs, vocab_size):
        self.d_keys, self.d_df, self.alphabet = keys, df, alphabet
        self.bits, self.ngram, self.n_docs, self.size = int(bits), int(ngram), int(n_docs), int(vocab_size)

    def feature_names(self):
        from ._ingest import decode_vocab_keys64
        keys = self.d_keys[:self.size].cpu().numpy().view(np.uint64)
        return decode_vocab_keys64(keys, self.ngram, self.bits, self.alphabet)


DENSE_KEY_BITS = 21      # the dense key table (2^(7n) slots) is used up to trigrams; beyond: sorted vocabulary


def tfidf_sorted(data, offsets, n_master, ngram, flags, dtype, device=None, stats=None):
    """K1, general form: 64-bit keys + sort-based vocabulary (ngram_size >= 4, or uint32 code points)."""
    from . import _ingest
    t = require_cuda()
    L = _lib.load()
    device = device or t.device("cuda", t.cuda.current_device())
    n_docs = len(offsets) - 1
    total = int(offsets[-1])
    raw_bytes = None
    if data.dtype == np.uint8:
        lut, alphabet = _ingest.byte_alphabet(data, flags)
        sym_width = 1
        d_sym = t.from_numpy(np.ascontiguousarray(data)).to(device) if total else _empty(1, t.uint8, device)
        d_lut = t.from_numpy(lut).to(device)
        raw_bytes = d_sym
    else:
        alphabet = np.unique(data)
        ids = np.searchsorted(alphabet, data).astype(np.uint32)
        sym_width = 4
        d_sym = t.from_numpy(ids.view(np.int32)).to(device) if total else _empty(1, t.int32, device)
        d_lut = None
    bits = _ingest.symbol_bits(len(alphabet))
    if int(ngram) * bits > 64:
        raise NotImplementedError(
            "ngram_size=%d over an alphabet of %d distinct characters needs %d-bit n-gram keys; the device vectoriser "
            "packs keys into 64 bits (ngram_size * ceil(log2(alphabet)) <= 64)" % (ngram, len(alphabet), ngram * bits))
    d_off = t.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64)).to(device)
    TRANSFER_BYTES["h2d"] += int(total * sym_width + 8 * len(offsets))
    np_dtype = np.float32 if np.dtype(dtype) == np.float32 else np.float64
    s_clean = _empty(total, t.int32, device)
    s_sort = _empty(total, t.int64, device)
    s_key = _empty(total, t.int64, device)
    s_tf = _empty(total, t.int32, device)
    row_nnz = _empty(n_docs + 1, t.int32, device)
    _lib.check(L.sg_tfidf64_count(_ptr(d_sym), sym_width, _ptr(d_off), n_docs, int(ngram), bits, _ptr(d_lut),
                                  _ptr(s_clean), _ptr(s_sort), _ptr(s_key), _ptr(s_tf), _ptr(row_nnz), _stream()))
    indptr = _empty(n_docs + 1, t.int64, device)
    indices = _empty(total, t.int32, device)
    val32 = _empty(total, t.float32, device)
    val64 = _empty(total, t.float64, device) if np_dtype == np.float64 else None
    vocab_keys = _empty(total, t.int64, device)
    df = _empty(total, t.int32, device)
    tail = t.zeros(2, dtype=t.int64, device=device)         # [0] V (int32 view), [1] nnz
    ws_bytes = int(L.sg_tfidf64_finalize_workspace_bytes(n_docs, total))
    ws = _empty(ws_bytes, t.uint8, device)
    dt = _lib.SG_DTYPE_F32 if np_dtype == np.float32 else _lib.SG_DTYPE_F64
    _lib.check(L.sg_tfidf64_finalize(_ptr(d_off), n_docs, n_docs, total, int(ngram), bits, dt, _ptr(s_key), _ptr(s_tf),
                                     _ptr(row_nnz), _ptr(indptr), _ptr(indices), _ptr(val64), _ptr(val32),
                                     _ptr(vocab_keys), _ptr(df), ctypes.c_void_p(tail.data_ptr()),
                                     ctypes.c_void_p(tail.data_ptr() + 8), _ptr(ws), ws_bytes, _stream()))
    LAUNCH_COUNTS["tfidf"] += 7
    n_master = int(n_master)
    head = t.cat([tail, indptr[n_master:n_master + 1]]).cpu().numpy()
    V = int(head[0:1].view(np.int32)[0])
    nnz = int(head[1])
    split = int(head[2])
    val = val64 if np_dtype == np.float64 else val32
    vocab = DeviceVocabulary64(vocab_keys, df, alphabet, bits, ngram, n_docs, V)
    if stats is not None:
        stats.update(n_docs=n_docs, total_bytes=total, nnz=nnz, vocab=V, h2d_bytes=int(total * sym_width + 8 * len(offsets)),
                     vectoriser="sorted vocabulary, %d-bit keys" % (int(ngram) * bits))
        if raw_bytes is not None:
            stats["raw"] = RawStrings(raw_bytes, d_off, n_master, n_docs)
    master = DeviceCSR((n_master, V), indptr[:n_master + 1], indices, val, val32, split, np_dtype, 1.0, base=0)
    master.nnz_parent = nnz
    if n_master == n_docs:
        master._df = df[:max(V, 1)]       # fitted on exactly these rows: the vectoriser's df is sg_feature_df(master)
        return master, None, vocab
    dup = DeviceCSR((n_docs - n_master, V), indptr[n_master:], indices, val, val32, nnz - split, np_dtype, 1.0,
                    base=split)
    dup.nnz_parent = nnz
    return master, dup, vocab


def tfidf(data, offsets, n_master, ngram, flags, dtype, device=None, stats=None, df_allreduce=None, n_docs_fit=None):
    """K1 from host buffers: packed strings (master ++ duplicates) -> TF-IDF CSR in HBM.  uint8 `data` = ASCII bytes
    (dense key table up to trigrams), anything else goes through the sorted-vocabulary vectoriser."""
    if data.dtype != np.uint8 or 7 * int(ngram) > DENSE_KEY_BITS:
        if df_allreduce is not None:
            raise NotImplementedError("the sharded vectoriser (df all-reduce) needs ASCII text and ngram_size <= 3")
        return tfidf_sorted(data, offsets, n_master, ngram, flags, dtype, device=device, stats=stats)
    d_bytes, d_off, total = upload_strings(data, offsets, device)
    TRANSFER_BYTES["h2d"] += int(total + 8 * len(offsets))
    if stats is not None:
        stats["h2d_bytes"] = int(total + 8 * len(offsets))
        stats["raw"] = RawStrings(d_bytes, d_off, n_master, len(offsets) - 1)
    return tfidf_resident(d_bytes, d_off, len(offsets) - 1, total, n_master, ngram, flags, dtype, stats=stats,
                          df_allreduce=df_allreduce, n_docs_fit=n_docs_fit)


def tfidf_resident(d_bytes, d_off, n_docs, total, n_master, ngram, flags, dtype, stats=None, df_allreduce=None,
                   n_docs_fit=None):
    """K1 on strings already resident in HBM.

    Device counterpart of _fit_vectorizer + transform (string_grouper.py:685-707): the vocabulary /
    df / idf are fitted on ALL rows, then rows [0, n_master) form the master matrix and the rest the
    duplicate matrix (views of the same device arrays).  Returns (master, duplicates | None, vocab).
    """
    t = require_cuda()
    L = _lib.load()
    device = d_off.device
    slots = int(L.sg_tfidf_table_slots(int(ngram)))
    if slots < 0:
        raise NotImplementedError("ngram_size=%r: the device vectoriser supports 1 <= ngram_size <= 4" % (ngram,))
    np_dtype = np.float32 if np.dtype(dtype) == np.float32 else np.float64
    df = t.zeros(slots, dtype=t.int32, device=device)
    rank = _empty(slots, t.int32, device)
    s_clean = _empty(total, t.uint8, device)
    s_sort = _empty(total, t.int32, device)
    s_key = _empty(total, t.int32, device)
    s_tf = _empty(total, t.int32, device)
    row_nnz = _empty(n_docs + 1, t.int32, device)
    _lib.check(L.sg_tfidf_count(_ptr(d_bytes), _ptr(d_off), n_docs, int(ngram), int(flags), _ptr(df), _ptr(s_clean),
                                _ptr(s_sort), _ptr(s_key), _ptr(s_tf), _ptr(row_nnz), _stream()))
    if df_allreduce is not None:
        df_allreduce(df)          # corpus sharded over GPUs: document frequencies are summed over the ranks (NCCL)
    indptr = _empty(n_docs + 1, t.int64, device)
    indices = _empty(total, t.int32, device)
    val32 = _empty(total, t.float32, device)
    val64 = _empty(total, t.float64, device) if np_dtype == np.float64 else None
    tail = t.zeros(2, dtype=t.int64, device=device)         # [0] V (int32 view), [1] nnz
    ws_bytes = int(L.sg_tfidf_finalize_workspace_bytes(n_docs, int(ngram)))
    ws = _empty(ws_bytes, t.uint8, device)
    dt = _lib.SG_DTYPE_F32 if np_dtype == np.float32 else _lib.SG_DTYPE_F64
    _lib.check(L.sg_tfidf_finalize(_ptr(d_off), n_docs, int(n_docs if n_docs_fit is None else n_docs_fit), int(ngram),
                                   dt, _ptr(df), _ptr(rank), _ptr(s_key), _ptr(s_tf),
                                   _ptr(row_nnz), _ptr(indptr), _ptr(indices), _ptr(val64), _ptr(val32),
                                   ctypes.c_void_p(tail.data_ptr()), ctypes.c_void_p(tail.data_ptr() + 8), _ptr(ws),
                                   ws_bytes, _stream()))
    LAUNCH_COUNTS["tfidf"] += 4
    n_master = int(n_master)
    head = t.cat([tail, indptr[n_master:n_master + 1]]).cpu().numpy()     # one read-back: V, nnz, split point
    V = int(head[0:1].view(np.int32)[0])
    nnz = int(head[1])
    split = int(head[2])
    val = val64 if np_dtype == np.float64 else val32
    vocab = DeviceVocabulary(df, rank, ngram, n_docs if n_docs_fit is None else n_docs_fit, V)
    if stats is not None:
        stats.update(n_docs=n_docs, total_bytes=total, nnz=nnz, vocab=V)
    master = DeviceCSR((n_master, V), indptr[:n_master + 1], indices, val, val32, split, np_dtype, 1.0, base=0)
    master.nnz_parent = nnz
    if n_master == n_docs:
        if df_allreduce is None and n_docs_fit is None:
            # fitted on exactly these rows: the vectoriser's df, in column order, is sg_feature_df(master)
            col_df = _empty(max(V, 1), t.int32, device)
            _lib.check(L.sg_tfidf_vocab_df(_ptr(df), _ptr(rank), int(ngram), _ptr(col_df), _stream()))
            master._df = col_df
        return master, None, vocab
    dup = DeviceCSR((n_docs - n_master, V), indptr[n_master:], indices, val, val32, nnz - split, np_dtype, 1.0,
                    base=split)
    dup.nnz_parent = nnz
    return master, dup, vocab


def as_device_matches(m):
    return m if isinstance(m, DeviceMatches) else matches_from_scipy(m)


def empty_csr(like, n_rows):
    """A CSR block with `n_rows` empty rows on the device of `like` (ranks that own no rows of a sharded matrix)."""
    t = torch()
    dev = like.device
    val = _empty(1, t.float32 if like.dtype == np.float32 else t.float64, dev)
    val32 = val if like.dtype == np.float32 else _empty(1, t.float32, dev)
    return DeviceCSR((n_rows, like.shape[1]), t.zeros(n_rows + 1, dtype=t.int64, device=dev),
                     _empty(1, t.int32, dev), val, val32, 0, like.dtype, like.norm_bound)


def offset_rows(m, row_offset, n_rows_total):
    """Row ids of a per-rank block -> ids in the full left matrix."""
    if m.nnz:
        m.d_row[:m.nnz] += int(row_offset)
    return DeviceMatches((int(n_rows_total), m.shape[1]), m.d_row, m.d_col, m.d_score, m.nnz, m.max_row,
                         out_dtype=m.out_dtype)


def allgather_csr(M, n_rows_total):
    """Right matrix sharded by rows over the ranks (sharded K1) -> the full matrix on every rank (NCCL all-gather
    over NVLink of row lengths, indices and values)."""
    from . import _dist
    t = torch()
    n = M.shape[0]
    lo, hi = M.base, M.base + M.nnz
    row_len = (M.d_indptr[1:n + 1] - M.d_indptr[:n]).contiguous()
    vals = (M.d_val[lo:hi].contiguous(),) if M.d_val is M.d_val32 else (M.d_val[lo:hi].contiguous(),
                                                                         M.d_val32[lo:hi].contiguous())
    indptr, indices, gvals = _dist.allgather_csr_rows(row_len, M.d_indices[lo:hi].contiguous(), vals)
    nnz = int(indptr[-1].item())
    if nnz == 0:
        indices = _empty(1, t.int32, M.device)
        gvals = tuple(_empty(1, v.dtype, M.device) for v in vals)
    val = gvals[0]
    val32 = gvals[0] if len(gvals) == 1 else gvals[1]
    out = DeviceCSR((int(n_rows_total), M.shape[1]), indptr, indices, val, val32, nnz, M.dtype, M.norm_bound)
    return out


def gather_shards(m):
    """Multi-GPU: all-gather the per-rank top-n lists (each rank computed its own block of left rows) so that
    every rank holds the full result in row order; the `vstack` of string_grouper.py:750 over NVLink."""
    from . import _dist
    row, col, score, nnz, max_row = _dist.gather_matches(m.shape, m.d_row, m.d_col, m.d_score, m.nnz, m.max_row)
    t = torch()
    if nnz == 0:
        row, col, score = _empty(1, t.int32, row.device), _empty(1, t.int32, row.device), _empty(1, t.float64, row.device)
    return DeviceMatches(m.shape, row, col, score, nnz, max_row, out_dtype=m.out_dtype)


def apply_pending(m):
    """Run the recorded _fix_diagonal / _symmetrize_matrix steps as one K4 launch (string_grouper.py:419-427:
    the LIL round trip also re-orders every row by column, which K4 does even when only one step is set)."""
    m = as_device_matches(m)
    return symmetrize(m, fix_diagonal=m.pending_fix_diagonal, mirror=m.pending_mirror)
