"""Device-side building blocks of the reduced-order sweep path.

Everything numerical happens in ``libmorfem_b200.so`` (hand-written sm_100a CUDA, ``morfem_b200/csrc``);
PyTorch supplies device memory (tensors are only allocators / ``data_ptr()`` hand-off), the current stream, and
``torch.distributed`` for the r x r all-reduces, the halo exchange and the result gather.  There is no CPU
fallback: every function raises if CUDA or the library is unavailable.

Reference call sites replaced (paths relative to the reference repo):
  orthonormalize        np.linalg.svd(S, full_matrices=False)[0]     implementation.py:226, :298, :210
  spmm / gemm_tn        (q_t @ a_i) @ q                              implementation.py:181-183
  project_rhs           q_t @ b                                      implementation.py:184
  sweep                 solve_finite_element_method + GSM loop       implementation.py:189-194, test_helpers.py:60-65
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _ffi

C128 = torch.complex128


def require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise _ffi.MorfemB200Error("morfem_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


F64 = torch.float64


def _check_mat(t: torch.Tensor, name: str):
    if t.dtype not in (C128, F64) or not t.is_cuda or t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"{name}: expected a row-major complex128 or float64 CUDA matrix, got {t.dtype} {tuple(t.shape)} strides {t.stride()}")


def _same_dtype(a: torch.Tensor, b: torch.Tensor, what: str) -> bool:
    """True when both operands are real float64 (the real twins run), False when both are complex128."""
    if a.dtype != b.dtype:
        raise ValueError(f"{what}: operands must share a dtype (float64 or complex128), got {a.dtype} and {b.dtype}")
    return a.dtype == F64


def to_device_c128(a, device=None) -> torch.Tensor:
    """Host ndarray (real or complex) -> contiguous complex128 device tensor."""
    device = device or require_cuda()
    arr = np.ascontiguousarray(np.asarray(a), dtype=np.complex128)
    return upload(arr, device)


def real_or_complex_to_device(a, device=None, widen: bool = False) -> torch.Tensor:
    """Host ndarray -> device tensor in its own field: complex input -> complex128, real input -> float64 (half the
    PCIe traffic and, with ``widen=False``, the real float64 twins of the stage-1/2 kernels).  ``widen=True`` converts
    real data to complex128 on the device (the complex128 kernels of the north star run on real data too)."""
    device = device or require_cuda()
    if isinstance(a, torch.Tensor):
        t = a.to(device, non_blocking=True)
        if t.dtype == C128 or (t.dtype == F64 and not widen):
            return t
        return t.to(C128) if (widen or t.is_complex()) else t.to(F64)
    arr = np.asarray(a)
    if np.iscomplexobj(arr):
        return to_device_c128(arr, device)
    t = upload(np.ascontiguousarray(arr, dtype=np.float64), device)
    return t.to(C128) if widen else t


class _Workspaces:
    """Grow-only byte buffers keyed by purpose, per device (the C ABI never allocates)."""

    def __init__(self):
        self._bufs = {}
        self._pinned = set()       # keys whose current buffer is referenced by a captured CUDA graph
        self._retired = []         # outgrown buffers that a graph may still replay into

    def get(self, key: str, nbytes: int, device) -> torch.Tensor:
        k = (key, str(device))
        buf = self._bufs.get(k)
        if buf is None or buf.numel() < nbytes:
            if buf is not None and k in self._pinned:
                self._retired.append(buf)          # a graph holds its raw pointer: keep the memory alive
                self._pinned.discard(k)
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
            self._bufs[k] = buf
        return buf

    def pin_all(self):
        """Called after a CUDA-graph capture: every buffer handed out so far may be baked into the graph."""
        self._pinned.update(self._bufs.keys())

    def clear(self):
        self._bufs.clear()
        self._pinned.clear()
        self._retired.clear()


workspaces = _Workspaces()


class KernelTimer:
    """Optional per-call CUDA-event timing of the C-ABI launches (bench.py's roofline leg).  Events are recorded
    on the launching (current) stream around each call; ``summary()`` synchronises and aggregates by kernel name
    with the ALGORITHMIC bytes and flops of each call (SURVEY.md section 8d formulas, restated in DESIGN.md)."""

    def __init__(self):
        self.records = []

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        for name, e0, e1, nbytes, flops in self.records:
            a = agg.setdefault(name, {"calls": 0, "ms": 0.0, "bytes": 0.0, "flops": 0.0})
            a["calls"] += 1
            a["ms"] += e0.elapsed_time(e1)
            a["bytes"] += nbytes
            a["flops"] += flops
        return agg


timer: Optional[KernelTimer] = None


class _timed:
    def __init__(self, name, nbytes=0.0, flops=0.0):
        self.name, self.nbytes, self.flops = name, float(nbytes), float(flops)

    def __enter__(self):
        if timer is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if timer is not None and exc[0] is None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            timer.records.append((self.name, self.e0, e1, self.nbytes, self.flops))
        return False


# ------------------------------------------------------------------------------------------ dense wrappers
def gemm_tn(a: torch.Tensor, b: torch.Tensor, conj: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``op(a)^T b`` (ra x rb), reduction over the rows; ``conj`` selects ``a^H``.  float64 operands run the real twin."""
    lib = _ffi.load()
    _check_mat(a, "a"); _check_mat(b, "b")
    real = _same_dtype(a, b, "gemm_tn")
    n, ra = a.shape
    rb = b.shape[1]
    if b.shape[0] != n:
        raise ValueError("gemm_tn: row counts differ")
    if out is None:
        out = torch.empty((ra, rb), dtype=a.dtype, device=a.device)
    same = a.data_ptr() == b.data_ptr() and ra == rb
    if real:
        nbytes = lib.mf_gemm_tn_f64_ws_bytes(ra, rb, n)
        ws = workspaces.get("gemm_tn", nbytes, a.device)
        with _timed("gemm_tn", nbytes=8.0 * n * (ra if same else ra + rb) + 8.0 * ra * rb, flops=2.0 * n * ra * rb):
            _ffi.check(lib.mf_gemm_tn_f64(_ptr(a), a.stride(0), ra, _ptr(b), b.stride(0), rb, n, _ptr(out), out.stride(0),
                                          _ptr(ws), ws.numel(), _stream()), "mf_gemm_tn_f64")
        return out
    nbytes = lib.mf_gemm_tn_ws_bytes(ra, rb, n)
    ws = workspaces.get("gemm_tn", nbytes, a.device)
    # complex flops are counted as the algorithmic 8 n ra rb (four real products per complex one) although the kernels issue three
    # (Gauss's form, dense_gemm.cu): TFLOP/s and shares of peak stay comparable with the four-product kernels
    with _timed("gemm_tn", nbytes=16.0 * n * (ra if same else ra + rb) + 16.0 * ra * rb, flops=8.0 * n * ra * rb):
        _ffi.check(lib.mf_gemm_tn_c128(_ptr(a), a.stride(0), ra, _ptr(b), b.stride(0), rb, n, int(conj), _ptr(out), out.stride(0),
                                       _ptr(ws), ws.numel(), _stream()), "mf_gemm_tn_c128")
    return out


def gemm_nn(a: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None, w_upper: bool = False) -> torch.Tensor:
    """``a @ w`` for a tall ``a`` (n x ra) and a small ``w`` (ra x rb).  float64 operands run the real twin.
    ``w_upper``: ``w`` is square upper triangular (the ``R^-1`` of a Cholesky-QR pass) -- zero tiles are skipped."""
    lib = _ffi.load()
    _check_mat(a, "a"); _check_mat(w, "w")
    real = _same_dtype(a, w, "gemm_nn")
    n, ra = a.shape
    if w.shape[0] != ra:
        raise ValueError("gemm_nn: inner dimensions differ")
    rb = w.shape[1]
    if out is None:
        out = torch.empty((n, rb), dtype=a.dtype, device=a.device)
    if w_upper:
        if rb != ra:
            raise ValueError("gemm_nn: w_upper needs a square w")
        tiles = (ra + 63) // 64                    # 64-column output tiles; tile j multiplies (j + 1) * 64 rows of w
        frac = (tiles + 1) / (2.0 * tiles)
        if real:
            with _timed("gemm_nn", nbytes=8.0 * n * (ra + rb) + 8.0 * ra * rb, flops=2.0 * n * ra * rb * frac):
                _ffi.check(lib.mf_trmm_nn_f64(_ptr(a), a.stride(0), n, ra, _ptr(w), w.stride(0), _ptr(out), out.stride(0), _stream()),
                           "mf_trmm_nn_f64")
        else:
            with _timed("gemm_nn", nbytes=16.0 * n * (ra + rb) + 16.0 * ra * rb, flops=8.0 * n * ra * rb * frac):
                _ffi.check(lib.mf_trmm_nn_c128(_ptr(a), a.stride(0), n, ra, _ptr(w), w.stride(0), _ptr(out), out.stride(0), _stream()),
                           "mf_trmm_nn_c128")
        return out
    if real:
        with _timed("gemm_nn", nbytes=8.0 * n * (ra + rb) + 8.0 * ra * rb, flops=2.0 * n * ra * rb):
            _ffi.check(lib.mf_gemm_nn_f64(_ptr(a), a.stride(0), n, ra, _ptr(w), w.stride(0), rb, _ptr(out), out.stride(0), _stream()),
                       "mf_gemm_nn_f64")
        return out
    with _timed("gemm_nn", nbytes=16.0 * n * (ra + rb) + 16.0 * ra * rb, flops=8.0 * n * ra * rb):
        _ffi.check(lib.mf_gemm_nn_c128(_ptr(a), a.stride(0), n, ra, _ptr(w), w.stride(0), rb, _ptr(out), out.stride(0), _stream()),
                   "mf_gemm_nn_c128")
    return out


def symmetrize(a: torch.Tensor) -> torch.Tensor:
    """``(a + a.T) / 2`` -- implementation.py:528, hoisted out of the per-point loop."""
    lib = _ffi.load()
    _check_mat(a, "a")
    r = a.shape[0]
    if a.dtype == F64:
        return ((a + a.T) * 0.5).contiguous()      # r x r, literally implementation.py:528
    out = torch.empty((r, r), dtype=C128, device=a.device)
    _ffi.check(lib.mf_symmetrize_c128(_ptr(a), a.stride(0), r, _ptr(out), out.stride(0), _stream()), "mf_symmetrize_c128")
    return out


# ----------------------------------------------------------------------------------------- sparse operands
@dataclass
class DeviceCSR:
    """CSR operand of the SpMM.  For a reference ``csc_array`` ``a`` the CSC arrays *are* the CSR arrays of
    ``a.T``, which is what ``q_t @ a`` multiplies by (scipy ``_rmatmul_dispatch``)."""
    rowptr: torch.Tensor   # int32, nrows + 1 (rebased to 0 for a row slice)
    colidx: torch.Tensor   # int32, global column index = row of Q
    vals: torch.Tensor     # float64 or complex128
    nrows: int
    ncols: int
    row0: int = 0          # first global row of this slice
    grouped: Optional[tuple] = None   # (G, ustart int64, ucols int32, uvals float64): row-grouped form (see group_rows)
    sorted_indices: bool = False      # column indices ascending within every row (required by group_rows)
    pattern_id: Optional[int] = None   # equal for operands whose sparsity patterns were found identical (mark_same_pattern)

    @property
    def nnz(self) -> int:
        return int(self.colidx.numel())

    @property
    def is_real(self) -> bool:
        return self.vals.dtype == torch.float64


# bytes moved over PCIe by the upload / download helpers (bench.py's e2e leg reads these)
transfer_bytes = {"h2d": 0, "d2h": 0}


def upload(arr: np.ndarray, device) -> torch.Tensor:
    """One host->device copy of a contiguous ndarray (no dtype conversion, no intermediate host copy).  The copy is queued
    on the current stream; from pinned memory it is asynchronous, so consecutive uploads and the first kernels overlap
    with the host work between them (every public call ends with a blocking download, which orders it before return)."""
    t = torch.from_numpy(arr)
    transfer_bytes["h2d"] += t.numel() * t.element_size()
    return t.to(device, non_blocking=True)


def download(t: torch.Tensor, out: Optional[torch.Tensor] = None) -> np.ndarray:
    """Device->host copy; ``out`` may be a pinned host tensor of the same shape/dtype."""
    transfer_bytes["d2h"] += t.numel() * t.element_size()
    if out is not None:
        out.copy_(t, non_blocking=False)
        return out.numpy()
    return t.cpu().numpy()


def csr_of_transpose(a_csc, device=None, row_range=None, col_offset: int = 0, group_for_r: Optional[int] = None) -> DeviceCSR:
    """Upload the CSR view of ``a.T`` for a scipy ``csc_array``/``csc_matrix`` ``a`` (no conversion work: the
    three CSC arrays are reused as they are).  ``row_range=(lo, hi)`` uploads only rows lo..hi-1 of ``a.T``;
    ``col_offset`` is subtracted from the column indices (halo-window relative indexing); ``group_for_r`` also builds
    the row-grouped form for basis size r on the device (real operators with sorted indices only)."""
    import scipy.sparse as sp
    device = device or require_cuda()
    a = a_csc if sp.issparse(a_csc) and a_csc.format == "csc" else sp.csc_array(a_csc)
    n_rows_t = a.shape[1]
    lo, hi = (0, n_rows_t) if row_range is None else row_range
    indptr = np.asarray(a.indptr)
    s, e = int(indptr[lo]), int(indptr[hi])
    if e - s >= 2 ** 31 or a.shape[0] >= 2 ** 31:
        raise ValueError("operator too large for int32 indices")
    if lo == 0 and indptr.dtype == np.int32:
        rowptr = indptr[:hi + 1]
    else:
        rowptr = (indptr[lo:hi + 1] - indptr[lo]).astype(np.int32)
    colidx = np.ascontiguousarray(a.indices[s:e], dtype=np.int32)
    data = np.asarray(a.data[s:e])
    vals = np.ascontiguousarray(data, dtype=np.complex128 if np.iscomplexobj(data) else np.float64)
    if col_offset:
        colidx = colidx - np.int32(col_offset)
    csr = DeviceCSR(upload(np.ascontiguousarray(rowptr), device), upload(colidx, device), upload(vals, device),
                    hi - lo, a.shape[0], lo, None, bool(a.has_sorted_indices))
    if group_for_r is not None:
        group_rows(csr, group_for_r)
    return csr


def _group_size(r: int, real: bool) -> int:
    lib = _ffi.load()
    return int(lib.mf_spmm_group_size_f64(r) if real else lib.mf_spmm_group_size(r))


def group_rows(a: DeviceCSR, r: int, real: bool = False) -> None:
    """Build the row-grouped form of a real CSR operand with sorted column indices on the device (once per operator and
    group size): G = mf_spmm_group_size(r) (mf_spmm_group_size_f64 for a float64 Q) consecutive rows share one column-union list, so the SpMM loads each needed
    Q row once per group.  No-op when already built for this G or when the values are complex."""
    lib = _ffi.load()
    g = _group_size(r, real)
    if not a.is_real or not a.sorted_indices or a.nrows == 0 or (a.grouped is not None and a.grouped[0] == g):
        return
    dev = a.colidx.device
    ngroups = (a.nrows + g - 1) // g
    counts = torch.empty(ngroups, dtype=torch.int32, device=dev)
    _ffi.check(lib.mf_spmm_group_count(_ptr(a.rowptr), _ptr(a.colidx), a.nrows, g, _ptr(counts), _stream()), "mf_spmm_group_count")
    ustart = torch.zeros(ngroups + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=ustart[1:])
    total = a.nnz          # capacity: a union is never larger than the rows' non-zero count (no device->host read needed)
    ucols = torch.empty(total, dtype=torch.int32, device=dev)
    uvals = torch.empty(total * g, dtype=torch.float64, device=dev)
    _ffi.check(lib.mf_spmm_group_fill(_ptr(a.rowptr), _ptr(a.colidx), _ptr(a.vals), a.nrows, g, _ptr(ustart), _ptr(ucols), _ptr(uvals),
                                      _stream()), "mf_spmm_group_fill")
    a.grouped = (g, ustart, ucols, uvals)


def spmm(a: DeviceCSR, q: torch.Tensor, out: Optional[torch.Tensor] = None, col_offset: int = 0) -> torch.Tensor:
    """``Y = A Q`` for the CSR operand; ``q`` holds rows ``col_offset ..`` of the global Q (halo window)."""
    lib = _ffi.load()
    _check_mat(q, "q")
    r = q.shape[1]
    real = q.dtype == F64
    if real and not a.is_real:
        raise ValueError("spmm: a real float64 Q needs a real operator (convert Q to complex128 for complex operators)")
    if out is None:
        out = torch.empty((a.nrows, r), dtype=q.dtype, device=q.device)
    w = 8.0 if real else 16.0
    if a.grouped is not None and col_offset == 0 and a.grouped[0] == _group_size(r, real):
        g, ustart, ucols, uvals = a.grouped
        nunion = (int(ustart[-1].item()) if timer is not None else 0)      # only the profiling pass needs the exact size
        if real:
            nbytes = nunion * (4.0 + 8.0 * g) + 8.0 * ustart.numel() + w * r * (a.nrows + q.shape[0])
            with _timed("spmm_csr", nbytes=nbytes, flops=2.0 * a.nnz * r):
                _ffi.check(lib.mf_spmm_grouped_f64(_ptr(ustart), _ptr(ucols), _ptr(uvals), a.nrows, g, _ptr(q), q.stride(0), r,
                                                   _ptr(out), out.stride(0), _stream()), "mf_spmm_grouped_f64")
            return out
        nbytes = nunion * (4.0 + 8.0 * g) + 8.0 * ustart.numel() + 16.0 * r * (a.nrows + q.shape[0])
        with _timed("spmm_csr", nbytes=nbytes, flops=4.0 * a.nnz * r):
            _ffi.check(lib.mf_spmm_grouped_c128(_ptr(ustart), _ptr(ucols), _ptr(uvals), a.nrows, g, _ptr(q), q.stride(0), r,
                                                _ptr(out), out.stride(0), _stream()), "mf_spmm_grouped_c128")
        return out
    colidx = a.colidx if col_offset == 0 else a.colidx - col_offset
    if real:
        with _timed("spmm_csr", nbytes=a.nnz * 12.0 + 4.0 * (a.nrows + 1) + w * r * (a.nrows + q.shape[0]), flops=2.0 * a.nnz * r):
            _ffi.check(lib.mf_spmm_csr_f64(_ptr(a.rowptr), _ptr(colidx), _ptr(a.vals), a.nrows, _ptr(q), q.stride(0), r,
                                           _ptr(out), out.stride(0), _stream()), "mf_spmm_csr_f64")
        return out
    valb = 8.0 if a.is_real else 16.0
    with _timed("spmm_csr", nbytes=a.nnz * (valb + 4.0) + 4.0 * (a.nrows + 1) + 16.0 * r * (a.nrows + q.shape[0]),
                flops=(4.0 if a.is_real else 8.0) * a.nnz * r):
        _ffi.check(lib.mf_spmm_csr_c128(_ptr(a.rowptr), _ptr(colidx), _ptr(a.vals), int(a.is_real), a.nrows, _ptr(q), q.stride(0), r,
                                        _ptr(out), out.stride(0), _stream()), "mf_spmm_csr_c128")
    return out


@dataclass
class DeviceWindows:
    """Operand of the TMA-staged SpMM (mf_spmm_window_*): CSR rows in blocks of RB with, per block, the list of distinct
    Q rows it references (the window) and, per non-zero, the 8-bit slot of its column inside that window."""
    rowptr: torch.Tensor    # int32, nrows + 1
    slot: torch.Tensor      # uint8, nnz
    vals: torch.Tensor      # float64, nnz
    wstart: torch.Tensor    # int32, nblocks + 1
    ucol: torch.Tensor      # int32, sum of window sizes
    nrows: int
    wmax: int
    nnz: int


def build_windows(a_csc, device=None, row_range=None, col_offset: int = 0) -> Optional[DeviceWindows]:
    """Window lists for the TMA-staged SpMM, built once per operator on the host (numpy): for every block of RB rows of
    ``a.T`` the sorted distinct column indices, and for every non-zero its position in its block's list.  Returns None when
    the operator does not qualify (complex values, a window above mf_spmm_window_max_rows(), a row with too many non-zeros)."""
    import scipy.sparse as sp
    lib = _ffi.load()
    device = device or require_cuda()
    a = a_csc if sp.issparse(a_csc) and a_csc.format == "csc" else sp.csc_array(a_csc)
    if np.iscomplexobj(a.data):
        return None
    rb = int(lib.mf_spmm_window_rows_per_block())
    lo, hi = (0, a.shape[1]) if row_range is None else row_range
    indptr = np.asarray(a.indptr)
    s, e = int(indptr[lo]), int(indptr[hi])
    rowptr = (indptr[lo:hi + 1] - indptr[lo]).astype(np.int64)
    cols = np.asarray(a.indices[s:e]).astype(np.int64) - col_offset
    nrows = hi - lo
    counts = np.diff(rowptr)
    if nrows == 0 or counts.max(initial=0) > int(lib.mf_spmm_window_max_nnz_per_row()):
        return None
    nblocks = (nrows + rb - 1) // rb
    blk = np.repeat(np.arange(nrows, dtype=np.int64) // rb, counts)
    ncols = int(a.shape[0])
    key = blk * ncols + cols
    ukey, inv = np.unique(key, return_inverse=True)
    ublk = ukey // ncols
    wstart = np.searchsorted(ublk, np.arange(nblocks + 1, dtype=np.int64)).astype(np.int64)
    wmax = int(np.diff(wstart).max(initial=0))
    if wmax > int(lib.mf_spmm_window_max_rows()):
        return None
    slot = (inv - wstart[blk]).astype(np.uint8)
    return DeviceWindows(upload(np.ascontiguousarray(rowptr.astype(np.int32)), device), upload(np.ascontiguousarray(slot), device),
                         upload(np.ascontiguousarray(a.data[s:e], dtype=np.float64), device),
                         upload(np.ascontiguousarray(wstart.astype(np.int32)), device),
                         upload(np.ascontiguousarray((ukey % ncols).astype(np.int32)), device), nrows, max(wmax, 1), int(e - s))


def spmm_window(a: DeviceWindows, q: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``Y = A Q`` through the TMA-staged kernel (Q row windows fetched into shared memory by bulk asynchronous copies)."""
    lib = _ffi.load()
    _check_mat(q, "q")
    r = q.shape[1]
    real = q.dtype == F64
    if out is None:
        out = torch.empty((a.nrows, r), dtype=q.dtype, device=q.device)
    w = 8.0 if real else 16.0
    fn = lib.mf_spmm_window_f64 if real else lib.mf_spmm_window_c128
    with _timed("spmm_window", nbytes=a.nnz * 9.0 + 4.0 * (a.nrows + 1) + 4.0 * a.ucol.numel() + w * r * (a.nrows + q.shape[0]),
                flops=(2.0 if real else 4.0) * a.nnz * r):
        _ffi.check(fn(_ptr(a.rowptr), _ptr(a.slot), _ptr(a.vals), _ptr(a.wstart), _ptr(a.ucol), a.nrows, a.wmax, _ptr(q), q.stride(0), r,
                      _ptr(out), out.stride(0), _stream()), "mf_spmm_window")
    return out


# The two-operator kernel walks the plain CSR pattern.  Measured on B200: r = 64 one pass 0.37 ms against 2 x 0.28 ms (row-grouped,
# G = 4); r = 256 1.10 ms against 2 x 0.46 ms (row-grouped, G = 2) -- the callers use it up to this basis size only.
SPMM2_MAX_R = 128


def same_pattern(a: DeviceCSR, b: DeviceCSR) -> bool:
    """True when two CSR operands were marked as sharing one sparsity pattern (``mark_same_pattern``)."""
    return a is not b and a.pattern_id is not None and a.pattern_id == b.pattern_id


def mark_same_pattern(a: DeviceCSR, b: DeviceCSR, a_host, b_host, row_range=None) -> bool:
    """Compare the host index arrays of two operators ONCE (at upload time, never inside a step) and, if they coincide
    on the uploaded rows, let ``spmm2`` serve both from one pass over the pattern.  Ct and Tt of a FEM model do."""
    if a is None or b is None or a.nrows != b.nrows or a.nnz != b.nnz or a.is_real != b.is_real:
        return False
    lo, hi = (0, a_host.shape[1]) if row_range is None else row_range
    pa, pb = np.asarray(a_host.indptr), np.asarray(b_host.indptr)
    if not np.array_equal(pa[lo:hi + 1], pb[lo:hi + 1]):
        return False
    s0, e0 = int(pa[lo]), int(pa[hi])
    if not np.array_equal(np.asarray(a_host.indices)[s0:e0], np.asarray(b_host.indices)[s0:e0]):
        return False
    a.pattern_id = b.pattern_id = id(a)
    return True


def spmm2(a0: DeviceCSR, a1: DeviceCSR, q: torch.Tensor, col_offset: int = 0):
    """``(A0 Q, A1 Q)`` for two operands that share one sparsity pattern (``same_pattern``): one pass, every Q row loaded
    once for both (mf_spmm_csr2_*)."""
    lib = _ffi.load()
    _check_mat(q, "q")
    if not same_pattern(a0, a1):
        raise ValueError("spmm2: the operands were not marked as sharing a sparsity pattern")
    r = q.shape[1]
    real = q.dtype == F64
    if real and not a0.is_real:
        raise ValueError("spmm2: a real float64 Q needs real operators")
    y0 = torch.empty((a0.nrows, r), dtype=q.dtype, device=q.device)
    y1 = torch.empty((a0.nrows, r), dtype=q.dtype, device=q.device)
    colidx = a0.colidx if col_offset == 0 else a0.colidx - col_offset
    w = 8.0 if real else 16.0
    valb = 8.0 if a0.is_real else 16.0
    nbytes = a0.nnz * (2 * valb + 4.0) + 4.0 * (a0.nrows + 1) + w * r * (2 * a0.nrows + q.shape[0])
    flops = 2 * (2.0 if real else (4.0 if a0.is_real else 8.0)) * a0.nnz * r
    with _timed("spmm_csr", nbytes=nbytes, flops=flops):
        if real:
            _ffi.check(lib.mf_spmm_csr2_f64(_ptr(a0.rowptr), _ptr(colidx), _ptr(a0.vals), _ptr(a1.vals), a0.nrows, _ptr(q), q.stride(0), r,
                                            _ptr(y0), y0.stride(0), _ptr(y1), y1.stride(0), _stream()), "mf_spmm_csr2_f64")
        else:
            _ffi.check(lib.mf_spmm_csr2_c128(_ptr(a0.rowptr), _ptr(colidx), _ptr(a0.vals), _ptr(a1.vals), int(a0.is_real), a0.nrows,
                                             _ptr(q), q.stride(0), r, _ptr(y0), y0.stride(0), _ptr(y1), y1.stride(0), _stream()),
                       "mf_spmm_csr2_c128")
    return y0, y1


@dataclass
class DeviceCSC:
    colptr: torch.Tensor
    rowidx: torch.Tensor
    vals: torch.Tensor
    nrows: int
    ncols: int

    @property
    def is_real(self) -> bool:
        return self.vals.dtype == torch.float64


def csc_to_device(b_csc, device=None) -> DeviceCSC:
    import scipy.sparse as sp
    device = device or require_cuda()
    b = b_csc if sp.issparse(b_csc) and b_csc.format == "csc" else sp.csc_array(b_csc)
    data = np.asarray(b.data)
    vals = np.ascontiguousarray(data, dtype=np.complex128 if np.iscomplexobj(data) else np.float64)
    return DeviceCSC(upload(np.ascontiguousarray(b.indptr, dtype=np.int32), device),
                     upload(np.ascontiguousarray(b.indices, dtype=np.int32), device),
                     upload(vals, device), b.shape[0], b.shape[1])


def project_rhs(b: DeviceCSC, q: torch.Tensor, row0: int = 0, conj: bool = False) -> torch.Tensor:
    """``q^T b`` (r x m) restricted to the rows ``row0 .. row0 + q.shape[0]`` held locally."""
    lib = _ffi.load()
    _check_mat(q, "q")
    r = q.shape[1]
    if q.dtype == F64:
        if not b.is_real:
            raise ValueError("project_rhs: a real float64 Q needs a real port matrix")
        out = torch.empty((r, b.ncols), dtype=F64, device=q.device)
        _ffi.check(lib.mf_project_rhs_f64(_ptr(b.colptr), _ptr(b.rowidx), _ptr(b.vals), b.ncols, _ptr(q), q.stride(0), r,
                                          row0, q.shape[0], _ptr(out), out.stride(0), _stream()), "mf_project_rhs_f64")
        return out
    out = torch.empty((r, b.ncols), dtype=C128, device=q.device)
    _ffi.check(lib.mf_project_rhs_c128(_ptr(b.colptr), _ptr(b.rowidx), _ptr(b.vals), int(b.is_real), b.ncols, _ptr(q), q.stride(0), r,
                                       row0, q.shape[0], int(conj), _ptr(out), out.stride(0), _stream()), "mf_project_rhs_c128")
    return out


# ------------------------------------------------------------------------------------------------ stage 1
def _allreduce(t: torch.Tensor, group) -> None:
    if group is None:
        return
    import torch.distributed as dist
    dist.all_reduce(torch.view_as_real(t) if t.is_complex() else t, op=dist.ReduceOp.SUM, group=group)


def _small_c128(t: torch.Tensor) -> torch.Tensor:
    """r x r matrices of the real path go through the complex128 factorisation kernels (tiny, off the roofline)."""
    return t if t.dtype == C128 else t.to(C128)


def _like_block(small: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """The small factor in the field of the tall block it multiplies (its imaginary part is exactly zero for real x)."""
    return small if x.dtype == C128 else small.real.contiguous()


class BasisInfo:
    """Diagnostics of the basis stage.  ``sigma`` (singular values of the snapshot block, descending) and
    ``jacobi_sweeps`` are produced on the device and fetched lazily, so that building the basis does not force a
    device->host synchronisation."""

    def __init__(self, sigma, passes, shifts, jacobi_sweeps, kept):
        self._sigma = sigma            # device tensor or ndarray
        self.passes = passes           # Cholesky-QR passes used
        self.shifts = shifts           # diagonal shift used in each pass (0 = plain Cholesky)
        self._sweeps = jacobi_sweeps   # device tensor or int
        self.kept = kept               # columns kept after truncation
        self.flags = None              # optimistic CholeskyQR2: device flag blocks awaiting verification
        self.converged = True          # False when the adaptive Cholesky-QR loop stopped at max_passes
        self.departure = None          # departure from orthonormality seen by the last adaptive pass
        self.q_ready = None            # basis_and_projection(defer_q=True): event to wait for before q is used
        self.keepalive = None          # ... and the operands of the side-stream product, released after that wait

    @property
    def sigma(self) -> np.ndarray:
        if isinstance(self._sigma, torch.Tensor):
            self._sigma = self._sigma.cpu().numpy()
        return self._sigma

    @property
    def jacobi_sweeps(self) -> int:
        if isinstance(self._sweeps, torch.Tensor):
            self._sweeps = int(self._sweeps.item())
        return self._sweeps



# ------------------------------------------------------------------ blocked r x r Cholesky / triangular inverse (r > 112)
_SMALL_NB = 64      # block size: the diagonal blocks run on the single-CTA shared-memory kernels


_FUSED_CHOL_MIN_R = 113   # from this size on the Cholesky and the inverse run as ONE cooperative kernel (mf_chol_inv_upper_c128)


def _potrf_upper(g: torch.Tensor, info: torch.Tensor, want_inverse: bool = False) -> Optional[torch.Tensor]:
    """In-place Cholesky ``G = R^H R`` (R upper) with ``info`` = 0 or the 1-based failing column.  Up to r = 112 one
    shared-memory kernel (returns None: invert with ``_trtri_upper``); above that the fused cooperative kernel, which
    produces ``R^-1`` in the same launch -- returned when ``want_inverse`` (the chain of ~80 small launches a blocked
    driver over the single-CTA kernels needs at r = 256 took 0.8 ms per Cholesky-QR pass)."""
    lib = _ffi.load()
    r = g.shape[0]
    if r < _FUSED_CHOL_MIN_R:
        _ffi.check(lib.mf_potrf_upper_c128(_ptr(g), g.stride(0), r, _ptr(info), _stream()), "mf_potrf_upper_c128")
        return None
    rinv = torch.empty((r, r), dtype=C128, device=g.device)
    nbytes = lib.mf_chol_inv_ws_bytes(r)
    ws = workspaces.get("chol_inv", nbytes, g.device)
    _ffi.check(lib.mf_chol_inv_upper_c128(_ptr(g), g.stride(0), r, _ptr(rinv), rinv.stride(0), _ptr(info), _ptr(ws), nbytes, _stream()),
               "mf_chol_inv_upper_c128")
    return rinv if want_inverse else None


def _unequilibrate(g: torch.Tensor, d: torch.Tensor, rinv_eq: Optional[torch.Tensor]) -> torch.Tensor:
    """``R = Rtilde D^-1`` in place (undo the equilibration ``G <- D G D``) and ``R^-1 = D Rtilde^-1``: from the fused
    kernel's inverse when there is one, else by the triangular-inverse kernel."""
    lib = _ffi.load()
    r = g.shape[0]
    _ffi.check(lib.mf_scale_cols_c128(_ptr(g), g.stride(0), r, r, _ptr(d), -1, _stream()), "mf_scale_cols_c128")
    if rinv_eq is None:
        return _trtri_upper(g)
    _ffi.check(lib.mf_scale_rows_c128(_ptr(rinv_eq), rinv_eq.stride(0), r, r, _ptr(d), 1, _stream()), "mf_scale_rows_c128")
    return rinv_eq


def _trtri_upper(rm: torch.Tensor) -> torch.Tensor:
    """``R^-1`` of an upper-triangular matrix: shared-memory kernel up to r = 96, above that the 2 x 2 block recursion
    ``[[A, B], [0, C]]^-1 = [[A^-1, -A^-1 B C^-1], [0, C^-1]]`` on top of it."""
    lib = _ffi.load()
    r = rm.shape[0]
    out = torch.zeros((r, r), dtype=C128, device=rm.device)

    def rec(lo: int, hi: int) -> None:
        n = hi - lo
        if n <= 96:
            blk = rm[lo:hi, lo:hi]
            tgt = out[lo:hi, lo:hi]
            _ffi.check(lib.mf_trtri_upper_c128(_ptr(blk), rm.stride(0), n, _ptr(tgt), out.stride(0), _stream()), "mf_trtri_upper_c128")
            return
        mid = lo + (n // 2 + _SMALL_NB - 1) // _SMALL_NB * _SMALL_NB
        rec(lo, mid)
        rec(mid, hi)
        t = gemm_nn(out[lo:mid, lo:mid].contiguous(), rm[lo:mid, mid:hi].contiguous())     # A^-1 B
        out[lo:mid, mid:hi] = -gemm_nn(t, out[mid:hi, mid:hi].contiguous())                 # -(A^-1 B) C^-1

    if r <= 96:
        _ffi.check(lib.mf_trtri_upper_c128(_ptr(rm), rm.stride(0), r, _ptr(out), out.stride(0), _stream()), "mf_trtri_upper_c128")
    else:
        rec(0, r)
    return out

@dataclass
class CholQR:
    """Result of the Cholesky-QR passes: ``S = x @ r_tot`` with ``x @ rinv`` orthonormal to rounding
    (``rinv`` inverts the triangular factor of the LAST pass, whose input was ``x``)."""
    x: torch.Tensor
    r_tot: torch.Tensor
    rinv: torch.Tensor
    passes: int
    shifts: list
    flags: Optional[torch.Tensor] = None     # optimistic mode: (passes, 32) uint8 flag blocks still to be verified
    converged: bool = True                   # adaptive mode: False when max_passes ended the loop (a RuntimeWarning was raised)
    departure: Optional[float] = None        # adaptive mode: max |G_ij - delta_ij| of the equilibrated Gram matrix of the last pass


def flags_ok(flags_host: torch.Tensor) -> bool:
    """Deferred verification of an optimistic CholeskyQR2: every Cholesky succeeded and the input of the LAST pass was
    already near-orthonormal (departure < 0.1), i.e. exactly the conditions the adaptive loop tests pass by pass."""
    ok = True
    n = flags_host.shape[0]
    for p in range(n):
        ok = ok and int(flags_host[p, 16:20].view(torch.int32)[0]) == 0
    dep = float(flags_host[n - 1, :8].view(torch.float64)[0])
    return ok and dep < 0.1


def _cholesky_qr2_optimistic(s: torch.Tensor, group=None) -> CholQR:
    """Plain CholeskyQR2 (two passes, no shift) with NO device->host read: the success flags stay on the device
    and are verified later (``flags_ok``).  This is the launch sequence CUDA-graph capture records."""
    lib = _ffi.load()
    dev = s.device
    n_loc, r = s.shape
    d = torch.empty(r, dtype=torch.float64, device=dev)
    flags = torch.zeros((2, 32), dtype=torch.uint8, device=dev)
    x, r_tot, rinv = s, None, None
    for p in range(2):
        g = gemm_tn(x, x, conj=True)
        _allreduce(g, group)
        g = _small_c128(g)
        stats = flags[p, :16].view(torch.float64)
        info = flags[p, 16:20].view(torch.int32)
        _ffi.check(lib.mf_equilibrate_c128(_ptr(g), g.stride(0), r, 0.0, _ptr(d), _ptr(stats), _stream()), "mf_equilibrate_c128")
        rinv = _unequilibrate(g, d, _potrf_upper(g, info, want_inverse=True))
        r_tot = g if r_tot is None else gemm_nn(g, r_tot)
        if p == 0:
            x = gemm_nn(x, _like_block(rinv, x), w_upper=True)
    return CholQR(x, r_tot, rinv, 2, [0.0, 0.0], flags)


def cholesky_qr(s: torch.Tensor, group=None, max_passes: int = 6, optimistic: bool = False) -> CholQR:
    """Cholesky-QR passes ``G = X^H X`` (DMMA, all-reduced over row shards) -> equilibrated (shifted if needed)
    Cholesky -> ``X <- X R^-1`` until the input of a pass is already near-orthonormal (CholeskyQR2, or shifted
    CholeskyQR3 for cond(S) >~ 1e8).  The last pass is NOT applied: the caller folds ``rinv`` into the rotation."""
    lib = _ffi.load()
    _check_mat(s, "s")
    if optimistic:
        return _cholesky_qr2_optimistic(s, group)
    dev = s.device
    n_loc, r = s.shape
    eps = np.finfo(np.float64).eps
    d = torch.empty(r, dtype=torch.float64, device=dev)
    # one 32-byte flag block so that a pass costs ONE device->host read: [0:16) stats (2 doubles), [16:20) potrf info
    flags = torch.zeros(32, dtype=torch.uint8, device=dev)
    stats = flags[:16].view(torch.float64)
    info = flags[16:20].view(torch.int32)
    x = s
    r_tot = None
    shifts = []
    bufs = [None, None]
    for p in range(max_passes):
        g = gemm_tn(x, x, conj=True)
        _allreduce(g, group)
        g = _small_c128(g)
        shift = 0.0
        while True:
            gw = g.clone()
            _ffi.check(lib.mf_equilibrate_c128(_ptr(gw), gw.stride(0), r, shift, _ptr(d), _ptr(stats), _stream()), "mf_equilibrate_c128")
            rinv_eq = _potrf_upper(gw, info, want_inverse=True)
            host_flags = flags.cpu()
            if int(host_flags[16:20].view(torch.int32)[0]) == 0:
                break
            shift = 64.0 * eps * r if shift == 0.0 else shift * 100.0
            if shift > 1e-2:
                raise _ffi.MorfemB200Error("orthonormalize: Cholesky breakdown persists (snapshot block numerically rank deficient "
                                           "beyond what shifted CholeskyQR can repair)")
        shifts.append(shift)
        departure = float(host_flags[:8].view(torch.float64)[0])
        # R = Rtilde D^-1 (undo the equilibration), Rinv = R^-1
        rinv = _unequilibrate(gw, d, rinv_eq)
        r_tot = gw if r_tot is None else gemm_nn(gw, r_tot)
        converged = departure < 0.1 and shift == 0.0
        if converged or p == max_passes - 1:
            if not converged:
                import warnings
                warnings.warn(f"orthonormalize: the Cholesky-QR passes did not reach a near-orthonormal block after {max_passes} passes "
                              f"(departure {departure:.2e}, last shift {shift:.1e}); the basis may be less orthonormal than the reference's SVD "
                              "(snapshot block numerically rank deficient)", RuntimeWarning, stacklevel=3)
            return CholQR(x, r_tot, rinv, p + 1, shifts, None, converged, departure)
        tgt = p % 2
        if bufs[tgt] is None:
            bufs[tgt] = torch.empty((n_loc, r), dtype=s.dtype, device=dev)
        x = gemm_nn(x, _like_block(rinv, x), out=bufs[tgt], w_upper=True)
    raise AssertionError("unreachable")


def basis_rotation(cq: CholQR, truncation_tol: float = 0.0) -> tuple[torch.Tensor, BasisInfo]:
    """One-sided Jacobi SVD of the accumulated triangular factor ``r_tot = U_r Sigma V^H``; returns
    ``w = rinv @ U_r[:, :keep]`` so that the basis is ``q = x @ w`` (columns ordered like the left singular vectors
    of the snapshot block, ``truncation_tol > 0`` drops directions with ``sigma_j <= tol * sigma_0``)."""
    lib = _ffi.load()
    r_tot = cq.r_tot
    dev = r_tot.device
    r = r_tot.shape[0]
    eps = np.finfo(np.float64).eps
    u = torch.empty((r, r), dtype=C128, device=dev)
    sigma = torch.empty(r, dtype=torch.float64, device=dev)
    sweeps = torch.zeros(1, dtype=torch.int32, device=dev)
    nbytes = lib.mf_jacobi_svd_ws_bytes(r)
    ws = workspaces.get("jacobi", nbytes, dev)
    if cq.x.dtype == F64 and lib.mf_jacobi_svd_f64_supported(r):
        # real block: the triangular factor is real; the real rotation kernel does half the FP64 work
        r_real = r_tot.real.contiguous()
        u_real = torch.empty((r, r), dtype=F64, device=dev)
        with _timed("jacobi_svd"):
            _ffi.check(lib.mf_jacobi_svd_f64(_ptr(r_real), r_real.stride(0), r, _ptr(u_real), u_real.stride(0), _ptr(sigma), 40, 4.0 * eps,
                                             _ptr(sweeps), _stream()), "mf_jacobi_svd_f64")
        u = u_real.to(C128)
    else:
        r_work = r_tot.clone()           # the SVD destroys its input; keep r_tot (S = x r_tot) for the caller
        with _timed("jacobi_svd"):
            _ffi.check(lib.mf_jacobi_svd_c128(_ptr(r_work), r_work.stride(0), r, _ptr(u), u.stride(0), _ptr(sigma), 40, 4.0 * eps,
                                              _ptr(sweeps), _ptr(ws), ws.numel(), _stream()), "mf_jacobi_svd_c128")
    keep = r
    if truncation_tol > 0.0:
        sig = sigma.cpu().numpy()
        if sig[0] > 0.0:
            keep = max(1, int(np.count_nonzero(sig > truncation_tol * sig[0])))
    w = gemm_nn(cq.rinv, u[:, :keep] if keep < r else u)
    info = BasisInfo(sigma, cq.passes, cq.shifts, sweeps, keep)
    info.converged, info.departure = cq.converged, cq.departure
    return w, info


def orthonormalize(s: torch.Tensor, truncation_tol: float = 0.0, group=None, n_global: Optional[int] = None,
                   max_passes: int = 6) -> tuple[torch.Tensor, BasisInfo]:
    """Orthonormal basis of span(S) with columns ordered like the left singular vectors of S.

    B200 replacement of ``np.linalg.svd(S, full_matrices=False)[0]`` (implementation.py:226/298/210):
    ``cholesky_qr`` (CholeskyQR2 / shifted CholeskyQR3), then ``basis_rotation`` (SVD of the small triangular
    factor) whose rotation is folded into the last application ``q = x @ w``.  Columns of the result equal the
    reference's ``U`` up to sign (rotations inside clustered singular subspaces).  ``truncation_tol > 0`` drops
    directions with ``sigma_j <= tol * sigma_0`` (default 0 keeps all r, like the reference).
    """
    cq = cholesky_qr(s, group=group, max_passes=max_passes)
    w, info = basis_rotation(cq, truncation_tol)
    q = gemm_nn(cq.x, _like_block(w, cq.x))
    return q, info


_side_streams = {}
_upload_streams = {}


def upload_stream(dev) -> "torch.cuda.Stream":
    """Per-device stream for host->device copies that should overlap with compute on the current stream."""
    st = _upload_streams.get(str(dev))
    if st is None:
        st = _upload_streams[str(dev)] = torch.cuda.Stream(device=dev)
    return st



def basis_and_projection(s: torch.Tensor, project_block, group=None, truncation_tol: float = 0.0, optimistic: bool = False,
                         defer_q: bool = False, want_q: bool = True):
    """Stages 1 + 2 with the small-matrix work taken off the critical path.

    ``project_block(x)`` must return ``(g_list, bt)``: the (all-reduced) r x r products ``x^T (A_i x)`` for every
    operator (``None`` for zero operators) and ``x^T b``, for the UN-ROTATED Cholesky-QR block ``x``.  Because the
    basis is ``q = x w`` with a small r x r' matrix ``w`` (inverse triangular factor times the SVD rotation),
    ``q^T A q = w^T (x^T A x) w``: the SpMMs and the long contractions do not wait for the Jacobi SVD, which runs
    (with ``q = x w`` itself) on a side stream concurrently with them.  Returns ``(q, [a_i_r], b_r, BasisInfo)``.

    The reduced operators only need ``w``: the current stream waits for the rotation, not for the tall product ``q = x w``,
    which keeps running on the side stream under the small ``w^T (.) w`` products.  With ``defer_q`` the current stream is
    not joined with it at all: ``info.q_ready`` is the event to wait for before ``q`` is used (or the step ends) -- the
    caller launches the sweep first.  ``want_q=False`` skips ``q`` (callers that only need the reduced model).
    """
    dev = s.device
    cq = cholesky_qr(s, group=group, optimistic=optimistic)
    main = torch.cuda.current_stream()
    side = _side_streams.get(str(dev))
    if side is None:
        side = _side_streams[str(dev)] = torch.cuda.Stream(device=dev)
    ev0 = torch.cuda.Event()
    ev0.record(main)
    g_list, bt = project_block(cq.x)                     # queued on the main stream
    side.wait_event(ev0)
    with torch.cuda.stream(side):
        w, info = basis_rotation(cq, truncation_tol)
        w = _like_block(w, cq.x)
        ev_w = torch.cuda.Event()
        ev_w.record(side)
        q = gemm_nn(cq.x, w) if want_q else None
        ev1 = torch.cuda.Event()
        ev1.record(side)
    main.wait_event(ev_w)
    if not torch.cuda.is_current_stream_capturing():
        for t in (w, q, info._sigma, info._sweeps):
            if isinstance(t, torch.Tensor):
                t.record_stream(main)
    # (for a real block the reduced model stays float64: the sweep has a real twin)
    reduced = [None if g is None else gemm_nn(gemm_tn(w, g, conj=False), w) for g in g_list]
    b_r = gemm_tn(w, bt, conj=False)
    info.flags = cq.flags            # None unless optimistic: the caller verifies with flags_ok(flags.cpu())
    info.q_ready = None
    info.keepalive = None
    if defer_q and want_q:
        info.q_ready = ev1           # the caller joins: current_stream().wait_event(info.q_ready)
        # the side stream is still reading the un-rotated block (cq.x, allocated on the main stream) when this function
        # returns: keep it referenced until the caller has joined, otherwise the caching allocator may hand its memory to
        # the next main-stream allocation (the sweep outputs) while `q = x w` is in flight -- also inside a captured graph
        info.keepalive = cq
    else:
        main.wait_event(ev1)
    return q, reduced, b_r, info


# ------------------------------------------------------------------------------------------- stages 3 + 4
@dataclass
class SweepResult:
    x: Optional[torch.Tensor]       # (F, r, m) complex128 or None
    gsm: Optional[torch.Tensor]     # (F, m, m) complex128 or None
    info: torch.Tensor              # (F,) int32: 0 or 1-based index of the first zero pivot


def sweep(a0s: Optional[torch.Tensor], a1s: Optional[torch.Tensor], a2s: Optional[torch.Tensor], br: torch.Tensor,
          c0: torch.Tensor, c1: torch.Tensor, c2: torch.Tensor, cb: torch.Tensor, zscale: Optional[torch.Tensor],
          want_x: bool = True, want_gsm: bool = True, variant: int = 0,
          x_out: Optional[torch.Tensor] = None, gsm_out: Optional[torch.Tensor] = None) -> SweepResult:
    """Batched reduced solves + S-parameters for the points described by the coefficient arrays.

    Operators must already be symmetrised (``symmetrize``); ``None`` stands for an all-zero operator (the
    reference projects and adds an empty ``a1`` -- test_helpers.py:57 -- which contributes exactly zero).
    """
    lib = _ffi.load()
    ops = [o for o in (a0s, a1s, a2s) if o is not None]
    if not ops:
        raise ValueError("sweep: all operators are None")
    for o in ops:
        _check_mat(o, "operator")
    _check_mat(br, "br")
    r, m = br.shape
    if all(o.dtype == F64 for o in ops) and br.dtype == F64:
        if variant in (0, 3, 5) and lib.mf_sweep_f64_variant_supported(r, m, variant):
            return _sweep_f64(lib, a0s, a1s, a2s, br, c0, c1, c2, cb, zscale, want_x, want_gsm, variant)
        a0s, a1s, a2s = (None if o is None else o.to(C128) for o in (a0s, a1s, a2s))     # no real kernel for this shape
        br = br.to(C128)
        ops = [o for o in (a0s, a1s, a2s) if o is not None]
    elif any(o.dtype != C128 for o in ops) or br.dtype != C128:
        raise ValueError("sweep: operators and port matrix must share a dtype (all float64 or all complex128)")
    lda = ops[0].stride(0)
    if any(o.stride(0) != lda or o.shape != (r, r) for o in ops):
        raise ValueError("sweep: operators must share shape (r, r) and leading dimension")
    nf = int(c0.numel())
    dev = br.device
    for c in (c0, c1, c2, cb) + ((zscale,) if zscale is not None else ()):
        if c.dtype != torch.float64 or not c.is_cuda or c.numel() != nf or not c.is_contiguous():
            raise ValueError("sweep: coefficient arrays must be contiguous float64 CUDA tensors of equal length")
    x = (x_out if x_out is not None else torch.empty((nf, r, m), dtype=C128, device=dev)) if want_x else None
    gsm = (gsm_out if gsm_out is not None else torch.empty((nf, m, m), dtype=C128, device=dev)) if want_gsm else None
    info = torch.zeros(nf, dtype=torch.int32, device=dev)
    nbytes = lib.mf_sweep_ws_bytes(r, m, nf, variant)
    ws = workspaces.get("sweep", nbytes, dev)
    flops_pt = (8.0 / 3.0) * r ** 3 + 8.0 * r * r * m + 16.0 * r * r + 8.0 * r * m * m
    bytes_pt = 16.0 * m * m * (gsm is not None) + 16.0 * r * m * (x is not None) + 40.0 + 4.0
    with _timed("sweep_lu_gsm", nbytes=bytes_pt * nf, flops=flops_pt * nf):
        _ffi.check(lib.mf_sweep_lu_gsm_c128(_ptr(a0s), _ptr(a1s), _ptr(a2s), lda, _ptr(br), br.stride(0), r, m,
                                            _ptr(c0), _ptr(c1), _ptr(c2), _ptr(cb), _ptr(zscale), nf,
                                            _ptr(x), _ptr(gsm), _ptr(info), variant, _ptr(ws), ws.numel(), _stream()),
                   "mf_sweep_lu_gsm_c128")
    return SweepResult(x, gsm, info)


def _sweep_f64(lib, a0s, a1s, a2s, br, c0, c1, c2, cb, zscale, want_x, want_gsm, variant=0) -> SweepResult:
    """Real reduced model: the float64 twins of the blocked kernels (half the bytes, a quarter of the flops)."""
    ops = [o for o in (a0s, a1s, a2s) if o is not None]
    r, m = br.shape
    lda = ops[0].stride(0)
    if any(o.stride(0) != lda or o.shape != (r, r) for o in ops):
        raise ValueError("sweep: operators must share shape (r, r) and leading dimension")
    nf = int(c0.numel())
    dev = br.device
    x = torch.empty((nf, r, m), dtype=F64, device=dev) if want_x else None
    gsm_ = torch.empty((nf, m, m), dtype=C128, device=dev) if want_gsm else None
    info = torch.zeros(nf, dtype=torch.int32, device=dev)
    flops_pt = (2.0 / 3.0) * r ** 3 + 2.0 * r * r * m + 4.0 * r * r + 2.0 * r * m * m
    bytes_pt = 16.0 * m * m * (gsm_ is not None) + 8.0 * r * m * (x is not None) + 40.0 + 4.0
    nbytes = lib.mf_sweep_f64_ws_bytes(r, m, nf, variant)
    ws = workspaces.get("sweep", nbytes, dev)
    with _timed("sweep_lu_gsm", nbytes=bytes_pt * nf, flops=flops_pt * nf):
        _ffi.check(lib.mf_sweep_lu_gsm_f64(_ptr(a0s), _ptr(a1s), _ptr(a2s), lda, _ptr(br), br.stride(0), r, m,
                                           _ptr(c0), _ptr(c1), _ptr(c2), _ptr(cb), _ptr(zscale), nf, _ptr(x), _ptr(gsm_), _ptr(info),
                                           variant, _ptr(ws), ws.numel(), _stream()),
                   "mf_sweep_lu_gsm_f64")
    return SweepResult(x, gsm_, info)


def gsm(x: torch.Tensor, bmat: torch.Tensor, cb: torch.Tensor, zscale: torch.Tensor) -> torch.Tensor:
    """Stage 4 alone: S-parameters from given solutions ``x`` (F, r, m) and port matrix ``bmat`` (r, m)."""
    lib = _ffi.load()
    nf, r, m = x.shape
    out = torch.empty((nf, m, m), dtype=C128, device=x.device)
    _ffi.check(lib.mf_gsm_c128(_ptr(x), _ptr(bmat), bmat.stride(0), r, m, _ptr(cb), _ptr(zscale), nf, _ptr(out), _stream()), "mf_gsm_c128")
    return out


def estimator(x: torch.Tensor, g_blocks, h_blocks, bb: Optional[torch.Tensor],
              c0: torch.Tensor, c1: torch.Tensor, c2: torch.Tensor, cb: torch.Tensor) -> torch.Tensor:
    """Greedy residual estimator (implementation.py:424-441) for all points; ``g_blocks`` is a 3x3 nested list and
    ``h_blocks`` a list of 3 device matrices (``None`` = zero block)."""
    lib = _ffi.load()
    nf, r, m = x.shape
    garr = (ctypes.c_void_p * 9)(*[None if g_blocks[a][b] is None else g_blocks[a][b].data_ptr() for a in range(3) for b in range(3)])
    harr = (ctypes.c_void_p * 3)(*[None if h is None else h.data_ptr() for h in h_blocks])
    err = torch.empty(nf, dtype=torch.float64, device=x.device)
    _ffi.check(lib.mf_estimator_c128(_ptr(x), r, m, nf, ctypes.cast(garr, ctypes.c_void_p), ctypes.cast(harr, ctypes.c_void_p), _ptr(bb),
                                     _ptr(c0), _ptr(c1), _ptr(c2), _ptr(cb), _ptr(err), _stream()), "mf_estimator_c128")
    return err
