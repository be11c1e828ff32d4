"""Resident matrices on the B200: thin handle classes over the C-ABI of include/spmv_b200.h.

PyTorch is plumbing only: it owns the dense vectors (x, y), the CUDA streams and -- in
distributed.py -- the process group.  The matrix arenas, plans and every kernel live in
libspmv_b200.so.  Nothing here falls back to PyTorch or the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N

ALGO_AUTO, ALGO_VECTOR, ALGO_TILE, ALGO_STREAM, ALGO_BINNED, ALGO_ROW, ALGO_ROW_IMAGE = 0, 1, 2, 3, 4, 5, 6
ALGO_NAMES = {0: "auto", 1: "csr_vector_kernel", 2: "csr_stream_kernel (ALGO_TILE is retired)", 3: "csr_stream_kernel", 4: "csr_binned_kernel", 5: "csr_row_kernel",
              6: "hll_rowu_kernel / hll_row_kernel / csr_pattern_kernel on the handle's private image (masked padding)"}
HLL_KERNEL_NAMES = {0: "hll_slice_kernel", 1: "hll_stream_kernel", 2: "hll_row_kernel"}
SYNTH_LAP2D, SYNTH_LAP3D, SYNTH_UNIFORM = 1, 2, 3


def _ptr(t):
    """Device (torch tensor) or host (numpy array) pointer as void*."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    return C.c_void_p(t.data_ptr())


def _stream(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


def _check_vec(t, n, what, dtype="float64"):
    """A device vector the kernels may read or write n elements of: a contiguous CUDA tensor of `dtype`."""
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == getattr(torch, dtype) and t.is_contiguous()
            and t.numel() >= n):
        raise ValueError(f"{what} must be a contiguous {dtype} CUDA tensor with at least {n} elements")


def _host_vectors(x, y, n, m, dtype):
    """x and y of a host round trip: x is converted to `dtype` and must hold n elements; a caller's y is written in place,
    so it must already be a contiguous numpy array of `dtype` with m elements."""
    x = np.ascontiguousarray(x, dtype)
    if x.ndim != 1 or x.size != n:
        raise ValueError(f"x must be a vector of {n} elements (got shape {x.shape})")
    if y is None:
        return x, np.zeros(m, dtype)
    if not (isinstance(y, np.ndarray) and y.dtype == dtype and y.ndim == 1 and y.size == m and y.flags.c_contiguous
            and y.flags.writeable):
        raise ValueError(f"y must be a writable contiguous {np.dtype(dtype).name} numpy vector of {m} elements")
    return x, y


def _check_dense(t, rows, what, dtype="float64"):
    """A row-major block of a multi-vector product: a 2-D CUDA tensor of `dtype` with `rows` rows whose columns are
    adjacent (column stride 1) and whose row stride, the leading dimension, is at least the column count.  Strides
    of dimensions of size 1 do not matter, as in torch.  Returns (columns, leading dimension)."""
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == getattr(torch, dtype) and t.dim() == 2):
        raise ValueError(f"{what} must be a 2-D {dtype} CUDA tensor")
    n, k = t.shape
    if n != rows:
        raise ValueError(f"{what} must have {rows} rows (got shape {tuple(t.shape)})")
    if k > 1 and t.stride(1) != 1:
        raise ValueError(f"{what} must have column stride 1 (got strides {t.stride()})")
    ld = t.stride(0) if n > 1 else k
    if ld < k:
        raise ValueError(f"{what} must have a row stride of at least {k} elements (got {ld})")
    return k, ld


def _dense_overlap(a, lda, b, ldb, k, size=8):
    """Do the row-major k-column blocks a (leading dimension lda) and b (ldb) of `size`-byte elements share an element?
    Exact when the leading dimensions are equal (interleaved column slices of one buffer do not overlap), conservative
    otherwise: then any intersection of the two address ranges counts."""
    if a.numel() == 0 or b.numel() == 0:
        return False
    return _block_overlap(a.data_ptr(), a.shape[0], lda, b.data_ptr(), b.shape[0], ldb, k, size)


def _block_overlap(pa, rows_a, lda, pb, rows_b, ldb, k, size):
    """_dense_overlap on addresses: blocks of rows_a and rows_b rows at pa and pb."""
    if k == 0 or rows_a == 0 or rows_b == 0:
        return False
    ea = pa + size * ((rows_a - 1) * lda + k)
    eb = pb + size * ((rows_b - 1) * ldb + k)
    if ea <= pb or eb <= pa:
        return False
    if lda != ldb or (pb - pa) % size:
        return True
    s = ((pb - pa) // size) % lda  # b's columns sit at residues [s, s + k) modulo ld, a's at [0, k)
    return s < k or s + k > lda


def _spmm_operands(X, Y, M, N_, dtype="float64"):
    k, ldx = _check_dense(X, N_, "X", dtype)
    ky, ldy = _check_dense(Y, M, "Y", dtype)
    if ky != k:
        raise ValueError(f"X and Y must have the same number of columns (got {k} and {ky})")
    if _dense_overlap(X, ldx, Y, ldy, k, X.element_size()):
        raise ValueError("Y must not overlap X")
    return k, ldx, ldy


def _check_host_dense(t, rows, what, dtype, writable=False):
    """A row-major block of a host-buffer multi-vector product: a 2-D numpy array or CPU torch tensor of `dtype` with
    `rows` rows, column stride 1 and a row stride (the leading dimension) of at least the column count, such as
    big[:, :k].  Returns (columns, leading dimension, address)."""
    import torch
    if isinstance(t, np.ndarray):
        if t.dtype != dtype or t.ndim != 2:
            raise ValueError(f"{what} must be a 2-D {np.dtype(dtype).name} array")
        n, k = t.shape
        s0, s1 = t.strides
        if t.size and ((k > 1 and s1 != t.itemsize) or (n > 1 and (s0 < 0 or s0 % t.itemsize))):
            raise ValueError(f"{what} must have column stride 1 and a positive row stride (got strides {t.strides} in bytes)")
        if writable and not t.flags.writeable:
            raise ValueError(f"{what} must be writable")
        ld, addr = (s0 // t.itemsize if n > 1 and t.size else k), t.ctypes.data
    elif isinstance(t, torch.Tensor):
        if t.device.type != "cpu" or t.dtype != getattr(torch, np.dtype(dtype).name) or t.dim() != 2:
            raise ValueError(f"{what} must be a 2-D {np.dtype(dtype).name} CPU tensor")
        n, k = t.shape
        if t.numel() and k > 1 and t.stride(1) != 1:
            raise ValueError(f"{what} must have column stride 1 (got strides {t.stride()})")
        ld, addr = (t.stride(0) if n > 1 and t.numel() else k), t.data_ptr()
    else:
        raise ValueError(f"{what} must be a numpy array or a CPU torch tensor")
    if n != rows:
        raise ValueError(f"{what} must have {rows} rows (got shape {tuple(t.shape)})")
    if ld < k:
        raise ValueError(f"{what} must have a row stride of at least {k} elements (got {ld})")
    return k, ld, addr or _NO_ROWS.ctypes.data  # an empty torch tensor has no address; its rows are never read


_NO_ROWS = np.zeros(1)


def _host_spmm_operands(X, Y, M, N_, dtype):
    """Checks X (N_ x k) and Y (M x k, allocated like X when None: numpy, or a torch tensor pinned when X is) of a
    host-buffer product.  Returns (Y, k, ldx, x address, ldy, y address)."""
    import torch
    k, ldx, px = _check_host_dense(X, N_, "X", dtype)
    if Y is None:
        if isinstance(X, np.ndarray):
            Y = np.zeros((M, k), dtype)
        else:
            Y = torch.zeros((M, k), dtype=X.dtype, pin_memory=X.is_pinned())
    ky, ldy, py = _check_host_dense(Y, M, "Y", dtype, writable=True)
    if ky != k:
        raise ValueError(f"X and Y must have the same number of columns (got {k} and {ky})")
    if _block_overlap(px, N_, ldx, py, M, ldy, k, np.dtype(dtype).itemsize):
        raise ValueError("Y must not overlap X")
    return Y, k, ldx, px, ldy, py


FORMAT_CSR, FORMAT_HLL = 0, 1


def row_forms(fmt: int):
    """The multi-row forms of the row kernels, [(rows per thread | hacks per warp, batch, CTAs per SM), ...]: form k is
    what SPMV_B200_ROW_MULTI=k+1 forces and what id 16+k of spmv_b200_{csr,hll}_row_form_f32 names."""
    out = []
    for k in range(N.lib().spmv_b200_row_forms(fmt)):
        r, b, c = C.c_int(), C.c_int(), C.c_int()
        N.check(N.lib().spmv_b200_row_form_describe(fmt, k, C.byref(r), C.byref(b), C.byref(c)))
        out.append((r.value, b.value, c.value))
    return out


def row_form_name(fmt: int, form: int, storage: str = "float") -> str:
    base = "csr_row" if fmt == FORMAT_CSR else "hll_row"
    if form >= 64:  # HLL only: offsets by arithmetic on a regular image
        return f"hll_rowu_kernel<{form - 64},{storage}>"
    if form >= 16:
        r, b, c = row_forms(fmt)[form - 16]
        return f"{base}m_kernel<{b},{r},{c},{storage}>"
    return f"{base}_kernel<{form},{storage}>" if form > 0 else "none"


def device_count() -> int:
    n = C.c_int()
    N.lib().spmv_b200_device_count(C.byref(n))
    return n.value


def device_info():
    name = C.create_string_buffer(256)
    sm, l2, mem = C.c_int(), C.c_longlong(), C.c_longlong()
    N.check(N.lib().spmv_b200_device_info(name, 256, C.byref(sm), C.byref(l2), C.byref(mem)))
    return {"name": name.value.decode(), "sm_count": sm.value, "l2_bytes": l2.value, "mem_bytes": mem.value}


class DeviceCSR:
    """A CSR matrix resident in HBM plus its row-binning plan (spmv_b200_csr)."""

    def __init__(self, handle, keepalive=None):
        self._h = handle
        self._keep = keepalive

    # -- construction ------------------------------------------------------------------------------
    @classmethod
    def upload(cls, M, N_, row_ptr, col_idx, values):
        """Host CSR arrays (reference CSRMatrix fields) -> device.  reference main_cuda.cu:135-145."""
        row_ptr = np.ascontiguousarray(row_ptr, np.int32)
        col_idx = np.ascontiguousarray(col_idx, np.int32)
        values = np.ascontiguousarray(values, np.float64)
        h = C.c_void_p()
        N.check(N.lib().spmv_b200_csr_upload(int(M), int(N_), int(row_ptr[-1]) if len(row_ptr) else 0,
                                             _ptr(row_ptr), _ptr(col_idx), _ptr(values), C.byref(h)))
        return cls(h)

    @classmethod
    def from_coo(cls, M, N_, I, J, val, stream=None):
        """COO -> CSR built on the device (spmv_b200_csr_from_coo[_device]).  I / J / val: numpy arrays (copied up) or
        CUDA tensors (used in place).  Replaces convert_in_csr (reference src/csr_matrix.c:63-126) for resident data."""
        h = C.c_void_p()
        if isinstance(I, np.ndarray):
            I = np.ascontiguousarray(I, np.int32)
            J = np.ascontiguousarray(J, np.int32)
            val = np.ascontiguousarray(val, np.float64)
            N.check(N.lib().spmv_b200_csr_from_coo(int(M), int(N_), int(len(I)), _ptr(I), _ptr(J), _ptr(val), C.byref(h)))
        else:
            N.check(N.lib().spmv_b200_csr_from_coo_device(int(M), int(N_), int(I.numel()), _ptr(I), _ptr(J), _ptr(val),
                                                          _stream(stream), C.byref(h)))
        return cls(h)

    @classmethod
    def from_host(cls, csr):
        """From a host.CSRMatrix produced by convert_in_csr."""
        return cls.upload(csr.M, csr.N, csr.row_ptr, csr.col_idx, csr.values)

    @classmethod
    def wrap(cls, M, N_, row_ptr, col_idx, values, stream=None):
        """CUDA tensors (int32, int32, float64) used in place; they must outlive this object."""
        h = C.c_void_p()
        N.check(N.lib().spmv_b200_csr_wrap_device(int(M), int(N_), int(values.numel()), _ptr(row_ptr), _ptr(col_idx),
                                                  _ptr(values), _stream(stream), C.byref(h)))
        return cls(h, keepalive=(row_ptr, col_idx, values))

    @classmethod
    def synth(cls, kind, p0, p1=0, p2=0, seed=0x5EED, row_begin=0, row_end=None, stream=None):
        """Rows [row_begin,row_end) of a synthetic matrix, generated on the device."""
        if row_end is None:
            row_end = {SYNTH_LAP2D: p0 * p0, SYNTH_LAP3D: p0 ** 3, SYNTH_UNIFORM: p0}[kind]
        h = C.c_void_p()
        N.check(N.lib().spmv_b200_synth_csr(kind, int(p0), int(p1), int(p2), int(seed), int(row_begin), int(row_end),
                                            _stream(stream), C.byref(h)))
        return cls(h)

    # -- introspection -----------------------------------------------------------------------------
    def info(self) -> N.CsrInfo:
        i = N.CsrInfo()
        N.check(N.lib().spmv_b200_csr_info(self._h, C.byref(i)))
        return i

    @property
    def shape(self):
        i = self.info()
        return i.M, i.N

    @property
    def nnz(self):
        return self.info().nnz

    def replan(self, tile_items=0, long_threshold=0, threads_per_row=0, stream=None):
        N.check(N.lib().spmv_b200_csr_replan(self._h, tile_items, long_threshold, threads_per_row, _stream(stream)))
        return self

    def download(self):
        i = self.info()
        row_ptr = np.zeros(i.M + 1, np.int32)
        col_idx = np.zeros(i.nnz, np.int32)
        values = np.zeros(i.nnz, np.float64)
        N.check(N.lib().spmv_b200_csr_download(self._h, _ptr(row_ptr), _ptr(col_idx), _ptr(values)))
        return row_ptr, col_idx, values

    # -- products ----------------------------------------------------------------------------------
    def spmv(self, x, y, accumulate=False, algo=ALGO_AUTO, stream=None):
        """y = A x (or y += A x) on CUDA tensors, asynchronous on ``stream``."""
        i = self.info()
        _check_vec(x, i.N, "x")
        _check_vec(y, i.M, "y")
        N.check(N.lib().spmv_b200_csr_spmv(self._h, _ptr(x), _ptr(y), int(bool(accumulate)), algo, _stream(stream)))
        return y

    def spmm(self, X, Y, accumulate=False, stream=None):
        """Y = A X (or Y += A X) for X of shape (N, k) and Y of shape (M, k): float64 CUDA tensors, row-major with column
        stride 1 and row stride >= k, so column slices such as Xbig[:, a:a+k] work.  One pass over the matrix for all
        k columns (spmv_b200_csr_spmm): each column bit for bit the serial loop on rows up to the long-row threshold.
        Asynchronous on ``stream``; raises ValueError before any launch on a bad or overlapping operand."""
        i = self.info()
        k, ldx, ldy = _spmm_operands(X, Y, i.M, i.N)
        if k and i.M:
            N.check(N.lib().spmv_b200_csr_spmm(self._h, k, _ptr(X), ldx, _ptr(Y), ldy, int(bool(accumulate)), _stream(stream)))
        return Y

    def partials_count(self) -> int:
        return N.lib().spmv_b200_csr_partials_count(self._h)

    def spmv_fused(self, x_ptr, y_ptr, prev_sumsq=None, partials=None, peers=None, stream=None):
        """y = (A x) / sqrt(*prev_sumsq), partials[cta] = sum y^2, boundary rows mirrored into peer memory.
        x_ptr / y_ptr are raw device addresses (ints) or tensors."""
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_csr_spmv_fused(self._h, raw(x_ptr), raw(y_ptr), raw(prev_sumsq) if prev_sumsq is not None else None,
                                                 raw(partials) if partials is not None else None,
                                                 C.byref(peers) if peers is not None else None, _stream(stream)))

    def flat_partials_count(self) -> int:
        return N.lib().spmv_b200_csr_flat_partials_count(self._h)

    def spmv_fused_flat(self, x_ptr, y_ptr, inv_norm=None, partials=None, peers=None, stream=None):
        """The FLAT fused product of the two-launch iterated product (spmv_b200_csr_spmv_fused_flat): y = (A x) * (*inv_norm)."""
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_csr_spmv_fused_flat(self._h, raw(x_ptr), raw(y_ptr), raw(inv_norm) if inv_norm is not None else None,
                                                      raw(partials) if partials is not None else None,
                                                      C.byref(peers) if peers is not None else None, _stream(stream)))

    def spmv_fused_mail(self, x_ptr, y_ptr, partials, mail, peers=None, stream=None):
        """The fused launch with the |w|^2 exchange through peer mailboxes (spmv_b200_csr_spmv_fused_mail)."""
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_csr_spmv_fused_mail(self._h, raw(x_ptr), raw(y_ptr), raw(partials),
                                                      C.byref(peers) if peers is not None else None, C.byref(mail),
                                                      _stream(stream)))

    def spmv_fused_async(self, x_ptr, y_ptr, partials, exchange, peers=None, stream=None):
        """The asynchronous fused launch (spmv_b200_csr_spmv_fused_async): boundary rows first, lagged scale."""
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_csr_spmv_fused_async(self._h, raw(x_ptr), raw(y_ptr), raw(partials),
                                                       C.byref(peers) if peers is not None else None, C.byref(exchange),
                                                       _stream(stream)))

    def remap_columns(self, starts, stride, stream=None):
        """In place: column c owned by part p (starts[p] <= c < starts[p+1]) becomes p*stride + c - starts[p]; the matrix
        then has len(starts)-1 times stride columns (spmv_b200_csr_remap_columns: the padded x of the one-collective
        allgather refresh)."""
        arr = (C.c_longlong * len(starts))(*[int(v) for v in starts])
        N.check(N.lib().spmv_b200_csr_remap_columns(self._h, len(starts) - 1, arr, int(stride), _stream(stream)))
        return self

    def interior_rows(self, col_lo, col_hi, stream=None):
        """[lo, hi): a contiguous row range whose columns all lie in [col_lo, col_hi) (largest one around the middle row)."""
        lo, hi = C.c_int(), C.c_int()
        N.check(N.lib().spmv_b200_csr_interior_rows(self._h, int(col_lo), int(col_hi), C.byref(lo), C.byref(hi), _stream(stream)))
        return lo.value, hi.value

    def set_image(self, mode, stream=None):
        """mode 0: drop the private column-major image; mode 1: build it with fp64 values on any matrix eligible in
        structure (owned arrays, rows of at most 12 nonzeros), whatever its size or timing; mode 2: the same with 1-byte
        value codes, on a matrix of at most 256 distinct value patterns; mode 3: the pattern form, one byte per row, on a
        matrix of at most 256 distinct rows (spmv_b200_csr_set_image).  Raises SpmvError otherwise, and modes 2 and 3
        then leave the handle as it was."""
        N.check(N.lib().spmv_b200_csr_set_image(self._h, int(mode), _stream(stream)))
        return self

    def image_form(self) -> str:
        """Name of the kernel that multiplies the private image, index type and, for the value codes, the stored value
        type included ("none" without one)."""
        i = self.info()
        if i.image_patterns > 0:
            return f"csr_pattern_kernel<{i.image_form - 256}>"
        args = "uint16_t" if i.image_index_bytes == 2 else "int"
        if i.image_value_bytes == 1:
            args += ",uint8_t"
        if i.image_form >= 64:
            return f"hll_rowu_kernel<{i.image_form - 64},double,true,{args}>"
        return f"hll_row_kernel<{i.image_form},double,true,{args}>" if i.image_form > 0 else "none"

    def spmv_rows(self, row_begin, row_end, x, y, stream=None):
        i = self.info()
        _check_vec(x, i.N, "x")
        _check_vec(y, i.M, "y")
        N.check(N.lib().spmv_b200_csr_spmv_rows(self._h, int(row_begin), int(row_end), _ptr(x), _ptr(y), _stream(stream)))
        return y

    def spmv_host(self, x, y=None, accumulate=False, algo=ALGO_AUTO):
        """Host numpy x -> H2D, product, D2H -> host numpy y (synchronous): the end-to-end call."""
        i = self.info()
        x, y = _host_vectors(x, y, i.N, i.M, np.float64)
        N.check(N.lib().spmv_b200_csr_spmv_host(self._h, _ptr(x), _ptr(y), int(bool(accumulate)), algo))
        return y

    def spmv_host_ptr(self, x_ptr: int, y_ptr: int, accumulate=False, algo=ALGO_AUTO):
        """Same, on raw host addresses (e.g. pinned torch tensors' data_ptr())."""
        N.check(N.lib().spmv_b200_csr_spmv_host(self._h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), int(bool(accumulate)), algo))

    def spmm_host(self, X, Y=None, accumulate=False):
        """Y = A X (or Y += A X) on host buffers, synchronous (spmv_b200_csr_spmm_host): X of shape (N, k) and Y of
        shape (M, k), float64 numpy arrays or CPU torch tensors with column stride 1 and row stride >= k (views such as
        big[:, :k] work).  Y is written in place, or allocated like X when None; pinned tensors give the overlap of the
        uploads, products and downloads.  Every column has the bits of spmm on the same handle.  Raises ValueError
        before any call on a bad or overlapping operand.  Returns Y."""
        i = self.info()
        Y, k, ldx, px, ldy, py = _host_spmm_operands(X, Y, i.M, i.N, np.float64)
        if k and i.M:
            N.check(N.lib().spmv_b200_csr_spmm_host(self._h, k, C.c_void_p(px), ldx, C.c_void_p(py), ldy, int(bool(accumulate))))
        return Y

    # -- fp32 storage, fp64 arithmetic (SURVEY.md section 8(f).3) ----------------------------------------------
    def enable_f32(self, stream=None):
        N.check(N.lib().spmv_b200_csr_enable_f32(self._h, _stream(stream)))
        return self

    def row_form_f32(self) -> str:
        """Name of the row kernel enable_f32 timed fastest for this matrix (spmv_b200_csr_row_form_f32)."""
        return row_form_name(FORMAT_CSR, N.lib().spmv_b200_csr_row_form_f32(self._h))

    def spmv_f32(self, x, y, accumulate=False, algo=ALGO_AUTO, stream=None):
        """y = A x on float32 CUDA tensors (float values, x, y; products and sums in double)."""
        i = self.info()
        _check_vec(x, i.N, "x", "float32")
        _check_vec(y, i.M, "y", "float32")
        N.check(N.lib().spmv_b200_csr_spmv_f32(self._h, _ptr(x), _ptr(y), int(bool(accumulate)), algo, _stream(stream)))
        return y

    def spmm_f32(self, X, Y, accumulate=False, stream=None):
        """Y = A X (or Y += A X) as spmm, on float32 tensors through the float copy of enable_f32 (products and sums in
        double, one rounding to float per element): on rows up to the long-row threshold each column is bit for bit
        spmv_f32(algo=ALGO_ROW) on that column (spmv_b200_csr_spmm_f32).  SpmvError without enable_f32."""
        i = self.info()
        k, ldx, ldy = _spmm_operands(X, Y, i.M, i.N, "float32")
        if k and i.M:
            N.check(N.lib().spmv_b200_csr_spmm_f32(self._h, k, _ptr(X), ldx, _ptr(Y), ldy, int(bool(accumulate)), _stream(stream)))
        return Y

    def spmv_host_f32(self, x, y=None):
        i = self.info()
        x, y = _host_vectors(x, y, i.N, i.M, np.float32)
        N.check(N.lib().spmv_b200_csr_spmv_host_f32(self._h, _ptr(x), _ptr(y)))
        return y

    def spmm_host_f32(self, X, Y=None, accumulate=False):
        """spmm_host on float32 buffers through the float copy of the values (enabled by the call itself): the bits of
        spmm_f32 on the same handle (spmv_b200_csr_spmm_host_f32).  Returns Y."""
        i = self.info()
        Y, k, ldx, px, ldy, py = _host_spmm_operands(X, Y, i.M, i.N, np.float32)
        if k and i.M:
            N.check(N.lib().spmv_b200_csr_spmm_host_f32(self._h, k, C.c_void_p(px), ldx, C.c_void_p(py), ldy, int(bool(accumulate))))
        return Y

    def algorithmic_bytes_f32(self) -> int:
        i = self.info()
        return 8 * i.nnz + 4 * (i.M + 1) + 4 * i.M + 4 * i.N

    def to_hll(self, stream=None) -> "DeviceHLL":
        h = C.c_void_p()
        N.check(N.lib().spmv_b200_hll_from_csr(self._h, _stream(stream), C.byref(h)))
        return DeviceHLL(h)

    def close(self):
        if self._h:
            N.lib().spmv_b200_csr_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def csr_spmv_raw(M, row_ptr, col_idx, values, x, y, threads_per_row=0, stream=None):
    """Plan-free vector-per-row product on raw CUDA tensors (drop-in for the reference's
    spmv_csr_warp_kernel launch, main_cuda.cu:238)."""
    N.check(N.lib().spmv_b200_csr_spmv_raw(int(M), int(values.numel()), _ptr(row_ptr), _ptr(col_idx), _ptr(values),
                                           _ptr(x), _ptr(y), threads_per_row, _stream(stream)))
    return y


class DeviceHLL:
    """Column-major, hack-aligned HLL image resident in HBM (spmv_b200_hll)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def from_host(cls, hll, M=None, N_=None):
        """From a host.HLLMatrix produced by convert_to_hll (reference row-major layout)."""
        h = C.c_void_p()
        N.check(N.lib().spmv_b200_hll_upload(C.byref(hll.c), int(hll.rows_total if M is None else M),
                                             int(hll.cols if N_ is None else N_), C.byref(h)))
        return cls(h)

    def info(self) -> N.HllInfo:
        i = N.HllInfo()
        N.check(N.lib().spmv_b200_hll_info(self._h, C.byref(i)))
        return i

    def download(self):
        """-> host.HLLMatrix in the reference layout (round trip of from_host)."""
        from .host import HLLMatrix
        out = HLLMatrix()
        N.check(N.lib().spmv_b200_hll_download(self._h, C.byref(out.c)))
        out._owned = True
        i = self.info()
        out.rows_total, out.cols = i.M, i.N
        return out

    def spmv(self, x, y, stream=None, slice_kernel=None):
        """y = A x.  slice_kernel: None = automatic choice, True = one-warp-per-hack slice kernel,
        False = persistent TMA stream kernel, "rows" = lane-per-row kernel in the serial order."""
        i = self.info()
        _check_vec(x, i.N, "x")
        _check_vec(y, i.M, "y")
        fn = {None: N.lib().spmv_b200_hll_spmv, True: N.lib().spmv_b200_hll_spmv_slice,
              False: N.lib().spmv_b200_hll_spmv_stream, "rows": N.lib().spmv_b200_hll_spmv_rows}[slice_kernel]
        N.check(fn(self._h, _ptr(x), _ptr(y), _stream(stream)))
        return y

    def spmm(self, X, Y, stream=None):
        """Y = A X for X of shape (N, k) and Y of shape (M, k), as DeviceCSR.spmm (spmv_b200_hll_spmm): each column bit
        for bit spmv_hll_serial, i.e. spmv(slice_kernel="rows") on that column.  No accumulate flag."""
        i = self.info()
        k, ldx, ldy = _spmm_operands(X, Y, i.M, i.N)
        if k and i.M:
            N.check(N.lib().spmv_b200_hll_spmm(self._h, k, _ptr(X), ldx, _ptr(Y), ldy, _stream(stream)))
        return Y

    def enable_f32(self, stream=None):
        N.check(N.lib().spmv_b200_hll_enable_f32(self._h, _stream(stream)))
        return self

    def row_form_f32(self) -> str:
        return row_form_name(FORMAT_HLL, N.lib().spmv_b200_hll_row_form_f32(self._h))

    def row_form(self) -> str:
        """Name of the fp64 lane-per-row kernel the plan-time timing chose (spmv_b200_hll_row_form)."""
        return row_form_name(FORMAT_HLL, N.lib().spmv_b200_hll_row_form(self._h), "double")

    def spmv_f32(self, x, y, stream=None):
        i = self.info()
        _check_vec(x, i.N, "x", "float32")
        _check_vec(y, i.M, "y", "float32")
        N.check(N.lib().spmv_b200_hll_spmv_f32(self._h, _ptr(x), _ptr(y), _stream(stream)))
        return y

    def spmm_f32(self, X, Y, stream=None):
        """Y = A X as spmm, on float32 tensors through the float copy of enable_f32: each column bit for bit the
        lane-per-row product in double, rounded once to float, on hacks of any width (spmv_b200_hll_spmm_f32).  No
        accumulate flag; SpmvError without enable_f32."""
        i = self.info()
        k, ldx, ldy = _spmm_operands(X, Y, i.M, i.N, "float32")
        if k and i.M:
            N.check(N.lib().spmv_b200_hll_spmm_f32(self._h, k, _ptr(X), ldx, _ptr(Y), ldy, _stream(stream)))
        return Y

    def spmv_host_f32(self, x, y=None):
        i = self.info()
        x, y = _host_vectors(x, y, i.N, i.M, np.float32)
        N.check(N.lib().spmv_b200_hll_spmv_host_f32(self._h, _ptr(x), _ptr(y)))
        return y

    def spmm_host_f32(self, X, Y=None):
        """spmm_host on float32 buffers (spmv_b200_hll_spmm_host_f32): the bits of spmm_f32 on the same handle."""
        i = self.info()
        Y, k, ldx, px, ldy, py = _host_spmm_operands(X, Y, i.M, i.N, np.float32)
        if k and i.M:
            N.check(N.lib().spmv_b200_hll_spmm_host_f32(self._h, k, C.c_void_p(px), ldx, C.c_void_p(py), ldy))
        return Y

    def algorithmic_bytes_f32(self) -> int:
        i = self.info()
        return 8 * i.slots + 8 * (i.num_hacks + 1) + 4 * i.M + 4 * i.N

    # -- fused iterated product (twins of DeviceCSR.spmv_fused / spmv_fused_mail) -------------------------------
    def partials_count(self) -> int:
        return N.lib().spmv_b200_hll_partials_count(self._h)

    def spmv_fused(self, x_ptr, y_ptr, prev_sumsq=None, partials=None, peers=None, stream=None):
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_hll_spmv_fused(self._h, raw(x_ptr), raw(y_ptr), raw(prev_sumsq) if prev_sumsq is not None else None,
                                                 raw(partials) if partials is not None else None,
                                                 C.byref(peers) if peers is not None else None, _stream(stream)))

    def spmv_fused_mail(self, x_ptr, y_ptr, partials, mail, peers=None, stream=None):
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_hll_spmv_fused_mail(self._h, raw(x_ptr), raw(y_ptr), raw(partials),
                                                      C.byref(peers) if peers is not None else None, C.byref(mail),
                                                      _stream(stream)))

    def flat_partials_count(self) -> int:
        return N.lib().spmv_b200_hll_flat_partials_count(self._h)

    def spmv_fused_flat(self, x_ptr, y_ptr, inv_norm=None, partials=None, peers=None, stream=None):
        def raw(v):
            return C.c_void_p(v) if isinstance(v, int) else _ptr(v)
        N.check(N.lib().spmv_b200_hll_spmv_fused_flat(self._h, raw(x_ptr), raw(y_ptr), raw(inv_norm) if inv_norm is not None else None,
                                                      raw(partials) if partials is not None else None,
                                                      C.byref(peers) if peers is not None else None, _stream(stream)))

    def spmv_hacks(self, hack_begin, hack_end, x, y, stream=None):
        i = self.info()
        _check_vec(x, i.N, "x")
        _check_vec(y, i.M, "y")
        N.check(N.lib().spmv_b200_hll_spmv_hacks(self._h, int(hack_begin), int(hack_end), _ptr(x), _ptr(y), _stream(stream)))
        return y

    def spmv_host(self, x, y=None):
        i = self.info()
        x, y = _host_vectors(x, y, i.N, i.M, np.float64)
        N.check(N.lib().spmv_b200_hll_spmv_host(self._h, _ptr(x), _ptr(y)))
        return y

    def spmv_host_ptr(self, x_ptr: int, y_ptr: int):
        N.check(N.lib().spmv_b200_hll_spmv_host(self._h, C.c_void_p(x_ptr), C.c_void_p(y_ptr)))

    def spmm_host(self, X, Y=None):
        """Y = A X on host buffers, as DeviceCSR.spmm_host (spmv_b200_hll_spmm_host): the bits of spmm on the same
        handle.  No accumulate flag.  Returns Y."""
        i = self.info()
        Y, k, ldx, px, ldy, py = _host_spmm_operands(X, Y, i.M, i.N, np.float64)
        if k and i.M:
            N.check(N.lib().spmv_b200_hll_spmm_host(self._h, k, C.c_void_p(px), ldx, C.c_void_p(py), ldy))
        return Y

    def close(self):
        if self._h:
            N.lib().spmv_b200_hll_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- dense-vector helpers of the iterated product -------------------------------------------------
def synth_vector(x, seed, stream=None):
    N.check(N.lib().spmv_b200_synth_vector(_ptr(x), x.numel(), int(seed), _stream(stream)))
    return x


def vec_fill(v, value, stream=None):
    N.check(N.lib().spmv_b200_vec_fill(_ptr(v), v.numel(), float(value), _stream(stream)))
    return v


def vec_ws_doubles() -> int:
    return N.lib().spmv_b200_vec_ws_doubles()


def vec_sumsq(v, ws, out, n=None, stream=None):
    N.check(N.lib().spmv_b200_vec_sumsq(_ptr(v), int(v.numel() if n is None else n), _ptr(ws), _ptr(out), _stream(stream)))
    return out


def vec_sum(src, n, out, stream=None):
    N.check(N.lib().spmv_b200_vec_sum(_ptr(src), int(n), _ptr(out), _stream(stream)))
    return out


class PeerBuffer:
    """A device buffer other ranks on the NVLink domain can map (cudaIpc)."""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        self.handle = (C.c_char * 64)()
        N.check(N.lib().spmv_b200_ipc_alloc(int(nbytes), C.byref(self.ptr), self.handle))
        self.nbytes = nbytes
        self.mapped = []

    def handle_bytes(self) -> bytes:
        return bytes(self.handle.raw)

    def open_peer(self, handle: bytes) -> int:
        h = (C.c_char * 64).from_buffer_copy(handle)
        p = C.c_void_p()
        N.check(N.lib().spmv_b200_ipc_open(h, C.byref(p)))
        self.mapped.append(p)
        return p.value

    def as_tensor(self, dtype_str="<f8", itemsize=8):
        import torch

        class _View:
            pass
        v = _View()
        v.__cuda_array_interface__ = {"shape": (self.nbytes // itemsize,), "typestr": dtype_str,
                                      "data": (self.ptr.value, False), "version": 2}
        return torch.as_tensor(v, device=torch.device("cuda", torch.cuda.current_device()))

    def close(self):
        for p in self.mapped:
            N.lib().spmv_b200_ipc_close(p)
        self.mapped = []
        if self.ptr:
            N.lib().spmv_b200_ipc_free(self.ptr)
            self.ptr = C.c_void_p()


def vec_push(src, n, peer_ptrs, ctas=0, stream=None):
    """peer_ptrs[p][i] = src[i]: a slice pushed into the other ranks' replicas with NVLink peer stores (spmv_b200_vec_push)."""
    arr = (C.c_void_p * max(len(peer_ptrs), 1))(*[C.c_void_p(int(p)) for p in peer_ptrs])
    N.check(N.lib().spmv_b200_vec_push(_ptr(src), int(n), len(peer_ptrs), arr, int(ctas), _stream(stream)))


def mail_exchange(partials, count, mail, sumsq_out, stream=None):
    """One CTA: fixed-order sum of the flat product's partials, publish into every rank's mailbox, wait for all ranks,
    leave |w|^2 in sumsq_out (spmv_b200_mail_exchange)."""
    N.check(N.lib().spmv_b200_mail_exchange(_ptr(partials), int(count), C.byref(mail), _ptr(sumsq_out), _stream(stream)))


def vec_scale_by_inv_norm(dst, src, sumsq, n=None, stream=None):
    N.check(N.lib().spmv_b200_vec_scale_by_inv_norm(_ptr(dst), _ptr(src), int(src.numel() if n is None else n),
                                                    _ptr(sumsq), _stream(stream)))
    return dst
