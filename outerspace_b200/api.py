"""Host-side mirror of the reference's interface for the functional SpGEMM path, over the C ABI.

Names follow the reference (simulator/SimSpGEMM.cpp, SimOuterSPACE.cpp) so that tests read like
tests of the reference would:

    coo, NRow, NCol = readcoo(path, sym=False)            # SimSpGEMM.cpp:55-100
    csc = coo2csr(coo, NCol, transpose=True)              # SimSpGEMM.cpp:102-152 (throws 233 -> DuplicateEntry)
    csr = coo2csr(coo2, NRow2)
    provider = TaskProvider(csc, csr)                     # SimOuterSPACE.cpp:44-144, runs on the GPU
    provider.mergedResult                                 # CSRMatrix, rows = max row id + 1

Everything that computes goes through ``libosp_b200.so`` (hand-written sm_100a CUDA).  There is no
CPU fallback: without the built library ``load_library`` raises, without a GPU ``Engine`` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from typing import Optional, Tuple

import numpy as np

from .formats import COO, CSRMatrix, ELEM

_LIB_PATH = os.environ.get("OSP_LIB_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libosp_b200.so")   # (OSP_LIB_PATH: development builds)

OSP_OK = 0
OSP_ERR_INVALID, OSP_ERR_CUDA, OSP_ERR_OOM, OSP_ERR_INDEX, OSP_ERR_IO, OSP_ERR_UNSUPPORTED, OSP_ERR_NO_DEVICE = range(1, 8)
OSP_ERR_DUPLICATE = 233

OSP_A_IS_CSR = 1
OSP_DEVICE_POINTERS = 2
OSP_ROWWISE_ORDER = 4
OSP_KSLICE_ORDER = 32
OSP_NO_FUSED_DENSE = 64
OSP_LONGROW_SWEEP = 128     # opt-in: verified on a B200, not faster (include/osp_b200.h)
OSP_FUSED_SHORT = 256       # opt-in: verified on a B200, slower (include/osp_b200.h)
OSP_NO_VALIDATE = 512       # the caller vouches for sorted, duplicate-free slices and in-range column ids
OSP_KWAY_MERGE = 1024       # k-way merge of the pre-sorted ways for rows of 4097..32768 partial products in <= 64 ways
OSP_PROFILE_PHASES = 8
OSP_PROFILE_KERNELS = 16

# every symbol include/osp_b200.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "osp_device_count", "osp_create", "osp_destroy", "osp_last_error", "osp_set_workspace_limit", "osp_set_result_limit", "osp_stream",
    "osp_spgemm", "osp_result_dims", "osp_result_copy", "osp_result_copy_rows", "osp_result_device", "osp_result_stats", "osp_result_kernels", "osp_result_free",
    "osp_task_sizes", "osp_csr2csc", "osp_readcoo", "osp_readcoo_buffer", "osp_coo_dims", "osp_coo_copy", "osp_coo_free", "osp_coo2csr",
    "osp_coo2csr_device", "osp_bias_relu", "osp_csr2compact", "osp_csc2rawcompact",
    "osp_readcoo_device", "osp_readcoo_buffer_device", "osp_coo_device", "osp_coo2csr_result",
    "osp_version", "osp_dist_unique_id", "osp_dist_create", "osp_dist_destroy", "osp_dist_rows", "osp_dist_spgemm",
]


class OspError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"osp error {code}: {message}")
        self.code = code


class DuplicateEntry(OspError):
    """The reference throws the int 233 from dupcheck (SimSpGEMM.cpp:43-53)."""


class SpgemmArgs(C.Structure):
    _fields_ = [
        ("a_slices", C.c_uint64), ("a_pos", C.c_void_p), ("a_data", C.c_void_p),
        ("n_k", C.c_uint64), ("b_pos", C.c_void_p), ("b_data", C.c_void_p),
        ("rows_c", C.c_uint64), ("cols_b", C.c_uint64), ("flags", C.c_uint32), ("reserved", C.c_uint32),
        ("a_nnz", C.c_uint64), ("b_nnz", C.c_uint64),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("rows_c", C.c_uint64), ("cols_b", C.c_uint64), ("n_k", C.c_uint64),
        ("nnz_a", C.c_uint64), ("nnz_b", C.c_uint64), ("nnz_c", C.c_uint64),
        ("products", C.c_uint64), ("algorithmic_bytes", C.c_uint64),
        ("merge_tiles", C.c_uint64), ("rows_medium", C.c_uint64), ("rows_long", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("row_chunks", C.c_uint64),
        ("ms_total", C.c_float), ("ms_convert", C.c_float), ("ms_multiply", C.c_float), ("ms_merge", C.c_float),
        ("ms_h2d", C.c_float), ("ms_d2h", C.c_float), ("ms_exchange", C.c_float), ("reserved_f", C.c_float),
        ("exchange_bytes_out", C.c_uint64),
    ]

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load_library() -> C.CDLL:
    """Loads the in-tree CUDA library; raises if it was not built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C outerspace_b200/csrc). This engine has no CPU fallback."
        )
    if "OSP_NCCL_LIB" not in os.environ:
        # multi-GPU path: use the NCCL build torch ships (found without importing torch)
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (spec.submodule_search_locations if spec and spec.submodule_search_locations else []):
            cand = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["OSP_NCCL_LIB"] = cand
                break
    lib = C.CDLL(_LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    lib.osp_version.restype = C.c_char_p
    lib.osp_device_count.restype = i32
    lib.osp_create.argtypes = [i32, C.POINTER(vp)]
    lib.osp_destroy.argtypes = [vp]
    lib.osp_destroy.restype = None
    lib.osp_last_error.argtypes = [vp]
    lib.osp_last_error.restype = C.c_char_p
    lib.osp_set_workspace_limit.argtypes = [vp, u64]
    lib.osp_set_result_limit.argtypes = [vp, u64]
    lib.osp_stream.argtypes = [vp]
    lib.osp_stream.restype = vp
    lib.osp_spgemm.argtypes = [vp, C.POINTER(SpgemmArgs), C.POINTER(vp)]
    lib.osp_result_dims.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    lib.osp_result_copy.argtypes = [vp, vp, vp]
    lib.osp_result_copy_rows.argtypes = [vp, u64, u64, vp, vp, u64]
    lib.osp_result_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.osp_result_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.osp_result_kernels.argtypes = [vp, C.POINTER(u64), vp, vp]
    lib.osp_result_free.argtypes = [vp]
    lib.osp_result_free.restype = None
    lib.osp_task_sizes.argtypes = [vp, C.POINTER(SpgemmArgs), vp, C.POINTER(u64), vp, C.POINTER(u64), vp]
    lib.osp_csr2csc.argtypes = [vp, u64, u64, vp, vp, u32, vp, vp]
    lib.osp_readcoo.argtypes = [C.c_char_p, i32, C.POINTER(vp)]
    lib.osp_readcoo_device.argtypes = [vp, C.c_char_p, i32, C.POINTER(vp)]
    lib.osp_readcoo_buffer_device.argtypes = [vp, C.c_char_p, u64, i32, C.POINTER(vp)]
    lib.osp_coo_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.osp_coo2csr_result.argtypes = [vp, vp, u64, i32, C.POINTER(vp)]
    lib.osp_coo_dims.argtypes = [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
    lib.osp_coo_copy.argtypes = [vp, vp, vp, vp]
    lib.osp_coo_free.argtypes = [vp]
    lib.osp_coo_free.restype = None
    lib.osp_coo2csr.argtypes = [u64, vp, vp, vp, u64, i32, vp, vp]
    lib.osp_coo2csr_device.argtypes = [vp, u64, vp, vp, vp, u64, u64, i32, u32, vp, vp]
    lib.osp_csr2compact.argtypes = [u64, vp, vp, C.POINTER(u64), vp, vp, vp, vp]
    lib.osp_csc2rawcompact.argtypes = [u64, vp, vp, vp, vp, vp]
    lib.osp_bias_relu.argtypes = [vp, vp, u64, vp, u32, C.POINTER(vp)]
    lib.osp_dist_unique_id.argtypes = [vp]
    lib.osp_dist_create.argtypes = [vp, vp, i32, i32, C.POINTER(vp)]
    lib.osp_dist_destroy.argtypes = [vp]
    lib.osp_dist_destroy.restype = None
    lib.osp_dist_rows.argtypes = [vp, u64, C.POINTER(u64), C.POINTER(u64)]
    lib.osp_dist_spgemm.argtypes = [vp, C.POINTER(SpgemmArgs), C.POINTER(vp)]
    _lib = lib
    return lib


def _ptr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None or a.size == 0 else a.ctypes.data


# ---------------------------------------------------------------------------------------------
# host loaders (reference surface)
# ---------------------------------------------------------------------------------------------
def readcoo(path: str, sym: bool = False) -> Tuple[COO, int, int]:
    lib = load_library()
    h = C.c_void_p()
    rc = lib.osp_readcoo(os.fsencode(path), int(sym), C.byref(h))
    if rc != OSP_OK:
        raise OspError(rc, f"readcoo({path!r}) failed")
    try:
        nrow, ncol, nnz = C.c_uint64(), C.c_uint64(), C.c_uint64()
        lib.osp_coo_dims(h, C.byref(nrow), C.byref(ncol), C.byref(nnz))
        n = nnz.value
        coo = COO(np.empty(n, np.uint32), np.empty(n, np.uint32), np.empty(n, np.float32))
        lib.osp_coo_copy(h, _ptr(coo.rows), _ptr(coo.cols), _ptr(coo.vals))
    finally:
        lib.osp_coo_free(h)
    return coo, nrow.value, ncol.value


def coo2csr(coo: COO, N: int, transpose: bool = False) -> CSRMatrix:
    lib = load_library()
    n = len(coo)
    out = CSRMatrix(np.zeros(N + 1, np.uint64), np.empty(n, ELEM))
    rows = np.ascontiguousarray(coo.rows, np.uint32)
    cols = np.ascontiguousarray(coo.cols, np.uint32)
    vals = np.ascontiguousarray(coo.vals, np.float32)
    rc = lib.osp_coo2csr(n, _ptr(rows), _ptr(cols), _ptr(vals), N, int(transpose), out.pos.ctypes.data, _ptr(out.data))
    if rc == OSP_ERR_DUPLICATE:
        raise DuplicateEntry(rc, "duplicate (row, col) entry")
    if rc != OSP_OK:
        raise OspError(rc, "coo2csr failed")
    return out


def csr2compact(m: CSRMatrix) -> Tuple[np.ndarray, COO]:
    """csr2compact (SimSpGEMM.cpp:154-219): (group_pos, triplets) -- group j = the (j+1)-th non-zero of every slice."""
    lib = load_library()
    n = C.c_uint64()
    rc = lib.osp_csr2compact(m.NRow(), m.pos.ctypes.data, _ptr(m.data), C.byref(n), None, None, None, None)
    if rc != OSP_OK:
        raise OspError(rc, "csr2compact failed")
    gpos = np.zeros(n.value + 1, np.uint64)
    rows, cols, vals = np.empty(m.nnz, np.uint32), np.empty(m.nnz, np.uint32), np.empty(m.nnz, np.float32)
    rc = lib.osp_csr2compact(m.NRow(), m.pos.ctypes.data, _ptr(m.data), C.byref(n), gpos.ctypes.data, _ptr(rows), _ptr(cols), _ptr(vals))
    if rc != OSP_OK:
        raise OspError(rc, "csr2compact failed")
    return gpos, COO(rows, cols, vals)


def csc2rawcompact(m: CSRMatrix) -> Tuple[np.ndarray, COO]:
    """csc2rawcompact (SimSpGEMM.cpp:221-243): (group_pos = pos, triplets with row = idx, col = slice id)."""
    lib = load_library()
    rows, cols, vals = np.empty(m.nnz, np.uint32), np.empty(m.nnz, np.uint32), np.empty(m.nnz, np.float32)
    rc = lib.osp_csc2rawcompact(m.NRow(), m.pos.ctypes.data, _ptr(m.data), _ptr(rows), _ptr(cols), _ptr(vals))
    if rc != OSP_OK:
        raise OspError(rc, "csc2rawcompact failed")
    return m.pos.copy(), COO(rows, cols, vals)


# ---------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------
class Result:
    """C = A*B resident in HBM."""

    def __init__(self, engine: "Engine", handle: C.c_void_p):
        self._engine = engine
        self._h = handle
        engine._results.add(self)              # a result must not outlive its context (Engine.close frees what is left)
        rows, nnz = C.c_uint64(), C.c_uint64()
        engine._lib.osp_result_dims(handle, C.byref(rows), C.byref(nnz))
        self.rows, self.nnz = rows.value, nnz.value

    def stats(self) -> dict:
        s = Stats()
        self._engine._lib.osp_result_stats(self._h, C.byref(s))
        return s.as_dict()

    def kernel_times(self) -> list:
        """[(kernel name, ms)] in launch order for a call made with OSP_PROFILE_KERNELS."""
        n = C.c_uint64()
        self._engine._lib.osp_result_kernels(self._h, C.byref(n), None, None)
        names, ms = (C.c_char_p * n.value)(), (C.c_float * n.value)()
        self._engine._lib.osp_result_kernels(self._h, C.byref(n), names, ms)
        return [(names[i].decode(), float(ms[i])) for i in range(n.value)]

    def device_pointers(self) -> Tuple[int, int]:
        p, d = C.c_void_p(), C.c_void_p()
        self._engine._lib.osp_result_device(self._h, C.byref(p), C.byref(d))
        return p.value or 0, d.value or 0

    def copy_into(self, pos: np.ndarray, data: np.ndarray) -> None:
        self._engine._check(self._engine._lib.osp_result_copy(self._h, pos.ctypes.data, _ptr(data)))

    def to_host(self) -> CSRMatrix:
        out = CSRMatrix(np.empty(self.rows + 1, np.uint64), np.empty(self.nnz, ELEM))
        self.copy_into(out.pos, out.data)
        return out

    def pos_to_host(self) -> np.ndarray:
        """C.pos alone (row pointer, rows + 1 offsets)."""
        pos = np.empty(self.rows + 1, np.uint64)
        self._engine._check(self._engine._lib.osp_result_copy_rows(self._h, 0, self.rows, pos.ctypes.data, None, 0))
        return pos

    def rows_to_host(self, row_begin: int, row_end: int) -> CSRMatrix:
        """Rows [row_begin, row_end) of C as a CSRMatrix of their own (pos rebased to 0)."""
        pos = np.empty(row_end - row_begin + 1, np.uint64)
        lib = self._engine._lib
        self._engine._check(lib.osp_result_copy_rows(self._h, row_begin, row_end, pos.ctypes.data, None, 0))
        data = np.empty(int(pos[-1] - pos[0]), ELEM)
        self._engine._check(lib.osp_result_copy_rows(self._h, row_begin, row_end, pos.ctypes.data, _ptr(data), len(data)))
        return CSRMatrix(pos - pos[0], data)

    def free(self) -> None:
        if self._h is not None:
            self._engine._lib.osp_result_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceCOO:
    """Triplets of a .mtx file resident in HBM (osp_readcoo_device): readcoo's entries, parsed on the GPU."""

    def __init__(self, engine: "Engine", handle: C.c_void_p):
        self._engine = engine
        self._h = handle
        engine._results.add(self)              # must not outlive its context, like a Result
        nrow, ncol, nnz = C.c_uint64(), C.c_uint64(), C.c_uint64()
        engine._lib.osp_coo_dims(handle, C.byref(nrow), C.byref(ncol), C.byref(nnz))
        self.nrow, self.ncol, self.nnz = nrow.value, ncol.value, nnz.value

    def device_pointers(self) -> Tuple[int, int, int]:
        """(rows, cols, vals): uint32, uint32 and float32 arrays of nnz entries in HBM."""
        r, c, v = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._engine._check(self._engine._lib.osp_coo_device(self._h, C.byref(r), C.byref(c), C.byref(v)))
        return r.value or 0, c.value or 0, v.value or 0

    def to_host(self) -> COO:
        coo = COO(np.empty(self.nnz, np.uint32), np.empty(self.nnz, np.uint32), np.empty(self.nnz, np.float32))
        self._engine._check(self._engine._lib.osp_coo_copy(self._h, _ptr(coo.rows), _ptr(coo.cols), _ptr(coo.vals)))
        return coo

    def to_csr(self, N: int, transpose: bool = False) -> Result:
        """coo2csr<transpose>(N) + dupcheck on the GPU into a device CSR (raises DuplicateEntry, OspError(OSP_ERR_INDEX))."""
        h = C.c_void_p()
        self._engine._check(self._engine._lib.osp_coo2csr_result(self._engine._h, self._h, N, int(transpose), C.byref(h)))
        return Result(self._engine, h)

    def free(self) -> None:
        if self._h is not None:
            self._engine._lib.osp_coo_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """One GPU's SpGEMM context (osp_ctx)."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.osp_create(device, C.byref(h))
        if rc != OSP_OK:
            raise OspError(rc, (self._lib.osp_last_error(None) or b"").decode())
        self._h = h
        self.device = device
        self._results = weakref.WeakSet()

    def close(self) -> None:
        if self._h is not None:
            for r in list(self._results):
                r.free()
            self._lib.osp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc == OSP_OK:
            return
        msg = (self._lib.osp_last_error(self._h) or b"").decode()
        raise (DuplicateEntry if rc == OSP_ERR_DUPLICATE else OspError)(rc, msg)

    def set_workspace_limit(self, nbytes: int) -> None:
        self._check(self._lib.osp_set_workspace_limit(self._h, nbytes))

    def set_result_limit(self, nbytes: int) -> None:
        """Cap on the up-front allocation of C's data (0 = automatic): see osp_set_result_limit."""
        self._check(self._lib.osp_set_result_limit(self._h, nbytes))

    @property
    def stream(self) -> int:
        return self._lib.osp_stream(self._h) or 0

    def _args(self, a_slices, a_pos, a_data, n_k, b_pos, b_data, rows_c, cols_b, flags) -> SpgemmArgs:
        return SpgemmArgs(a_slices, a_pos, a_data, n_k, b_pos, b_data, rows_c, cols_b, flags, 0, 0, 0)

    def spgemm(self, a: CSRMatrix, b: CSRMatrix, a_is_csr: bool = False, rows_c: int = 0, cols_b: int = 0,
               flags: int = 0) -> Result:
        """C = A*B with host operands laid out as the reference's CSRMatrix (A as CSC unless a_is_csr)."""
        f = flags | (OSP_A_IS_CSR if a_is_csr else 0)
        self._last_args = self._args(a.NRow(), a.pos.ctypes.data, _ptr(a.data), b.NRow(), b.pos.ctypes.data,
                                     _ptr(b.data), rows_c, cols_b, f)
        self._keepalive = (a, b)
        h = C.c_void_p()
        self._check(self._lib.osp_spgemm(self._h, C.byref(self._last_args), C.byref(h)))
        return Result(self, h)

    def spgemm_device(self, a_slices: int, a_pos_ptr: int, a_data_ptr: int, n_k: int, b_pos_ptr: int, b_data_ptr: int,
                      a_is_csr: bool = False, rows_c: int = 0, cols_b: int = 0, flags: int = 0, a_nnz: int = 0,
                      b_nnz: int = 0) -> Result:
        """Same, with operands already resident in HBM (raw device pointers)."""
        f = flags | OSP_DEVICE_POINTERS | (OSP_A_IS_CSR if a_is_csr else 0)
        self._last_args = self._args(a_slices, a_pos_ptr, a_data_ptr, n_k, b_pos_ptr, b_data_ptr, rows_c, cols_b, f)
        self._last_args.a_nnz, self._last_args.b_nnz = a_nnz, b_nnz
        h = C.c_void_p()
        self._check(self._lib.osp_spgemm(self._h, C.byref(self._last_args), C.byref(h)))
        return Result(self, h)

    def task_sizes(self, result: Result) -> Tuple[np.ndarray, np.ndarray]:
        """(multiply tasks [n,2] = (nnzc, nnzr) per non-empty k, merge tasks [rows,2] = (#ways, output nnz))
        for the operands of the last spgemm call -- what getMultiplyTasks/getMergeTasks expose."""
        nm, ng = C.c_uint64(), C.c_uint64()
        self._check(self._lib.osp_task_sizes(self._h, C.byref(self._last_args), result._h, C.byref(nm), None, C.byref(ng), None))
        mult = np.zeros((nm.value, 2), np.uint32)
        merge = np.zeros((ng.value, 2), np.uint32)
        self._check(self._lib.osp_task_sizes(self._h, C.byref(self._last_args), result._h, C.byref(nm), _ptr(mult) or 0,
                                             C.byref(ng), _ptr(merge) or 0))
        return mult, merge

    def csr2csc(self, m: CSRMatrix, n_minor: int) -> CSRMatrix:
        """Device CSR->CSC (or CSC->CSR) of one operand, stable: coo2csr<true> on the GPU."""
        out = CSRMatrix(np.empty(n_minor + 1, np.uint64), np.empty(m.nnz, ELEM))
        self._check(self._lib.osp_csr2csc(self._h, m.NRow(), n_minor, m.pos.ctypes.data, _ptr(m.data), 0,
                                          out.pos.ctypes.data, _ptr(out.data)))
        return out

    def bias_relu(self, c: "Result", cols: int, bias: Optional[np.ndarray] = None) -> "Result":
        """relu(C + bias) kept sparse, on the device: the step between two layers (NN_models/models.py:18-31)."""
        b = None if bias is None else np.ascontiguousarray(bias, np.float32)
        if b is not None and b.size != cols:
            raise ValueError("bias must hold one value per column")
        h = C.c_void_p()
        self._check(self._lib.osp_bias_relu(self._h, c._h, cols, None if b is None else b.ctypes.data, 0, C.byref(h)))
        return Result(self, h)

    def coo2csr(self, coo: "COO", N: int, transpose: bool = False, n_other: int = 0) -> CSRMatrix:
        """coo2csr<transpose> + dupcheck on the GPU (SimSpGEMM.cpp:43-53,102-152); raises DuplicateEntry (233)."""
        n = len(coo)
        out = CSRMatrix(np.zeros(N + 1, np.uint64), np.empty(n, ELEM))
        rows = np.ascontiguousarray(coo.rows, np.uint32)
        cols = np.ascontiguousarray(coo.cols, np.uint32)
        vals = np.ascontiguousarray(coo.vals, np.float32)
        self._check(self._lib.osp_coo2csr_device(self._h, n, _ptr(rows), _ptr(cols), _ptr(vals), N, n_other, int(transpose), 0,
                                                 out.pos.ctypes.data, _ptr(out.data)))
        return out

    def readcoo_device(self, path: str, sym: bool = False) -> DeviceCOO:
        """readcoo(path, sym) with the text parsed on the GPU; the triplets stay in HBM."""
        h = C.c_void_p()
        self._check(self._lib.osp_readcoo_device(self._h, os.fsencode(path), int(sym), C.byref(h)))
        return DeviceCOO(self, h)

    def readcoo_buffer_device(self, text: bytes, sym: bool = False) -> DeviceCOO:
        """The same for Matrix Market text in memory."""
        h = C.c_void_p()
        self._check(self._lib.osp_readcoo_buffer_device(self._h, bytes(text), len(text), int(sym), C.byref(h)))
        return DeviceCOO(self, h)

    def csr2csc_device(self, n_major: int, n_minor: int, pos_ptr: int, data_ptr: int, pos_out_ptr: int,
                       data_out_ptr: int) -> None:
        self._check(self._lib.osp_csr2csc(self._h, n_major, n_minor, pos_ptr, data_ptr, OSP_DEVICE_POINTERS,
                                          pos_out_ptr, data_out_ptr))

    def coo2csr_device(self, nnz: int, rows_ptr: int, cols_ptr: int, vals_ptr: int, N: int, n_other: int,
                       pos_out_ptr: int, data_out_ptr: int, transpose: bool = False) -> None:
        """coo2csr with the triplet arrays and the outputs resident in HBM (raw device pointers); n_other is required."""
        self._check(self._lib.osp_coo2csr_device(self._h, nnz, rows_ptr, cols_ptr, vals_ptr, N, n_other, int(transpose),
                                                 OSP_DEVICE_POINTERS, pos_out_ptr, data_out_ptr))


_default_engine: Optional[Engine] = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(0)
    return _default_engine


class TaskProvider:
    """Mirror of the reference's TaskProvider (SimOuterSPACE.cpp:44-144): constructing it runs the
    multiply and merge phases (here: on the GPU) for lmatCSC x rmatCSR.

    Differences from the as-written reference, which is buggy (SURVEY.md 8a rows a11/a12): the result
    carries true column ids and sums duplicates (the semantics of cscMulcsr + deduplicateCOO), and
    ``mergedResult`` is readable.  A k-dimension mismatch raises instead of asserting (:47).
    """

    def __init__(self, lmatCSC: CSRMatrix, rmatCSR: CSRMatrix, engine: Optional[Engine] = None):
        self._engine = engine or default_engine()
        res = self._engine.spgemm(lmatCSC, rmatCSR, a_is_csr=False)
        try:
            self.mergedResult = res.to_host()
            self.stats = res.stats()
            self._mult, self._merge = self._engine.task_sizes(res)
        finally:
            res.free()

    def getMultiplyTasks(self) -> np.ndarray:
        """[n_tasks, 2] = (lmatCol.size, rmatRow.size) per non-empty k (MultiplyTask, :34-37)."""
        return self._mult

    def getMergeTasks(self) -> np.ndarray:
        """[rows, 2] = (inputs.size(), output.size) per output row (MergeTask, :39-42)."""
        return self._merge
