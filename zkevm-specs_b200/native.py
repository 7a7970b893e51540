"""ctypes binding of libzkcheck.so (the C-ABI in include/zkcheck.h) and its nvcc build.

The product has NO CPU fallback: if the library cannot be built/loaded, or no CUDA device is
present when a check is requested, these functions raise."""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
from typing import Optional, Sequence

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.environ.get("ZKCHECK_LIB") or os.path.join(PKG_DIR, "libzkcheck.so")  # ZKCHECK_LIB: tuning builds

# ids of include/zkcheck.h
CIRCUIT_BYTECODE, CIRCUIT_STATE, CIRCUIT_COPY, CIRCUIT_EVM, CIRCUIT_EXP, CIRCUIT_TX, CIRCUIT_SIG, CIRCUIT_PI = range(8)
(TABLE_FIXED, TABLE_BYTECODE, TABLE_RW, TABLE_TX, TABLE_BLOCK, TABLE_COPY, TABLE_KECCAK, TABLE_MPT,
 TABLE_PUSH, TABLE_WITHDRAWAL, TABLE_CALLDATA_GAS, TABLE_EXP, TABLE_STEP_AUX) = range(13)
CHALLENGE_KECCAK, CHALLENGE_LOOKUP, CHALLENGE_PI_KECCAK, CHALLENGE_PI_BYTE_BASE, PARAM_PI_CIRCUIT_LEN = range(5)
CIRCUIT_WITHDRAWAL = 8
PARAM_WITHDRAWAL_MAX = 5
FLAG_WRAP, FLAG_EVM_FIRST_STEP, FLAG_EVM_LAST_STEP = 1, 2, 4
ERR_ASSERT, ERR_LOOKUP_UNSAT, ERR_LOOKUP_AMBIGUOUS, ERR_RANGE_RAISE, ERR_VALUE, ERR_NOT_IMPLEMENTED = range(6)
PASS = 0xFFFFFFFF

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _sources():
    out = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))]
    out += [os.path.join(ROOT, "include", f) for f in ("zkcheck.h", "zk_constraints.h")]
    return out


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/api.cu (unity build) for sm_100a into libzkcheck.so, in-tree."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libzkcheck.so (no CPU fallback exists)")
    cmd = [nvcc, *NVCC_FLAGS, "-o", LIB_PATH, os.path.join(CSRC, "api.cu"), "-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stderr)
    return LIB_PATH


_LIB: Optional[ctypes.CDLL] = None
_U64P = ctypes.POINTER(ctypes.c_uint64)
_U32P = ctypes.POINTER(ctypes.c_uint32)
_U8P = ctypes.POINTER(ctypes.c_uint8)

EXPORTS = [
    "zk_ctx_create", "zk_ctx_destroy", "zk_last_error", "zk_set_challenge", "zk_upload_columns",
    "zk_bind_columns_device", "zk_upload_row_flags", "zk_upload_table", "zk_bind_table_device",
    "zk_upload_table_flags", "zk_check", "zk_check_async", "zk_result_device", "zk_fetch_result",
    "zk_allreduce_results", "zk_circuit_cols", "zk_table_cols", "zk_n_constraints",
    "zk_constraint_info", "zk_launch_count", "zk_invalidate_indexes", "zk_enable_timing",
    "zk_last_timing", "zk_upload_columns_packed", "zk_upload_table_packed",
    "zk_upload_bytecode_table_from_code", "zk_nccl_unique_id", "zk_nccl_comm_init", "zk_nccl_comm_destroy",
    "zk_keccak256_batch", "zk_assign_keccak_table", "zk_assign_bytecode_circuit", "zk_assign_state_circuit",
    "zk_assign_copy_circuit", "zk_download_columns", "zk_resident_rows", "zk_assign_withdrawal_circuit",
]


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        if is_stale() and not os.environ.get("ZKCHECK_LIB"):  # a tuning build is used as it is
            build()
        L = ctypes.CDLL(LIB_PATH)
        vp, u64, u32, i32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int
        L.zk_ctx_create.argtypes = [i32, ctypes.POINTER(vp)]
        L.zk_ctx_destroy.argtypes = [vp]
        L.zk_ctx_destroy.restype = None
        L.zk_last_error.argtypes = [vp]
        L.zk_last_error.restype = ctypes.c_char_p
        L.zk_set_challenge.argtypes = [vp, i32, _U64P]
        L.zk_upload_columns.argtypes = [vp, i32, u64, u32, vp, vp]
        L.zk_bind_columns_device.argtypes = [vp, i32, u64, u32, vp]
        L.zk_upload_row_flags.argtypes = [vp, i32, u64, vp, vp]
        L.zk_upload_table.argtypes = [vp, i32, u64, u32, vp, vp]
        L.zk_bind_table_device.argtypes = [vp, i32, u64, u32, vp]
        L.zk_upload_table_flags.argtypes = [vp, i32, u64, vp, vp]
        L.zk_upload_columns_packed.argtypes = [vp, i32, u64, u32, vp, u64, vp, vp, vp]
        L.zk_upload_table_packed.argtypes = [vp, i32, u64, u32, vp, u64, vp, vp, vp]
        L.zk_upload_bytecode_table_from_code.argtypes = [vp, u64, vp, vp, vp, vp, vp]
        L.zk_check.argtypes = [vp, i32, u64, u64, u64, u32, _U32P, _U64P, vp]
        L.zk_check_async.argtypes = [vp, i32, u64, u64, u64, u32, vp]
        L.zk_result_device.argtypes = [vp, i32, ctypes.POINTER(vp), ctypes.POINTER(vp)]
        L.zk_fetch_result.argtypes = [vp, i32, _U32P, _U64P, vp]
        L.zk_allreduce_results.argtypes = [vp, i32, vp, vp]
        L.zk_nccl_unique_id.argtypes = [vp, vp]
        L.zk_nccl_comm_init.argtypes = [vp, i32, i32, vp, ctypes.POINTER(vp)]
        L.zk_nccl_comm_destroy.argtypes = [vp, vp]
        L.zk_keccak256_batch.argtypes = [vp, u64, vp, vp, vp, vp]
        L.zk_assign_keccak_table.argtypes = [vp, u64, vp, vp, vp]
        L.zk_assign_bytecode_circuit.argtypes = [vp, u32, u64, vp, vp, vp, vp, vp]
        L.zk_assign_state_circuit.argtypes = [vp, u64, vp, u64, vp, vp, vp, vp]
        L.zk_assign_copy_circuit.argtypes = [vp, u64, vp, vp, vp, vp]
        L.zk_assign_withdrawal_circuit.argtypes = [vp, u64, vp, u64, vp]
        L.zk_download_columns.argtypes = [vp, i32, vp, vp, vp]
        L.zk_resident_rows.argtypes = [vp, i32]
        L.zk_resident_rows.restype = ctypes.c_int64
        L.zk_circuit_cols.argtypes = [i32]
        L.zk_table_cols.argtypes = [i32]
        L.zk_n_constraints.argtypes = [i32]
        L.zk_constraint_info.argtypes = [i32, i32, ctypes.c_char_p, i32]
        L.zk_launch_count.argtypes = [vp]
        L.zk_launch_count.restype = u64
        L.zk_invalidate_indexes.argtypes = [vp]
        L.zk_enable_timing.argtypes = [vp, i32]
        L.zk_last_timing.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
        _LIB = L
    return _LIB


def constraint_catalogue(circuit_id: int):
    """[(name+doc, error class)] for a circuit, from the library itself."""
    L = lib()
    out = []
    buf = ctypes.create_string_buffer(256)
    for i in range(L.zk_n_constraints(circuit_id)):
        cls = L.zk_constraint_info(circuit_id, i, buf, 256)
        out.append((buf.value.decode(), cls))
    return out


class NativeError(RuntimeError):
    pass


def _host_ptr(a: np.ndarray):
    return ctypes.c_void_p(a.ctypes.data)


class Context:
    """One zk_ctx: owns the device copies of witness matrices, tables and lookup indexes."""

    def __init__(self, device: int = 0) -> None:
        self._L = lib()
        h = ctypes.c_void_p()
        rc = self._L.zk_ctx_create(device, ctypes.byref(h))
        if rc != 0:
            raise NativeError(f"zk_ctx_create failed: {self._L.zk_last_error(None).decode()}")
        self._h = h
        self.device = device
        # None: upload_columns / upload_table ship canonical 32-byte cells.  "min": they pack every
        # matrix to its measured minimal column widths first and ship the packed buffer
        # (zk_upload_*_packed); results are identical (tests/test_gpu_packed.py).
        self.packed_uploads = None

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._L.zk_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def _ck(self, rc: int, what: str) -> None:
        if rc != 0:
            raise NativeError(f"{what}: {self._L.zk_last_error(self._h).decode()} (rc={rc})")

    @staticmethod
    def _matrix(a) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint64)
        assert a.ndim == 3 and a.shape[2] == 4, "matrix must be uint64[n_cols][n_rows][4]"
        return a

    def set_challenge(self, which: int, value: int) -> None:
        limbs = (ctypes.c_uint64 * 4)(*[(int(value) >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)])
        self._ck(self._L.zk_set_challenge(self._h, which, limbs), "zk_set_challenge")

    def upload_columns(self, circuit_id: int, matrix, flags=None, stream: int = 0) -> None:
        m = self._matrix(matrix)
        if self.packed_uploads == "min" and m.shape[1]:
            from . import packing
            self._keep = getattr(self, "_keep", {})
            pm = self._keep[("c", circuit_id)] = packing.pack_matrix(m)  # host buffer outlives the async copy
            return self.upload_columns_packed(circuit_id, pm, flags=flags, stream=stream)
        self._ck(self._L.zk_upload_columns(self._h, circuit_id, m.shape[1], m.shape[0], _host_ptr(m),
                                           ctypes.c_void_p(stream)), "zk_upload_columns")
        if flags is not None:
            f = np.ascontiguousarray(flags, dtype=np.uint8)
            self._ck(self._L.zk_upload_row_flags(self._h, circuit_id, f.shape[0], _host_ptr(f),
                                                 ctypes.c_void_p(stream)), "zk_upload_row_flags")

    def upload_columns_packed(self, circuit_id: int, pm, flags=None, stream: int = 0, host_ptr: int = 0) -> None:
        """pm: packing.PackedMatrix (narrow columns in one host buffer); `host_ptr` overrides the
        buffer address (e.g. a pinned copy of pm.buf)"""
        self._keep = getattr(self, "_keep", {})
        self._keep[("cp", circuit_id)] = pm  # the host buffer outlives the asynchronous copy
        self._ck(self._L.zk_upload_columns_packed(
            self._h, circuit_id, pm.n_rows, pm.n_cols, ctypes.c_void_p(host_ptr or pm.buf.ctypes.data), pm.nbytes,
            _host_ptr(pm.offsets), _host_ptr(pm.widths), ctypes.c_void_p(stream)), "zk_upload_columns_packed")
        if flags is not None:
            f = np.ascontiguousarray(flags, dtype=np.uint8)
            self._ck(self._L.zk_upload_row_flags(self._h, circuit_id, f.shape[0], _host_ptr(f),
                                                 ctypes.c_void_p(stream)), "zk_upload_row_flags")

    def upload_table_packed(self, table_id: int, pm, flags=None, stream: int = 0, host_ptr: int = 0) -> None:
        self._keep = getattr(self, "_keep", {})
        self._keep[("tp", table_id)] = pm
        self._ck(self._L.zk_upload_table_packed(
            self._h, table_id, pm.n_rows, pm.n_cols, ctypes.c_void_p(host_ptr or pm.buf.ctypes.data), pm.nbytes,
            _host_ptr(pm.offsets), _host_ptr(pm.widths), ctypes.c_void_p(stream)), "zk_upload_table_packed")
        if flags is not None:
            f = np.ascontiguousarray(flags, dtype=np.uint8)
            self._ck(self._L.zk_upload_table_flags(self._h, table_id, f.shape[0], _host_ptr(f),
                                                   ctypes.c_void_p(stream)), "zk_upload_table_flags")

    def upload_bytecode_table_from_code(self, code: np.ndarray, is_code_bits: np.ndarray, code_offsets: np.ndarray,
                                        hashes: np.ndarray, stream: int = 0, ptrs=None) -> None:
        """Bytecode.table_assignments on the device (include/zkcheck.h): `code` uint8 (all contracts
        concatenated), `is_code_bits` uint8 bitmap (LSB first), `code_offsets` uint64[n+1], `hashes`
        uint64[n][4] = (lo limb0, lo limb1, hi limb0, hi limb1).  `ptrs` = optional (code, bits) host
        addresses of pinned copies."""
        code = np.ascontiguousarray(code, dtype=np.uint8)
        bits = np.ascontiguousarray(is_code_bits, dtype=np.uint8)
        offs = np.ascontiguousarray(code_offsets, dtype=np.uint64)
        hs = np.ascontiguousarray(hashes, dtype=np.uint64)
        assert hs.shape == (len(offs) - 1, 4) and len(bits) >= (len(code) + 7) // 8 and int(offs[-1]) == len(code)
        self._keep = getattr(self, "_keep", {})
        self._keep["bytecode_src"] = (code, bits, offs, hs)
        pc, pb = ptrs if ptrs else (code.ctypes.data, bits.ctypes.data)
        self._ck(self._L.zk_upload_bytecode_table_from_code(
            self._h, len(offs) - 1, ctypes.c_void_p(pc), ctypes.c_void_p(pb), _host_ptr(offs), _host_ptr(hs),
            ctypes.c_void_p(stream)), "zk_upload_bytecode_table_from_code")

    # ---- witness assignment on the device (include/zkcheck.h "witness assignment") ----------------
    def assign_bytecode_circuit(self, k: int, code: np.ndarray, is_code_bits: np.ndarray, code_offsets: np.ndarray,
                                hashes: np.ndarray, stream: int = 0) -> None:
        """assign_bytecode_circuit (bytecode_circuit.py:104-167) on the device: the 2^k rows of ZK_CIRCUIT_BYTECODE from
        the raw code (same arguments as upload_bytecode_table_from_code), value_rlc under CHALLENGE_KECCAK"""
        code = np.ascontiguousarray(code, dtype=np.uint8)
        bits = np.ascontiguousarray(is_code_bits, dtype=np.uint8)
        offs = np.ascontiguousarray(code_offsets, dtype=np.uint64)
        hs = np.ascontiguousarray(hashes, dtype=np.uint64)
        assert hs.shape == (len(offs) - 1, 4) and len(bits) >= (len(code) + 7) // 8 and int(offs[-1]) == len(code)
        self._ck(self._L.zk_assign_bytecode_circuit(self._h, k, len(offs) - 1, _host_ptr(code),
                                                    _host_ptr(bits), _host_ptr(offs), _host_ptr(hs), ctypes.c_void_p(stream)),
                 "zk_assign_bytecode_circuit")

    def assign_state_circuit(self, ops, flags=None, stream: int = 0) -> None:
        """op2row (state_circuit.py:827-857) on the device: `ops` = a PackedMatrix (or canonical uint64[15][n][4]) of the 15
        operation cells (rw_counter, is_write, tag, id, address, field_tag, storage_key lo/hi, value lo/hi, initial_value
        lo/hi, root lo/hi, selector); the address limbs and key bytes of the 57-cell row are derived on the device"""
        from . import packing
        pm = ops if isinstance(ops, packing.PackedMatrix) else packing.pack_matrix(self._matrix(ops), widths=[32] * 15)
        assert pm.n_cols == 15
        self._keep = getattr(self, "_keep", {})
        self._keep["state_ops"] = pm
        offs = np.ascontiguousarray(pm.offsets, dtype=np.uint64)
        widths = np.ascontiguousarray(pm.widths, dtype=np.uint8)
        fl = None if flags is None else np.ascontiguousarray(flags, dtype=np.uint8)
        self._ck(self._L.zk_assign_state_circuit(self._h, pm.n_rows, _host_ptr(pm.buf), pm.nbytes,
                                                 _host_ptr(offs), _host_ptr(widths), None if fl is None else _host_ptr(fl),
                                                 ctypes.c_void_p(stream)), "zk_assign_state_circuit")

    def assign_copy_circuit(self, events: np.ndarray, data: np.ndarray, is_code_bits=None, stream: int = 0) -> None:
        """CopyCircuit.copy (evm_circuit/typing.py:1010-1147) on the device: `events` uint64[n][16] (include/zkcheck.h), `data`
        the copied byte values of all events (0 where the source is out of bounds), rlc_acc under CHALLENGE_KECCAK"""
        ev = np.ascontiguousarray(events, dtype=np.uint64)
        assert ev.ndim == 2 and ev.shape[1] == 16
        data = np.ascontiguousarray(data, dtype=np.uint8)
        assert int(ev[:, 5].sum()) == len(data)
        bits = None if is_code_bits is None else np.ascontiguousarray(is_code_bits, dtype=np.uint8)
        self._ck(self._L.zk_assign_copy_circuit(self._h, ev.shape[0], _host_ptr(ev), _host_ptr(data),
                                                None if bits is None else _host_ptr(bits), ctypes.c_void_p(stream)),
                 "zk_assign_copy_circuit")

    def assign_withdrawal_circuit(self, records: np.ndarray, max_withdrawals: int, stream: int = 0) -> None:
        """withdrawals2witness on the device (include/zkcheck.h): `records` uint64[n][5][4] = (id, validator_id, address,
        amount, root) as canonical cells.  Writes the MAX-row withdrawal matrix (hash = keccak256 of the RLP encoding,
        padding rows Row(0, 0, 0, 0, Word(0), last root)) and the keccak table, RLC under CHALLENGE_KECCAK"""
        rec = np.ascontiguousarray(records, dtype=np.uint64)
        assert rec.ndim == 3 and rec.shape[1:] == (5, 4)
        self._keep = getattr(self, "_keep", {})
        self._keep["wd_records"] = rec  # the host buffer outlives the asynchronous copy
        self._ck(self._L.zk_assign_withdrawal_circuit(self._h, rec.shape[0], _host_ptr(rec), max_withdrawals,
                                                      ctypes.c_void_p(stream)), "zk_assign_withdrawal_circuit")

    def download_columns(self, circuit_id: int, stream: int = 0):
        """the resident matrix of a circuit as canonical cells + its row flags: (uint64[n_cols][n_rows][4], uint8[n_rows])"""
        n_cols, n_rows = self._L.zk_circuit_cols(circuit_id), self.resident_rows(circuit_id)
        out = np.zeros((n_cols, n_rows, 4), dtype=np.uint64)
        fl = np.zeros(max(n_rows, 1), dtype=np.uint8)
        self._ck(self._L.zk_download_columns(self._h, circuit_id, _host_ptr(out), _host_ptr(fl), ctypes.c_void_p(stream)),
                 "zk_download_columns")
        return out, fl[:n_rows]

    def resident_rows(self, circuit_id: int) -> int:
        return int(self._L.zk_resident_rows(self._h, circuit_id))

    def bind_columns_device(self, circuit_id: int, n_rows: int, n_cols: int, dev_ptr: int) -> None:
        self._ck(self._L.zk_bind_columns_device(self._h, circuit_id, n_rows, n_cols,
                                                ctypes.c_void_p(dev_ptr)), "zk_bind_columns_device")

    def upload_table(self, table_id: int, matrix, flags=None, stream: int = 0) -> None:
        m = self._matrix(matrix)
        if self.packed_uploads == "min" and m.shape[1]:
            from . import packing
            self._keep = getattr(self, "_keep", {})
            pm = self._keep[("t", table_id)] = packing.pack_matrix(m)
            return self.upload_table_packed(table_id, pm, flags=flags, stream=stream)
        self._ck(self._L.zk_upload_table(self._h, table_id, m.shape[1], m.shape[0], _host_ptr(m),
                                         ctypes.c_void_p(stream)), "zk_upload_table")
        if flags is not None:
            f = np.ascontiguousarray(flags, dtype=np.uint8)
            self._ck(self._L.zk_upload_table_flags(self._h, table_id, f.shape[0], _host_ptr(f),
                                                   ctypes.c_void_p(stream)), "zk_upload_table_flags")

    def bind_table_device(self, table_id: int, n_rows: int, n_cols: int, dev_ptr: int) -> None:
        self._ck(self._L.zk_bind_table_device(self._h, table_id, n_rows, n_cols,
                                              ctypes.c_void_p(dev_ptr)), "zk_bind_table_device")

    def n_constraints(self, circuit_id: int) -> int:
        return self._L.zk_n_constraints(circuit_id)

    def check(self, circuit_id: int, row_begin: int, row_end: int, row_base: int = 0,
              flags: int = FLAG_WRAP, stream: int = 0):
        n = self.n_constraints(circuit_id)
        ff = np.empty(n, dtype=np.uint32)
        fc = np.empty(n, dtype=np.uint64)
        self._ck(self._L.zk_check(self._h, circuit_id, row_begin, row_end, row_base, flags,
                                  ff.ctypes.data_as(_U32P), fc.ctypes.data_as(_U64P),
                                  ctypes.c_void_p(stream)), "zk_check")
        return ff, fc

    def check_async(self, circuit_id: int, row_begin: int, row_end: int, row_base: int = 0,
                    flags: int = FLAG_WRAP, stream: int = 0) -> None:
        self._ck(self._L.zk_check_async(self._h, circuit_id, row_begin, row_end, row_base, flags,
                                        ctypes.c_void_p(stream)), "zk_check_async")

    def fetch_result(self, circuit_id: int, stream: int = 0):
        n = self.n_constraints(circuit_id)
        ff = np.empty(n, dtype=np.uint32)
        fc = np.empty(n, dtype=np.uint64)
        self._ck(self._L.zk_fetch_result(self._h, circuit_id, ff.ctypes.data_as(_U32P),
                                         fc.ctypes.data_as(_U64P), ctypes.c_void_p(stream)),
                 "zk_fetch_result")
        return ff, fc

    def result_device_ptrs(self, circuit_id: int):
        a, b = ctypes.c_void_p(), ctypes.c_void_p()
        self._ck(self._L.zk_result_device(self._h, circuit_id, ctypes.byref(a), ctypes.byref(b)),
                 "zk_result_device")
        return a.value, b.value

    def invalidate_indexes(self) -> None:
        self._L.zk_invalidate_indexes(self._h)

    def enable_timing(self, on: bool = True) -> None:
        self._ck(self._L.zk_enable_timing(self._h, int(on)), "zk_enable_timing")

    def last_timing(self):
        """(index build ms, check kernel ms) of the most recent check, device-timed"""
        a, b = ctypes.c_float(), ctypes.c_float()
        self._ck(self._L.zk_last_timing(self._h, ctypes.byref(a), ctypes.byref(b)), "zk_last_timing")
        return a.value, b.value

    def upload_columns_ptr(self, circuit_id: int, n_rows: int, n_cols: int, host_ptr: int, stream: int = 0) -> None:
        self._ck(self._L.zk_upload_columns(self._h, circuit_id, n_rows, n_cols, ctypes.c_void_p(host_ptr),
                                           ctypes.c_void_p(stream)), "zk_upload_columns")

    def upload_table_ptr(self, table_id: int, n_rows: int, n_cols: int, host_ptr: int, stream: int = 0) -> None:
        self._ck(self._L.zk_upload_table(self._h, table_id, n_rows, n_cols, ctypes.c_void_p(host_ptr),
                                         ctypes.c_void_p(stream)), "zk_upload_table")

    def launch_count(self) -> int:
        return int(self._L.zk_launch_count(self._h))

    # ---- Keccak-256 on the device ------------------------------------------------------------
    @staticmethod
    def _concat(messages):
        offs = np.zeros(len(messages) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(m) for m in messages])
        data = np.frombuffer(b"".join(bytes(m) for m in messages) or b"\0", dtype=np.uint8).copy()
        return data, offs

    def keccak256_batch(self, messages, stream: int = 0):
        """digests of a list of byte strings, hashed on the device"""
        data, offs = self._concat(messages)
        out = np.zeros((len(messages), 4), dtype=np.uint64)
        self._ck(self._L.zk_keccak256_batch(self._h, len(messages), _host_ptr(data), _host_ptr(offs), _host_ptr(out),
                                            ctypes.c_void_p(stream)), "zk_keccak256_batch")
        return [out[k].tobytes() for k in range(len(messages))]

    def assign_keccak_table(self, messages, stream: int = 0) -> None:
        """KeccakCircuit.add for every message, on the device: the resident keccak table becomes one row per message"""
        data, offs = self._concat(messages)
        self._keep = getattr(self, "_keep", {})
        self._keep["keccak_src"] = (data, offs)
        self._ck(self._L.zk_assign_keccak_table(self._h, len(messages), _host_ptr(data), _host_ptr(offs),
                                                ctypes.c_void_p(stream)), "zk_assign_keccak_table")

    # ---- multi-GPU: one NCCL communicator per context, results folded in place --------------
    def nccl_unique_id(self) -> bytes:
        """rank 0 draws the 128-byte NCCL id; ship it to the other ranks (gloo, MPI, a file, ...)"""
        buf = (ctypes.c_uint8 * 128)()
        self._ck(self._L.zk_nccl_unique_id(self._h, buf), "zk_nccl_unique_id")
        return bytes(buf)

    def nccl_init(self, world: int, rank: int, unique_id: bytes) -> None:
        buf = (ctypes.c_uint8 * 128).from_buffer_copy(unique_id)
        comm = ctypes.c_void_p()
        self._ck(self._L.zk_nccl_comm_init(self._h, world, rank, buf, ctypes.byref(comm)), "zk_nccl_comm_init")
        self._comm = comm

    def allreduce_results(self, circuit_id: int, stream: int = 0) -> None:
        """MIN of first_fail / SUM of fail_count over the communicator's ranks, in place on the device"""
        self._ck(self._L.zk_allreduce_results(self._h, circuit_id, self._comm, ctypes.c_void_p(stream)),
                 "zk_allreduce_results")

    def nccl_destroy(self) -> None:
        if getattr(self, "_comm", None):
            self._L.zk_nccl_comm_destroy(self._h, self._comm)
            self._comm = None


_DEFAULT: dict = {}


def default_context(device: int = 0) -> Context:
    if device not in _DEFAULT:
        _DEFAULT[device] = Context(device)
    return _DEFAULT[device]


def first_failure(first_fail: np.ndarray, circuit_id: int):
    """(row, constraint id, error class) of the failure the reference would hit first:
    smallest row, then smallest id (ids follow the reference's program order)."""
    bad = np.nonzero(first_fail != PASS)[0]
    if len(bad) == 0:
        return None
    rows = first_fail[bad].astype(np.int64)
    k = int(bad[np.argmin(rows)])  # argmin returns the first (smallest id) among equal rows
    cat = constraint_catalogue(circuit_id)
    return int(first_fail[k]), k, cat[k][1], cat[k][0]
