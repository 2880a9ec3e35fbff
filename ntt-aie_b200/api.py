"""ctypes binding of include/nttb200.h.  Device buffers are passed as raw pointers
(``tensor.data_ptr()`` of int32 CUDA tensors, or any integer address); torch is used
by callers for memory and streams only -- nothing here imports it."""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "lib", "libnttb200.so")

ORDER_GOLDEN = 0
ORDER_AIE_DEVICE = 1
FORCE_GENERIC = 2
REDUCE_INPUT = 4
INPUT_BITREV = 8
OUTPUT_BITREV = 16
GEN_POWERS = 0
GEN_BITREV = 1
RNS_ADD = 0
RNS_SUB = 1
RNS_MUL = 2
RNS_ROUND = 1
AUTO_COEFF = 0
AUTO_EVAL = 1
PACK_SCALED = 0
PACK_CENTRED = 1
KS_COEFF_IN = 1
KS_COEFF_OUT = 2

_lib = None
_i32p = ctypes.POINTER(ctypes.c_int32)


class NttError(RuntimeError):
    def __init__(self, status: int, where: str):
        lib = load_library()
        msg = lib.nttb200_strerror(status).decode()
        detail = lib.nttb200_last_error().decode()
        super().__init__(f"{where}: {msg}" + (f" [{detail}]" if detail else ""))
        self.status = status


def lib_path() -> str:
    return _LIB_PATH


def load_library():
    """Load libnttb200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"{_LIB_PATH} is missing: build it with `python ntt-aie_b200/build.py` "
            "(there is no CPU fallback)")
    lib = ctypes.CDLL(_LIB_PATH)
    vp, sz, i32, u32, i64 = (ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int32, ctypes.c_uint32,
                             ctypes.c_int64)
    sig = {
        "nttb200_make_roots": (ctypes.c_int, [i32, _i32p, i32, i32]),
        "nttb200_make_bitrev_table": (ctypes.c_int, [i32, _i32p, i32, i32]),
        "nttb200_powmod": (i32, [i32, i64, i32]),
        "nttb200_plan_create": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, u32, u32, _i32p,
                                               u32]),
        "nttb200_plan_destroy": (ctypes.c_int, [vp]),
        "nttb200_plan_create_generated": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, u32, u32, u32,
                                                         u32, u32, u32, u32]),
        "nttb200_plan_table": (ctypes.c_int, [vp, _i32p]),
        "nttb200_reduce": (ctypes.c_int, [vp, vp, vp, sz, vp]),
        "nttb200_bitrev_permute": (ctypes.c_int, [vp, vp, vp, sz, vp]),
        "nttb200_transpose": (ctypes.c_int, [vp, vp, vp, sz, ctypes.c_int, vp]),
        "nttb200_gs_batch": (ctypes.c_int, [vp, vp, vp, sz, ctypes.c_int, vp]),
        "nttb200_ct_batch": (ctypes.c_int, [vp, vp, vp, sz, ctypes.c_int, vp]),
        "nttb200_gs_stage_range": (ctypes.c_int, [vp, vp, vp, sz, ctypes.c_int, ctypes.c_int, vp]),
        "nttb200_gs_host": (ctypes.c_int, [vp, vp, vp, sz, ctypes.c_int]),
        "nttb200_gs_stage_range_scatter": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int,
                                                          ctypes.POINTER(vp), ctypes.c_int,
                                                          ctypes.c_int, vp]),
        "nttb200_host_alloc": (ctypes.c_int, [ctypes.POINTER(vp), sz, ctypes.c_int]),
        "nttb200_host_free": (ctypes.c_int, [vp]),
        "nttb200_pointwise": (ctypes.c_int, [vp, vp, vp, vp, sz, vp]),
        "nttb200_scale": (ctypes.c_int, [vp, vp, vp, sz, i32, vp]),
        "nttb200_polymul_negacyclic": (ctypes.c_int, [vp, vp, vp, vp, vp, sz, vp]),
        "nttb200_rns_plan_create": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, u32,
                                                   ctypes.POINTER(u32), ctypes.POINTER(_i32p), u32]),
        "nttb200_rns_plan_create_logn": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, u32, u32,
                                                        ctypes.POINTER(u32), ctypes.POINTER(_i32p), u32]),
        "nttb200_rns_plan_create_generated": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, u32, u32,
                                                             ctypes.POINTER(u32), u32, ctypes.POINTER(u32),
                                                             u32]),
        "nttb200_rns_plan_destroy": (ctypes.c_int, [vp]),
        "nttb200_rns_gs_batch": (ctypes.c_int, [vp, vp, vp, sz, vp]),
        "nttb200_rns_ct_batch": (ctypes.c_int, [vp, vp, vp, sz, vp]),
        "nttb200_rns_polymul_negacyclic": (ctypes.c_int, [vp, vp, vp, vp, vp, sz, vp]),
        "nttb200_rns_pointwise": (ctypes.c_int, [vp, u32, vp, vp, vp, sz, sz, vp]),
        "nttb200_rns_scale": (ctypes.c_int, [vp, vp, vp, sz, ctypes.POINTER(u32), vp]),
        "nttb200_rns_dot": (ctypes.c_int, [vp, vp, vp, vp, u32, sz, sz, ctypes.c_int, vp]),
        "nttb200_rns_gs_scaled_batch": (ctypes.c_int, [vp, vp, vp, sz, vp]),
        "nttb200_rns_automorphism": (ctypes.c_int, [vp, vp, vp, sz, ctypes.POINTER(u32), u32, u32, vp]),
        "nttb200_rns_conv_create": (ctypes.c_int, [ctypes.POINTER(vp), vp, vp, u32]),
        "nttb200_rns_conv_destroy": (ctypes.c_int, [vp]),
        "nttb200_rns_base_convert": (ctypes.c_int, [vp, vp, sz, vp, sz, sz, vp]),
        "nttb200_rns_mod_down": (ctypes.c_int, [vp, vp, vp, sz, u32, vp]),
        "nttb200_rns_base_convert_exact": (ctypes.c_int, [vp, vp, sz, vp, sz, sz, vp]),
        "nttb200_rns_scale_round": (ctypes.c_int, [vp, vp, vp, sz, u32, vp]),
        "nttb200_ckks_encoder_create": (ctypes.c_int, [ctypes.POINTER(vp), vp, u32]),
        "nttb200_ckks_encoder_destroy": (ctypes.c_int, [vp]),
        "nttb200_ckks_encode": (ctypes.c_int, [vp, vp, ctypes.c_double, vp, sz, vp]),
        "nttb200_ckks_decode": (ctypes.c_int, [vp, vp, sz, u32, ctypes.c_double, vp, sz, vp]),
        "nttb200_packed_encoder_create": (ctypes.c_int, [ctypes.POINTER(vp), vp, u32, u32]),
        "nttb200_packed_encoder_destroy": (ctypes.c_int, [vp]),
        "nttb200_packed_encode": (ctypes.c_int, [vp, vp, u32, vp, sz, vp]),
        "nttb200_packed_decode": (ctypes.c_int, [vp, vp, u32, vp, sz, vp]),
        "nttb200_rns_keyswitch_create": (ctypes.c_int, [ctypes.POINTER(vp), vp, vp, u32, u32, u32]),
        "nttb200_rns_keyswitch_destroy": (ctypes.c_int, [vp]),
        "nttb200_rns_keyswitch_apply": (ctypes.c_int, [vp, vp, sz, vp, ctypes.POINTER(u32), u32, vp, sz, u32, vp]),
        "nttb200_rns_lintrans_keys": (ctypes.c_int, [u32, ctypes.POINTER(u32), u32, u32, ctypes.POINTER(u32),
                                                     ctypes.POINTER(u32)]),
        "nttb200_rns_lintrans_apply": (ctypes.c_int, [vp, vp, vp, ctypes.POINTER(u32), u32, u32, vp, u32, vp, sz, vp]),
        "nttb200_strerror": (ctypes.c_char_p, [ctypes.c_int]),
        "nttb200_last_error": (ctypes.c_char_p, []),
        "nttb200_kernel_launches": (ctypes.c_uint64, []),
        "nttb200_plan_last_path": (ctypes.c_char_p, [vp]),
        "nttb200_plan_logn": (u32, [vp]),
        "nttb200_plan_modulus": (u32, [vp]),
        "nttb200_version": (ctypes.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


EXPORTED_SYMBOLS = (
    "nttb200_make_roots", "nttb200_make_bitrev_table", "nttb200_powmod", "nttb200_plan_create",
    "nttb200_plan_destroy", "nttb200_plan_create_generated", "nttb200_plan_table", "nttb200_reduce",
    "nttb200_bitrev_permute", "nttb200_transpose",
    "nttb200_gs_batch", "nttb200_ct_batch", "nttb200_gs_stage_range",
    "nttb200_gs_host", "nttb200_gs_stage_range_scatter", "nttb200_host_alloc", "nttb200_host_free",
    "nttb200_pointwise", "nttb200_scale", "nttb200_polymul_negacyclic",
    "nttb200_rns_plan_create", "nttb200_rns_plan_create_logn", "nttb200_rns_plan_create_generated",
    "nttb200_rns_plan_destroy", "nttb200_rns_gs_batch",
    "nttb200_rns_ct_batch", "nttb200_rns_polymul_negacyclic",
    "nttb200_rns_pointwise", "nttb200_rns_scale", "nttb200_rns_dot", "nttb200_rns_gs_scaled_batch",
    "nttb200_rns_automorphism", "nttb200_rns_conv_create", "nttb200_rns_conv_destroy", "nttb200_rns_base_convert", "nttb200_rns_mod_down",
    "nttb200_rns_base_convert_exact", "nttb200_rns_scale_round",
    "nttb200_ckks_encoder_create", "nttb200_ckks_encoder_destroy", "nttb200_ckks_encode", "nttb200_ckks_decode",
    "nttb200_packed_encoder_create", "nttb200_packed_encoder_destroy", "nttb200_packed_encode",
    "nttb200_packed_decode",
    "nttb200_rns_keyswitch_create", "nttb200_rns_keyswitch_destroy", "nttb200_rns_keyswitch_apply",
    "nttb200_rns_lintrans_keys", "nttb200_rns_lintrans_apply",
    "nttb200_strerror", "nttb200_last_error", "nttb200_kernel_launches", "nttb200_plan_last_path",
    "nttb200_plan_logn", "nttb200_plan_modulus", "nttb200_version",
)


def _check(status: int, where: str) -> None:
    if status != 0:
        raise NttError(status, where)


def version() -> str:
    return load_library().nttb200_version().decode()


def kernel_launches() -> int:
    return int(load_library().nttb200_kernel_launches())


# ------------------------------------------------------------------ host tables
def make_roots(n: int, p: int, g: int) -> np.ndarray:
    """``root[0] = 1; make_roots(n, root, p, g)`` of the reference host
    (src/test.cpp:27-32,137-139), 64-bit safe for every p <= 2^30."""
    roots = np.zeros(n, dtype=np.int32)
    _check(load_library().nttb200_make_roots(n, roots.ctypes.data_as(_i32p), p, g), "make_roots")
    return roots


def make_bitrev_table(n: int, p: int, base: int) -> np.ndarray:
    table = np.zeros(n, dtype=np.int32)
    _check(load_library().nttb200_make_bitrev_table(n, table.ctypes.data_as(_i32p), p, base),
           "make_bitrev_table")
    return table


def powmod(b: int, e: int, m: int) -> int:
    return int(load_library().nttb200_powmod(b, e, m))


def negacyclic_tables(n: int, q: int, g: int):
    """(forward psi^bitrev table, inverse psi^-bitrev table) for x^n + 1 mod q;
    q must be a prime with 2n | q-1 and g a primitive root."""
    if (q - 1) % (2 * n):
        raise ValueError("2n must divide q-1")
    psi = powmod(g, (q - 1) // (2 * n), q)
    psi_inv = powmod(psi, q - 2, q)
    return make_bitrev_table(n, q, psi), make_bitrev_table(n, q, psi_inv)


class HostBuffer:
    """Page-locked host memory from the library (successor of the reference's host-only
    buffer objects, src/test.cpp:115-134).  `.array` is a numpy int32 view."""

    def __init__(self, words: int, write_combined: bool = False):
        self._lib = load_library()
        p = ctypes.c_void_p()
        _check(self._lib.nttb200_host_alloc(ctypes.byref(p), words * 4, 1 if write_combined else 0),
               "host_alloc")
        self.ptr = int(p.value)
        self.words = words
        self.array = np.ctypeslib.as_array((ctypes.c_int32 * words).from_address(self.ptr))

    def free(self) -> None:
        if getattr(self, "ptr", 0):
            self.array = None
            self._lib.nttb200_host_free(ctypes.c_void_p(self.ptr))
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# ------------------------------------------------------------------------- plan
def _addr(x) -> int:
    """Raw address of a device/host buffer: torch tensor, numpy array or int."""
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return int(x.data_ptr())
    if isinstance(x, np.ndarray):
        return int(x.ctypes.data)
    raise TypeError(f"cannot take the address of {type(x)!r}")


def _stream(stream) -> Optional[int]:
    if stream is None:
        return None
    if isinstance(stream, int):
        return stream
    return int(stream.cuda_stream)  # torch.cuda.Stream


class Plan:
    """One (N, q, twiddle table) on one GPU -- the successor of the compile-time
    constants + bo_root of the reference (src/aie2.py:14-19, src/test.cpp:119-144)."""

    def __init__(self, logn: int, q: int, table: np.ndarray, device: int = 0, flags: int = 0):
        table = np.ascontiguousarray(table, dtype=np.int32)
        if table.size != (1 << logn):
            raise ValueError("table must hold N = 2^logn words")
        self._lib = load_library()
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_plan_create(ctypes.byref(handle), device, logn, q,
                                             table.ctypes.data_as(_i32p), flags), "plan_create")
        self._h = handle
        self.logn, self.n, self.q, self.device, self.flags = logn, 1 << logn, q, device, flags

    @classmethod
    def generated(cls, logn: int, q: int, kind: int, base: int, gen_logn: Optional[int] = None,
                  block_mult: int = 1, device: int = 0, flags: int = 0) -> "Plan":
        """Plan whose table is generated ON THE DEVICE (nothing is shipped):
        table[h+i] = gen(h*block_mult + i), gen(e) = base^e (GEN_POWERS) or
        base^bitrev(e) over gen_logn bits (GEN_BITREV).  See nttb200_plan_create_generated."""
        self = cls.__new__(cls)
        self._lib = load_library()
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_plan_create_generated(
            ctypes.byref(handle), device, logn, q, kind, base,
            logn if gen_logn is None else gen_logn, block_mult, flags), "plan_create_generated")
        self._h = handle
        self.logn, self.n, self.q, self.device, self.flags = logn, 1 << logn, q, device, flags
        return self

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.nttb200_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def last_path(self) -> str:
        return self._lib.nttb200_plan_last_path(self._h).decode()

    def table(self) -> np.ndarray:
        """The plan's table as the reference host would hold it in bo_root."""
        out = np.empty(self.n, dtype=np.int32)
        _check(self._lib.nttb200_plan_table(self._h, out.ctypes.data_as(_i32p)), "plan_table")
        return out

    def bitrev_permute(self, d_in, d_out, batch: int, stream=None) -> None:
        """out[b][i] = in[b][bitrev(i)] (in place allowed)."""
        _check(self._lib.nttb200_bitrev_permute(self._h, _addr(d_in), _addr(d_out), batch,
                                                _stream(stream)), "bitrev_permute")

    def transpose(self, d_in, d_out, batch: int, to_batch_minor: bool, stream=None) -> None:
        """[batch][N] -> [N][batch] (to_batch_minor) or back; out of place."""
        _check(self._lib.nttb200_transpose(self._h, _addr(d_in), _addr(d_out), batch,
                                           1 if to_batch_minor else 0, _stream(stream)), "transpose")

    def reduce(self, d_in, d_out, count: int, stream=None) -> None:
        """out = in mod q for arbitrary int32 words (the golden's `%` on first touch)."""
        _check(self._lib.nttb200_reduce(self._h, _addr(d_in), _addr(d_out), count,
                                        _stream(stream)), "reduce")

    def gs(self, d_in, d_out, batch: int, stage: int = -1, stream=None) -> None:
        """Golden network ``ntt(a, n, roots, p, stage)`` (src/test.cpp:34-60) on device."""
        _check(self._lib.nttb200_gs_batch(self._h, _addr(d_in), _addr(d_out), batch, stage,
                                          _stream(stream)), "gs_batch")

    def ct(self, d_in, d_out, batch: int, stage: int = -1, stream=None) -> None:
        _check(self._lib.nttb200_ct_batch(self._h, _addr(d_in), _addr(d_out), batch, stage,
                                          _stream(stream)), "ct_batch")

    def gs_stage_range(self, d_in, d_out, batch: int, stage_begin: int, stage_end: int,
                       stream=None) -> None:
        _check(self._lib.nttb200_gs_stage_range(self._h, _addr(d_in), _addr(d_out), batch,
                                                stage_begin, stage_end, _stream(stream)),
               "gs_stage_range")

    def gs_stage_range_scatter(self, d_buf, stage_begin: int, stage_end: int, peer_ptrs, rank: int,
                               stream=None) -> None:
        """Stages [stage_begin, logn) of one vector with the results stored into the peers'
        receive buffers (the all-to-all fused into the last pass)."""
        world = len(peer_ptrs)
        arr = (ctypes.c_void_p * world)(*[int(x) for x in peer_ptrs])
        _check(self._lib.nttb200_gs_stage_range_scatter(self._h, _addr(d_buf), stage_begin,
                                                        stage_end, arr, world, rank,
                                                        _stream(stream)), "gs_stage_range_scatter")

    def gs_host(self, h_in, h_out, batch: int, stage: int = -1) -> None:
        """Host buffers in, host buffers out (the reference's BO sync + launch + sync,
        src/test.cpp:148-168)."""
        _check(self._lib.nttb200_gs_host(self._h, _addr(h_in), _addr(h_out), batch, stage),
               "gs_host")

    def pointwise(self, d_a, d_b, d_c, count: int, stream=None) -> None:
        _check(self._lib.nttb200_pointwise(self._h, _addr(d_a), _addr(d_b), _addr(d_c), count,
                                           _stream(stream)), "pointwise")

    def scale(self, d_a, d_c, count: int, scalar: int, stream=None) -> None:
        _check(self._lib.nttb200_scale(self._h, _addr(d_a), _addr(d_c), count, scalar,
                                       _stream(stream)), "scale")


class RnsPlan:
    """Polynomials of N = 2^logn (4096..65536) in RNS form: L channels with their own primes
    and tables, data laid out [batch][L][N]; one launch per pass serves all channels."""

    def __init__(self, qs, tables, device: int = 0, logn: int = 12):
        self._lib = load_library()
        self.limbs = len(qs)
        n = 1 << logn
        tabs = [np.ascontiguousarray(t, dtype=np.int32) for t in tables]
        if len(tabs) != self.limbs or any(t.size != n for t in tabs):
            raise ValueError(f"one {n}-word table per modulus")
        qarr = (ctypes.c_uint32 * self.limbs)(*[int(q) for q in qs])
        parr = (_i32p * self.limbs)(*[t.ctypes.data_as(_i32p) for t in tabs])
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_rns_plan_create_logn(ctypes.byref(handle), device, logn, self.limbs,
                                                      qarr, parr, 0), "rns_plan_create_logn")
        self._h = handle
        self.qs = [int(q) for q in qs]
        self.logn, self.n, self.device = logn, n, device

    @classmethod
    def generated(cls, logn: int, qs, kind: int, bases, device: int = 0) -> "RnsPlan":
        """Plan whose channel tables are generated ON THE DEVICE: channel l's table is the
        one Plan.generated(logn, qs[l], kind, bases[l]) builds.  kind = GEN_BITREV with
        bases[l] = psi_l gives the forward table, psi_l^-1 the inverse one."""
        self = cls.__new__(cls)
        self._lib = load_library()
        self.limbs = len(qs)
        if len(bases) != self.limbs:
            raise ValueError("one base per modulus")
        qarr = (ctypes.c_uint32 * self.limbs)(*[int(q) for q in qs])
        barr = (ctypes.c_uint32 * self.limbs)(*[int(b) for b in bases])
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_rns_plan_create_generated(ctypes.byref(handle), device, logn, self.limbs,
                                                           qarr, kind, barr, 0), "rns_plan_create_generated")
        self._h = handle
        self.qs = [int(q) for q in qs]
        self.logn, self.n, self.device = logn, 1 << logn, device
        return self

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.nttb200_rns_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def gs(self, d_in, d_out, batch: int, stream=None) -> None:
        _check(self._lib.nttb200_rns_gs_batch(self._h, _addr(d_in), _addr(d_out), batch,
                                              _stream(stream)), "rns_gs_batch")

    def ct(self, d_in, d_out, batch: int, stream=None) -> None:
        _check(self._lib.nttb200_rns_ct_batch(self._h, _addr(d_in), _addr(d_out), batch,
                                              _stream(stream)), "rns_ct_batch")

    def gs_scaled(self, d_in, d_out, batch: int, stream=None) -> None:
        """GS on every channel with every output times N^-1 mod q_l: the inverse NTT of a plan
        holding psi_l^-bitrev tables."""
        _check(self._lib.nttb200_rns_gs_scaled_batch(self._h, _addr(d_in), _addr(d_out), batch,
                                                     _stream(stream)), "rns_gs_scaled_batch")

    def pointwise(self, op: int, d_a, d_b, d_c, batch: int, b_batch: Optional[int] = None,
                  stream=None) -> None:
        """c = a op b per channel (op: RNS_ADD / RNS_SUB / RNS_MUL).  b_batch = 1 broadcasts one
        [L][N] operand over the batch; None means b_batch = batch."""
        _check(self._lib.nttb200_rns_pointwise(self._h, op, _addr(d_a), _addr(d_b), _addr(d_c), batch,
                                               batch if b_batch is None else b_batch, _stream(stream)),
               "rns_pointwise")

    def scale(self, d_a, d_c, batch: int, scalars, stream=None) -> None:
        """c[b][l] = a[b][l] * scalars[l] mod q_l (one host scalar per channel)."""
        if len(scalars) != self.limbs:
            raise ValueError("one scalar per modulus")
        arr = (ctypes.c_uint32 * self.limbs)(*[int(s) for s in scalars])
        _check(self._lib.nttb200_rns_scale(self._h, _addr(d_a), _addr(d_c), batch, arr, _stream(stream)),
               "rns_scale")

    def automorphism(self, d_in, d_out, batch: int, galois, domain: int = AUTO_EVAL, stream=None) -> None:
        """out[c][b][l] = sigma_{galois[c]}(in[b][l]): X -> X^g on every channel, in the evaluation
        (rns_ct) order (AUTO_EVAL) or on coefficients (AUTO_COEFF).  galois: one odd g in [1, 2N) or
        a sequence of 1..64 of them; d_out holds [len(galois)][batch][L][N]."""
        gs = [int(galois)] if isinstance(galois, (int, np.integer)) else [int(g) for g in galois]
        arr = (ctypes.c_uint32 * max(len(gs), 1))(*gs)
        _check(self._lib.nttb200_rns_automorphism(self._h, _addr(d_in), _addr(d_out), batch, arr, len(gs),
                                                  domain, _stream(stream)), "rns_automorphism")


class RnsConv:
    """Basis conversion from the primes of `src` (S channels, product B) to those of `dst`
    (T channels), coefficient domain.  The object copies what it needs: the plans may be closed
    afterwards.  See nttb200_rns_conv_create for the rules."""

    def __init__(self, src: RnsPlan, dst: RnsPlan):
        self._lib = load_library()
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_rns_conv_create(ctypes.byref(handle), src._h, dst._h, 0), "rns_conv_create")
        self._h = handle
        self.src_qs, self.dst_qs = list(src.qs), list(dst.qs)
        self.logn, self.n = src.logn, src.n

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.nttb200_rns_conv_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def convert(self, d_in, d_out, batch: int, in_stride: int = 0, out_stride: int = 0, exact: bool = False,
                stream=None) -> None:
        """Fast base conversion (ModUp): out[b][j] = sum_i [in[b][i] (B/b_i)^-1]_{b_i} (B/b_i) mod c_j,
        i.e. (x + alpha B) mod c_j with 0 <= alpha < S.  exact: the centred value instead,
        x_c mod c_j with x_c = x (mod B) in (-B/2, B/2] (see nttb200_rns_base_convert_exact for the
        rounding band).  Strides in words between polynomials (0: dense S*N / T*N)."""
        if exact:
            _check(self._lib.nttb200_rns_base_convert_exact(self._h, _addr(d_in), in_stride, _addr(d_out),
                                                            out_stride, batch, _stream(stream)),
                   "rns_base_convert_exact")
        else:
            _check(self._lib.nttb200_rns_base_convert(self._h, _addr(d_in), in_stride, _addr(d_out), out_stride,
                                                      batch, _stream(stream)), "rns_base_convert")

    def mod_down(self, d_in, d_out, batch: int, round: bool = False, stream=None) -> None:
        """Divide by B and drop the source channels: d_in [batch][T+S][N] (target channels
        first), d_out [batch][T][N]; floor((X + (floor(B/2) if round else 0)) / B) - alpha."""
        _check(self._lib.nttb200_rns_mod_down(self._h, _addr(d_in), _addr(d_out), batch,
                                              RNS_ROUND if round else 0, _stream(stream)), "rns_mod_down")

    def scale_round(self, d_in, d_out, batch: int, t: int = 1, stream=None) -> None:
        """round(t X / B) on the target channels: d_in [batch][T+S][N] (target channels first),
        d_out [batch][T][N]; 1 <= t < 2^32.  The BFV tensor-product scaling (t/Q) and, with
        t = 1, the exact rounded division by B."""
        _check(self._lib.nttb200_rns_scale_round(self._h, _addr(d_in), _addr(d_out), batch, t, _stream(stream)),
               "rns_scale_round")


class CkksEncoder:
    """CKKS slot encoding on the moduli and N of `plan`: n = N/2 complex slots, slot j holding
    m(zeta^(5^j mod 2N)) with zeta = e^(i pi / N).  Slots are complex128 [batch][n] tensors,
    polynomials int32 [batch][L][N] residues in the coefficient domain.  The object copies what
    it needs: the plan may be closed afterwards.  See nttb200_ckks_encoder_create for the rules."""

    def __init__(self, plan: RnsPlan):
        self._lib = load_library()
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_ckks_encoder_create(ctypes.byref(handle), plan._h, 0), "ckks_encoder_create")
        self._h = handle
        self.qs = list(plan.qs)
        self.logn, self.n, self.slots = plan.logn, plan.n, plan.n // 2

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.nttb200_ckks_encoder_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def encode(self, d_slots, d_out, batch: int, scale: float, stream=None) -> None:
        """d_out[b][l][k] = rint(scale * m_k) mod q_l, m the real polynomial whose slots are d_slots[b]."""
        _check(self._lib.nttb200_ckks_encode(self._h, _addr(d_slots), float(scale), _addr(d_out), batch,
                                             _stream(stream)), "ckks_encode")

    def decode(self, d_in, d_slots, batch: int, scale: float, channels: Optional[int] = None, in_stride: int = 0,
               stream=None) -> None:
        """d_slots[b] = the slots of x_c / scale, x_c the centred CRT value of the first `channels`
        rows (default min(L, 4)) of polynomial b at d_in + b * in_stride (0: dense)."""
        c = min(len(self.qs), 4) if channels is None else channels
        _check(self._lib.nttb200_ckks_decode(self._h, _addr(d_in), in_stride, c, float(scale), _addr(d_slots),
                                             batch, _stream(stream)), "ckks_decode")


class PackedEncoder:
    """Packed integer slots mod t (BFV / BGV batch encoding) on the moduli and N of `plan`: N slots
    as a 2 x N/2 matrix, slot r N/2 + j holding m(psi^e) mod t with e = 5^j mod 2N (row 0) or
    2N - (5^j mod 2N) (row 1), psi the smallest primitive 2N-th root mod t.  t: a prime below 2^30
    with t = 1 (mod 2N), dividing no channel modulus.  Slots are int32 [batch][N] tensors,
    polynomials int32 [batch][L][N] residues in the coefficient domain.  The object copies what it
    needs: the plan may be closed afterwards.  See nttb200_packed_encoder_create for the rules."""

    def __init__(self, plan: RnsPlan, t: int):
        self._lib = load_library()
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_packed_encoder_create(ctypes.byref(handle), plan._h, int(t), 0),
               "packed_encoder_create")
        self._h = handle
        self.qs, self.t = list(plan.qs), int(t)
        self.logn, self.n = plan.logn, plan.n

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.nttb200_packed_encoder_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def encode(self, d_slots, d_out, batch: int, centred: bool = False, stream=None) -> None:
        """d_out[b][l] = round(Q m / t) mod q_l (BFV), or with centred m_c mod q_l, m_c in (-t/2, t/2]
        (BGV, BFV plaintext operand); m the plaintext whose slots are d_slots[b] mod t (signed words)."""
        _check(self._lib.nttb200_packed_encode(self._h, _addr(d_slots), PACK_CENTRED if centred else PACK_SCALED,
                                               _addr(d_out), batch, _stream(stream)), "packed_encode")

    def decode(self, d_in, d_slots, batch: int, centred: bool = False, stream=None) -> None:
        """d_slots[b] = the slots of the plaintext d_in[b] (canonical residues mod t, coefficient
        domain), in [0, t), or in (-t/2, t/2] with centred."""
        _check(self._lib.nttb200_packed_decode(self._h, _addr(d_in), PACK_CENTRED if centred else 0,
                                               _addr(d_slots), batch, _stream(stream)), "packed_decode")


class KeySwitcher:
    """Hybrid key switching on the [Q | P] channels of a forward / inverse plan pair: Q the first
    q_limbs channels, digits of alpha primes (dnum = ceil(q_limbs / alpha), the last one may be
    shorter), P the rest.  The object copies what it needs: the plans may be closed afterwards.
    See nttb200_rns_keyswitch_create for the rules and the key layout."""

    def __init__(self, qp_fwd: RnsPlan, qp_inv: RnsPlan, q_limbs: int, alpha: int):
        self._lib = load_library()
        handle = ctypes.c_void_p()
        _check(self._lib.nttb200_rns_keyswitch_create(ctypes.byref(handle), qp_fwd._h, qp_inv._h, q_limbs, alpha, 0),
               "rns_keyswitch_create")
        self._h = handle
        self.qs = list(qp_fwd.qs)
        self.q_limbs, self.alpha = q_limbs, alpha
        self.dnum = -(-q_limbs // alpha)
        self.logn, self.n = qp_fwd.logn, qp_fwd.n

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.nttb200_rns_keyswitch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def switch(self, d_in, d_keys, d_out, batch: int, galois=1, in_stride: int = 0, coeff_in: bool = False,
               coeff_out: bool = False, stream=None) -> None:
        """d_out[c][b] = (u0, u1) = ModDown(sum_i sigma_g(ModUp(x_b)_i) * key[c][i]) with g = galois[c]:
        d_in [batch][L][N] on Q (rows at d_in + b * in_stride, 0: dense), d_keys
        [count][dnum][2][L+K][N] on Q P in the rns_ct order, d_out [count][batch][2][L][N].  galois:
        one odd g in [1, 2N) (1: relinearisation) or a sequence of 1..64 of them (hoisted rotations).
        coeff_in / coeff_out: input / output in coefficients instead of the rns_ct order."""
        gs = [int(galois)] if isinstance(galois, (int, np.integer)) else [int(g) for g in galois]
        arr = (ctypes.c_uint32 * max(len(gs), 1))(*gs)
        flags = (KS_COEFF_IN if coeff_in else 0) | (KS_COEFF_OUT if coeff_out else 0)
        _check(self._lib.nttb200_rns_keyswitch_apply(self._h, _addr(d_in), in_stride, _addr(d_keys), arr, len(gs),
                                               _addr(d_out), batch, flags, _stream(stream)), "rns_keyswitch_apply")

    def linear_transform(self, d_ct, d_diags, offsets, n1: int, d_keys, d_out, batch: int, stream=None) -> None:
        """y = M z on the slots of every ciphertext, M given by its generalised diagonals
        y[s] = sum_k d_k[s] z[(s + k) mod N/2], by baby-step giant-step with n1 babies: d_ct
        [batch][2][L][N] in the rns_ct order, d_diags [count][L][N] the encoded d_k in the rns_ct order
        and the order of offsets (each in [0, N/2)), d_keys [nkeys][dnum][2][L+K][N] for the elements of
        lintrans_galois(N, offsets, n1) in that order (None when there are none), d_out [batch][2][L][N],
        not rescaled."""
        offs = [int(k) for k in offsets]
        arr = (ctypes.c_uint32 * max(len(offs), 1))(*offs)
        nkeys = len(lintrans_galois(self.n, offs, n1))
        _check(self._lib.nttb200_rns_lintrans_apply(self._h, _addr(d_ct), _addr(d_diags), arr, len(offs), n1,
                                                    0 if d_keys is None else _addr(d_keys), nkeys, _addr(d_out),
                                                    batch, _stream(stream)),
               "rns_lintrans_apply")


def rns_polymul_negacyclic(fwd: RnsPlan, inv: RnsPlan, d_a, d_b, d_c, batch: int, stream=None) -> None:
    _check(fwd._lib.nttb200_rns_polymul_negacyclic(fwd._h, inv._h, _addr(d_a), _addr(d_b),
                                                   _addr(d_c), batch, _stream(stream)),
           "rns_polymul_negacyclic")


def rns_dot(plan: RnsPlan, d_a, d_w, d_c, terms: int, batch: int, w_batch: Optional[int] = None,
            accumulate: bool = False, stream=None) -> None:
    """c = (c if accumulate else 0) + sum_k a[k] * w[k] per channel.  d_a: [terms][batch][L][N],
    d_w: [terms][w_batch][L][N] with w_batch = batch (None) or 1 (one key for the batch)."""
    _check(plan._lib.nttb200_rns_dot(plan._h, _addr(d_a), _addr(d_w), _addr(d_c), terms, batch,
                                     batch if w_batch is None else w_batch, 1 if accumulate else 0,
                                     _stream(stream)), "rns_dot")


def galois_rotation(n: int, steps: int) -> int:
    """Galois element of a CKKS slot rotation by `steps` (negative: the other way) at ring
    degree n: 5^steps mod 2n.  5 has order n/2 modulo 2n, so -r is 5^(r mod n/2)."""
    return pow(5, steps % (n // 2), 2 * n)


def lintrans_galois(n: int, offsets, n1: int) -> list:
    """The Galois elements whose keys KeySwitcher.linear_transform needs at ring degree n, in the
    order it reads them: the baby rotations j = k mod n1 >= 1 that occur, ascending, then the giant
    rotations n1 i (i = k // n1 >= 1) that occur, ascending."""
    lib = load_library()
    offs = [int(k) for k in offsets]
    arr = (ctypes.c_uint32 * max(len(offs), 1))(*offs)
    count = ctypes.c_uint32()
    logn = n.bit_length() - 1
    _check(lib.nttb200_rns_lintrans_keys(logn, arr, len(offs), n1, None, ctypes.byref(count)), "rns_lintrans_keys")
    out = (ctypes.c_uint32 * max(count.value, 1))()
    _check(lib.nttb200_rns_lintrans_keys(logn, arr, len(offs), n1, out, ctypes.byref(count)), "rns_lintrans_keys")
    return [int(g) for g in out[:count.value]]


def galois_conjugate(n: int) -> int:
    """Galois element of complex conjugation of the CKKS slots: 2n - 1 (X -> X^-1)."""
    return 2 * n - 1


def polymul_negacyclic(fwd: Plan, inv: Plan, d_a, d_b, d_c, batch: int, stream=None) -> None:
    _check(fwd._lib.nttb200_polymul_negacyclic(fwd._h, inv._h, _addr(d_a), _addr(d_b), _addr(d_c),
                                               batch, _stream(stream)), "polymul_negacyclic")


def ntt(a: np.ndarray, n: int, roots: np.ndarray, p: int, stage: int = -1, device: int = 0,
        flags: int = 0) -> np.ndarray:
    """Drop-in for the golden call ``ntt(a, n, roots_rev, p, stage)`` (src/test.cpp:34):
    host arrays in, transformed copy out, computed on the GPU through
    ``nttb200_gs_host``.  ``a`` may be 1-D (one polynomial) or 2-D (a batch).  Like the
    golden, inputs need not be reduced (``a[i] = i`` with n > p is fine): they are taken
    mod p on first touch."""
    a = np.ascontiguousarray(a, dtype=np.int32)
    if a.shape[-1] != n or n & (n - 1) or n < 2:
        raise ValueError("last dimension must be n, a power of two >= 2")
    out = np.empty_like(a)
    batch = a.size // n
    with Plan(n.bit_length() - 1, p, roots, device=device, flags=flags) as plan:
        plan.gs_host(a, out, batch, stage)
    return out
