"""ntt-aie_b200 -- B200-native NTT engine, Python host mirror of the C ABI.

The product is ``lib/libnttb200.so`` (hand-written sm_100a CUDA behind the C ABI in
``include/nttb200.h``).  This package is the thin ctypes mirror of that ABI with the
reference's operator names (``make_roots``, ``ntt`` -- src/test.cpp:27-60); it holds
no compute of its own and has NO CPU fallback: if the library cannot be loaded, or
no B200 is visible, calls raise.

The directory name contains a hyphen (it is the reference's name), so import it via
the root-level shim: ``import ntt_aie_b200``.
"""
from .api import (  # noqa: F401
    NttError,
    Plan,
    HostBuffer,
    RnsPlan,
    RnsConv,
    CkksEncoder,
    PackedEncoder,
    KeySwitcher,
    rns_polymul_negacyclic,
    rns_dot,
    RNS_ADD,
    RNS_SUB,
    RNS_MUL,
    RNS_ROUND,
    AUTO_COEFF,
    AUTO_EVAL,
    PACK_SCALED,
    PACK_CENTRED,
    KS_COEFF_IN,
    KS_COEFF_OUT,
    galois_rotation,
    galois_conjugate,
    lintrans_galois,
    ORDER_AIE_DEVICE,
    ORDER_GOLDEN,
    FORCE_GENERIC,
    REDUCE_INPUT,
    INPUT_BITREV,
    OUTPUT_BITREV,
    GEN_POWERS,
    GEN_BITREV,
    kernel_launches,
    lib_path,
    load_library,
    make_bitrev_table,
    make_roots,
    ntt,
    polymul_negacyclic,
    EXPORTED_SYMBOLS,
    negacyclic_tables,
    powmod,
    version,
)
