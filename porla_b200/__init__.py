"""porla_b200 -- B200-native multi-scalar-multiplication engine behind Porla's libmultiexp C-ABI.

The product is ``libmultiexp.so`` (CUDA, sm_100a; sources in ``porla_b200/csrc``, C-ABI in
``include/porla_multiexp.h``).  This Python package is only the host-side mirror of the reference's
C++ glue (``/root/reference/porla/Utils/utils.h:235-305``: ``bn254_add``, ``bn254_mult``,
``bn254_neg``, ``bn254_set_infinity``, ``bn254_scalar_set_int``, ``bn254_multi_exp``,
``bn254_compare``) over ``ctypes``, used by the tests and the benchmark.  There is no Python or CPU
implementation of the MSM here: if the shared library is missing, importing ``porla_b200.lib``
raises, and without a GPU every MSM entry point aborts the process with a diagnostic.
"""
from .lib import (  # noqa: F401
    LIB_PATH,
    CURVE_BN254,
    CURVE_SECP256K1,
    SCALAR_BE32,
    SCALAR_LE32,
    POINT_BE64,
    POINT_LE64,
    GoSlice,
    load,
    bn254_add,
    bn254_mult,
    bn254_neg,
    bn254_set_infinity,
    bn254_scalar_set_int,
    bn254_multi_exp,
    bn254_multi_exp_batch,
    bn254_compare,
    bn254_butterfly_stage,
    Kzg,
    Table,
    MultiTable,
    msm_host,
    msm_host_devices,
    secp256k1_ecmult_multi_var,
    secp256k1_butterfly_stage,
    secp256k1_ecmult_multi_gej,
    secp256k1_ecmult_const_batch,
    SecpGenerators,
)
