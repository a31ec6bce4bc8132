"""The C-ABI library loads on a machine without a GPU and exports every symbol the header declares."""
import ctypes as C
import os
import re
import subprocess

import porla_b200 as pb
from porla_b200 import lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "porla_multiexp.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set()
    for m in re.finditer(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", src):
        n = m.group(1)
        if n in ("defined", "sizeof") or n.startswith("porla_secp256k1_ecmult_multi_callback"):
            continue
        names.add(n)
    return {n for n in names if n.startswith("porla_") or n in L.LEGACY_SYMBOLS or n.startswith("compute_") or n.startswith("bn254_")} - {"fn"}


def test_library_exports_every_declared_symbol():
    lib = C.CDLL(pb.LIB_PATH)
    want = declared_symbols()
    assert set(L.LEGACY_SYMBOLS) <= want and len(L.LEGACY_SYMBOLS) == 14
    assert set(L.NEW_SYMBOLS) <= want, set(L.NEW_SYMBOLS) - want
    for name in sorted(want):
        assert hasattr(lib, name), name


def test_legacy_symbols_match_reference_header_names():
    """Same 14 names, in the same order, as the reference's cgo header (Utils/libmultiexp.h:71-84), which
    include/porla_multiexp.h restates first."""
    expected = ["init_key", "init_SRS", "init_SRS_from_data", "compute_digest", "compute_digest_complement",
                "compute_digest_from_srs", "compute_multi_exp", "compare_commitment", "create_proof", "verify_proof",
                "add_point", "mult_point", "neg_point", "set_inf_point"]
    assert L.LEGACY_SYMBOLS == expected
    names = re.findall(r"extern\s+\w+\s+(\w+)\(", open(os.path.join(ROOT, "include", "porla_multiexp.h")).read())
    assert names[:14] == expected


def test_library_is_sm100a_cuda_code():
    out = subprocess.run(["cuobjdump", "-lelf", pb.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        return  # cuobjdump not available
    assert "sm_100a" in out.stdout


def test_product_does_not_import_the_oracle():
    """The oracle is test infrastructure: nothing under porla_b200/ may import, link or load it."""
    banned = ("import oracle", "from oracle", "liboracle", "libsecp_ref", "oracle/", "curves_py")
    for dirpath, _, files in os.walk(os.path.join(ROOT, "porla_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                for b in banned:
                    assert b not in txt, (f, b)
