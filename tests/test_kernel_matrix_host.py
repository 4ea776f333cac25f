"""CPU: every instantiation of the templated aggregation and GEMM kernels in the built library has a case in
tests/test_gpu_kernel_matrix.py (or an EXEMPT entry with its reason), and every kernel those cases expect exists.
Adding a kernel variant without a test, or removing one a test still expects, fails here."""
import re
import shutil
import subprocess

import pytest

from relationprediction_b200 import _lib
from test_gpu_kernel_matrix import CASES, EXEMPT, normalize_kernel_name

FAMILIES = ("k_basis_agg", "k_basis_dc", "k_block_agg", "k_block_dw", "k_block_rel", "k_block_relg",
            "k_block_stg", "k_block_team", "k_gemm_tf32x3", "k_gemm_tn_tf32x3")


def library_kernels():
    """Normalised names of every kernel in the built library (cuobjdump -symbols, demangled by cu++filt)."""
    _lib.load()
    dump = subprocess.run(["cuobjdump", "-symbols", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"\b_Z\w+", dump)))
    demangled = subprocess.run(["cu++filt"], input="\n".join(mangled), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    return {n for n in (normalize_kernel_name(x) for x in demangled) if n}


def test_name_normaliser_agrees_across_demanglers():
    cupti = "void (anonymous namespace)::k_block_team<8, 1, true, true, 4, 4, 3, 8>(WorkItem const*, int, float*)"
    filt = "void <unnamed>::k_block_team<(int)8, (int)1, (bool)1, (bool)1, (int)4, (int)4, (int)3, (int)8>(T1, T2)"
    assert normalize_kernel_name(cupti) == normalize_kernel_name(filt) == "k_block_team<8,1,1,1,4,4,3,8>"
    assert normalize_kernel_name("k_split_b(float const*, long, int, int, int, float*, float*)") == "k_split_b"
    assert normalize_kernel_name("void k_gemm_tf32x3<0>(float const*)") == "k_gemm_tf32x3<0>"
    assert normalize_kernel_name("aten::topk_out") is None


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None,
                    reason="cuobjdump / cu++filt not on PATH")
def test_every_kernel_instantiation_has_a_case():
    in_lib = {n for n in library_kernels() if n.split("<")[0] in FAMILIES}
    assert len(in_lib) > 100, sorted(in_lib)
    covered = {k for c in CASES for k in c.expect}
    missing = sorted(in_lib - covered - set(EXEMPT))
    assert not missing, "instantiations without a case in test_gpu_kernel_matrix.CASES: %s" % missing
    stale = sorted((covered | set(EXEMPT)) - library_kernels())
    assert not stale, "kernels named by CASES / EXEMPT that the library does not contain: %s" % stale
    assert not covered & set(EXEMPT), sorted(covered & set(EXEMPT))
