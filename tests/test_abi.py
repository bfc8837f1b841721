"""C-ABI library: loads and exports every symbol include/b200fm.h declares (no compute calls; runs without a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200fm.h")).read()
    return sorted(set(re.findall(r"\b(b200fm_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    from b200fm import lib
    return lib


def test_library_exports_every_declared_symbol(built):
    lib = built.load()
    syms = _declared_symbols()
    assert len(syms) >= 8
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/b200fm.h but not exported"
    assert lib.b200fm_abi_version() == 1
    assert set(built.SIGNATURES) | {"b200fm_last_error"} == set(syms), "ctypes table out of sync with the header"


def test_argument_validation_without_gpu(built):
    lib = built.load()
    # bad arguments are rejected before any CUDA call
    rc = lib.b200fm_gemm_bf16(0, 0, 0, 0, 0, None, 8, None, 8, None, 8, None, 0, None, None, 0, 1.0, None, None)
    assert rc != 0 and b"empty problem" in lib.b200fm_last_error()
    rc = lib.b200fm_vq_argmax(None, None, None, None, 5, 16, 7, 1, None)
    assert rc != 0 and b"latent dim" in lib.b200fm_last_error()


def test_ops_refuse_cpu_tensors(built):
    import torch
    from b200fm import ops
    with pytest.raises(built.B200FMError):
        ops.vq_argmax(torch.zeros(4, 32), torch.zeros(8, 32))


def test_runtime_options_roundtrip(built):
    """b200fm_set_option / b200fm_get_option (no GPU needed): defaults, override, unknown names are errors with a message."""
    from b200fm import lib
    assert lib.get_option("pdl") == 1 and lib.get_option("gemm_cta_pairs") == 1 and lib.get_option("ln_bwd_v2") == 1
    assert lib.get_option("gemv") == 1 and lib.get_option("gemv_prefetch") == 1 and lib.get_option("gemm_debug") == 0
    assert lib.get_option("gemm_tma_store") == 1 and lib.get_option("comm_slim") == 1 and lib.get_option("attn_bwd_warps") == 8
    lib.set_option("pdl", 0)
    assert lib.get_option("pdl") == 0
    lib.set_option("pdl", 1)
    assert lib.get_option("pdl") == 1
    with pytest.raises(lib.B200FMError, match="unknown option"):
        lib.set_option("no_such_option", 1)


def test_library_is_tcgen05_tma_code(built):
    """The shipped library is sm_100a code that uses the Blackwell tensor path: tcgen05.mma (SASS UTCHMMA), TMA tensor loads (UTMALDG),
    TMA tensor stores in the GEMM epilogue (UTMASTG), TMEM read-out (LDTM) -- and no legacy mma.sync (HMMA) anywhere."""
    import re
    import shutil
    import subprocess
    from b200fm import build, lib
    # the toolkit that built the library ships cuobjdump next to nvcc, whether or not it is on PATH
    cuobjdump = shutil.which("cuobjdump", path=os.path.dirname(build.NVCC)) or shutil.which("cuobjdump")
    if cuobjdump is None:
        pytest.skip("cuobjdump not found")
    sass = subprocess.run([cuobjdump, "-sass", lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout
    assert "sm_100a" in sass or "SM100" in sass.upper()
    per_fn, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            per_fn[cur] = set()
            continue
        if cur is not None:
            for k in ("UTCHMMA", "UTMALDG", "UTMASTG", "LDTM", "HMMA"):
                if re.search(r"(?<![A-Z])" + k + r"(?![A-Z])", line):
                    per_fn[cur].add(k)
    gemm = [v for f, v in per_fn.items() if "gemm_kernel" in f]
    attn = [v for f, v in per_fn.items() if "attention_fwd_kernel" in f or "attention_bwd_kernel" in f]
    assert gemm and all({"UTCHMMA", "UTMALDG", "LDTM"} <= v for v in gemm)
    assert any("UTMASTG" in v for v in gemm)
    assert attn and all({"UTCHMMA", "UTMALDG", "LDTM"} <= v for v in attn)
    assert not any("HMMA" in v for v in per_fn.values())
