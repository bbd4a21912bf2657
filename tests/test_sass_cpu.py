"""The built library really is Blackwell-native code: the SASS of its hot kernels contains the tcgen05 / TMA / TMEM instructions
(no GPU needed: cuobjdump disassembles the sm_100a cubin).  Mnemonics:
UTCHMMA = tcgen05.mma (.2CTA = cta_group::2), UTMALDG / UTMASTG = TMA load / store, LDTM = tcgen05.ld, UTCBAR = tcgen05.commit."""
import os
import re
import shutil
import subprocess

import pytest

SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ddpm_torch_b200", "libddpm_b200.so")


def _cuobjdump():
    """cuobjdump from PATH, else from the toolkit csrc/build.sh compiles with ($NVCC, by default /usr/local/cuda/bin/nvcc)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.dirname(nvcc))


@pytest.fixture(scope="module")
def sass():
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump not found")
    if not os.path.exists(SO):
        pytest.fail("libddpm_b200.so is not built (python -c 'import __graft_entry__ as g; g.build()')")
    txt = subprocess.run([tool, "-sass", SO], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in txt
    per = {}
    cur = None
    for ln in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = m.group(1); per[cur] = set(); continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]+)", ln)
        if m and cur:
            per[cur].add(m.group(1))
    return per


def ops_of(per, needle):
    hits = [ops for fn, ops in per.items() if needle in fn]
    assert hits, f"no kernel matching {needle}"
    return hits


def has(ops, prefix):
    return any(o.startswith(prefix) for o in ops)


def test_haloed_pair_conv_uses_cta_group_2_mma_tma_and_tmem(sass):
    for ops in ops_of(sass, "conv3x3_halo2_kernel"):
        assert has(ops, "UTCHMMA.2CTA") and has(ops, "UTMALDG") and has(ops, "UTMASTG") and has(ops, "LDTM") and has(ops, "UTCBAR.2CTA")
        assert has(ops, "UCGABAR")                      # cluster barrier of the pair


def test_gemm_engine_and_attention_use_tcgen05(sass):
    for needle in ("umma_gemm_kernel", "attn_kernel", "conv3x3_halo_kernel"):
        for ops in ops_of(sass, needle):
            assert has(ops, "UTCHMMA") and has(ops, "UTMALDG") and has(ops, "LDTM"), needle


def test_no_legacy_tensor_core_paths(sass):
    """mma.sync / wmma (HMMA) kernels are the baseline this project replaces: none may be in the library."""
    for fn, ops in sass.items():
        assert not any(o.startswith("HMMA") or o.startswith("IMMA") for o in ops), fn
