"""CPU check of the BUILT library's machine code (`cuobjdump -sass`, no GPU needed): the hot-path kernels are Blackwell-native - tcgen05 MMAs
(`UTCHMMA`), TMEM loads (`LDTM`), TMA tensor loads / stores (`UTMALDG` / `UTMASTG`), the in-place residual as a TMA reduce-add (`UTMAREDG`) or a
vector reduction (`REDG...F32x4`) - and the Swin-v1 forward attention kernels contain no legacy `HMMA` (mma.sync)."""
import collections
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "cs-vit_b200", "lib", "libcsvit_sm100.so")
MNEMONICS = re.compile(r"\b(UTCHMMA|UTMALDG|UTMASTG|UTMAREDG|LDTM|HMMA)\b|\b(REDG)\.E\.ADD\.F32x4")
# PATH first, else $CUDA_HOME/bin, else /usr/local/cuda/bin (csrc/Makefile's default nvcc): an unprivileged shell often lacks it on PATH
CUOBJDUMP = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin"))


@pytest.fixture(scope="module")
def sass_counts():
    if not os.path.exists(LIB):
        pytest.skip("library not built (run __graft_entry__.build())")
    if not CUOBJDUMP or not shutil.which("c++filt"):
        pytest.skip("cuobjdump / c++filt not available")
    out = subprocess.run([CUOBJDUMP, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = counts.setdefault(m.group(1), collections.Counter())
        elif cur is not None:
            for a, b in MNEMONICS.findall(line):
                cur[a or b] += 1
    names = list(counts)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {re.sub(r"\(.*", "", d).replace("void csvit::", ""): counts[n] for n, d in zip(names, dem)}


def _kernels(counts, prefix):
    ks = {k: c for k, c in counts.items() if k.startswith(prefix)}
    assert ks, f"no kernel named {prefix}* in the library"
    return ks


def test_gemm_engine_is_tcgen05_with_tma_and_reductions(sass_counts):
    for name, c in _kernels(sass_counts, "gemm_pair_kernel").items():
        assert c["UTCHMMA"] and c["UTMALDG"] and c["UTMASTG"] and c["LDTM"] and not c["HMMA"], (name, dict(c))
    eight = {k: c for k, c in _kernels(sass_counts, "gemm_pair_kernel").items() if k.endswith(", 8>")}
    assert eight and all(c["UTMAREDG"] and c["REDG"] for c in eight.values()), "in-place residual reductions missing from the pair kernel"
    for name, c in _kernels(sass_counts, "gemm_tc_kernel").items():
        assert c["UTCHMMA"] and c["UTMALDG"] and c["UTMAREDG"] and not c["HMMA"], (name, dict(c))
    for name, c in _kernels(sass_counts, "mlp_fused_kernel").items():
        assert c["UTCHMMA"] and c["UTMALDG"] and c["UTMAREDG"] and not c["HMMA"], (name, dict(c))


def test_swin_forward_attention_has_no_legacy_mma(sass_counts):
    for prefix in ("swin_attn_core_kernel", "swin_attn_fused_kernel", "swinv2_attn_tc_kernel"):
        for name, c in _kernels(sass_counts, prefix).items():
            assert c["UTCHMMA"] and c["LDTM"] and not c["HMMA"], (name, dict(c))
