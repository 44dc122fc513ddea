"""CPU check of the built library's machine code for the FP8 GEMMs (`cuobjdump -sass`, no GPU needed): every E4M3 instantiation of the
single-CTA and CTA-pair kernels issues 8-bit tcgen05 MMAs (`UTCQMMA`, kind::f8f6f4) with TMA tensor loads (`UTMALDG`), and neither
16-bit tcgen05 MMAs (`UTCHMMA`) nor legacy `HMMA` (mma.sync)."""
import collections
import re
import subprocess

import pytest

from test_sass import CUOBJDUMP, LIB, os, shutil


@pytest.fixture(scope="module")
def qmma_counts():
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
            for mn in re.findall(r"\b(UTCQMMA|UTCHMMA|UTMALDG|LDTM|HMMA)\b", line):
                cur[mn] += 1
    names = list(counts)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {re.sub(r"\(.*", "", d).replace("void csvit::", ""): counts[n] for n, d in zip(names, dem)}


def test_fp8_gemms_are_8bit_tcgen05(qmma_counts):
    fp8 = {k: c for k, c in qmma_counts.items() if k.startswith(("gemm_tc_fp8_kernel", "gemm_pair_fp8_kernel"))}
    assert len(fp8) == 8, sorted(fp8)       # single CTA: BN 128 / 256 x cluster 1 / 2 / 4; pair: 8 / 16 epilogue warps
    for name, c in fp8.items():
        assert c["UTCQMMA"] and c["UTMALDG"] and c["LDTM"] and not c["UTCHMMA"] and not c["HMMA"], (name, dict(c))
    others = {k: c for k, c in qmma_counts.items() if k not in fp8 and c["UTCQMMA"]}
    assert not others, f"8-bit MMAs outside the fp8 GEMM instantiations: {sorted(others)}"
