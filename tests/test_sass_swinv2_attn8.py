"""CPU check of the built library's machine code for the SwinV2 8 x 8-window attention (`cuobjdump -sass`, no GPU needed): every
instantiation of swinv2_w8_attn_kernel (forward) and swinv2_w8_bwd_kernel (backward) runs on tcgen05 MMAs (`UTCHMMA`) with TMEM loads
(`LDTM`) and TMA tensor loads (`UTMALDG`), and contains no legacy `HMMA` (mma.sync)."""
import pytest

from test_sass import _kernels, sass_counts  # noqa: F401  (module-scoped fixture)


@pytest.mark.parametrize("prefix,count", [("swinv2_w8_attn_kernel", 4), ("swinv2_w8_bwd_kernel", 2)])
def test_swinv2_attention8_is_tcgen05(sass_counts, prefix, count):  # noqa: F811
    kernels = _kernels(sass_counts, prefix)
    assert len(kernels) == count, sorted(kernels)          # {fp16, bf16} (x {inference, training} for the forward)
    for name, c in kernels.items():
        assert c["UTCHMMA"] and c["LDTM"] and c["UTMALDG"] and not c["HMMA"], (name, dict(c))
