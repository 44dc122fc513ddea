"""CPU check of the built library's machine code for the SwinV2 attention backward (`cuobjdump -sass`, no GPU needed): every
instantiation of swinv2_attn_bwd_kernel runs on tcgen05 MMAs (`UTCHMMA`) with TMEM loads (`LDTM`) and TMA tensor loads (`UTMALDG`),
and contains no legacy `HMMA` (mma.sync)."""
from test_sass import _kernels, sass_counts  # noqa: F401  (module-scoped fixture)


def test_swinv2_attention_backward_is_tcgen05(sass_counts):  # noqa: F811
    kernels = _kernels(sass_counts, "swinv2_attn_bwd_kernel")
    assert len(kernels) == 2, sorted(kernels)              # fp16 and bf16
    for name, c in kernels.items():
        assert c["UTCHMMA"] and c["LDTM"] and c["UTMALDG"] and not c["HMMA"], (name, dict(c))
