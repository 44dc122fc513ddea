"""FP8 inference mode of the SwinV2 backbone (``precision="fp8"``): E4M3 Q/K/V and fc1 GEMMs with per-token and per-channel scales.

* GEMM: ``ops.linear_fp8`` / ``ops.swinv2_qkv_fp8`` against the fp64 matmul of the dequantised operands (exactly representable), at
  every SwinV2-B / SwinV2-T stage's Q/K/V and fc1 shape and batch 3, 32 and 256 (both GEMM kernels, ragged M, K = 96 ... 1024).
* ``layernorm_post`` E4M3 copy: copy and row scales bit-identical to the torch expression, fp32 out bit-identical to the 16-bit call.
* Backbone: error against the fp32 mode within 1.25 x that of an fp32 emulation of the fp8 mode (the oracle restatement with the same
  quantisation of the Q/K/V and fc1 operands) + 1e-3.
* Poser and streams: finite, graphed == eager, and both streaming sessions bit-identical to fp8 ``predict_batch``.
Outputs are NaN-filled before every kernel (``torch.use_deterministic_algorithms``) and must end finite.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

E4M3_MAX = 448.0


@pytest.fixture(autouse=True)
def _nan_fill():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)      # torch.empty is NaN-filled
    yield
    torch.use_deterministic_algorithms(prev)


def rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def quant_rows(x: torch.Tensor):
    """Per-row E4M3 quantisation, the formula of layernorm_post's fp8 copy: (copy, scale).  Both divisions are tensor by tensor: torch
    turns a division by a Python scalar into a multiplication by its reciprocal, and ``448 / t`` into ``448 * t.reciprocal()``, neither of
    which is the correctly rounded quotient the kernel computes."""
    amax = x.abs().amax(dim=1)
    m = torch.full_like(amax, E4M3_MAX)
    scale = amax / m
    q = x * (m / torch.where(amax > 0, amax, torch.ones_like(amax)))[:, None]
    q = torch.where(amax[:, None] > 0, q, torch.zeros_like(q)).to(torch.float8_e4m3fn)
    return q, scale


# ---------------------------------------------------------------------------------------------------- GEMM
STAGE_C = {"swinv2_b": (128, 256, 512, 1024), "swinv2_t": (96, 192, 384, 768)}
TOKENS = (4096, 1024, 256, 64)        # per image and stage at 256^2
GEMM_CASES = [(v, s, B, kind) for v in STAGE_C for s in range(4) for B in (3, 32, 256) for kind in ("qkv", "fc1")]


def _operands(M, N, K, seed):
    from cs_vit import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    # rows of different magnitudes (a spread of ~200x at 1M rows, within the fp16 range of the outputs) and one all-zero row
    x = torch.randn(M, K, device="cuda", generator=g) * torch.exp(torch.randn(M, 1, device="cuda", generator=g))
    x[min(5, M - 1)] = 0.0
    a8, rs = quant_rows(x)
    w = 0.05 * torch.randn(N, K, device="cuda", generator=g)
    w8, cs = ops.quantize_weight_fp8(w)
    bias = 0.1 * torch.randn(N, device="cuda", generator=g)
    acc = (a8.double() * rs.double()[:, None]) @ (w8.double() * cs.double()[:, None]).t()     # exact: the dequantised operands
    return a8, rs, w8, cs, bias, acc


@pytest.mark.parametrize("variant,stage,B,kind", GEMM_CASES)
def test_fp8_gemm_matches_fp64(variant, stage, B, kind):
    from cs_vit import ops
    C = STAGE_C[variant][stage]
    M, K = B * TOKENS[stage], C
    N = 3 * C if kind == "qkv" else 4 * C
    a8, rs, w8, cs, bias, acc = _operands(M, N, K, seed=1000 * stage + B)
    if kind == "qkv":
        bias[C:2 * C] = 0.0                   # no key bias (V2:414)
    ref = acc + bias.double()
    if kind == "qkv":
        heads = C // 32
        qs = (1.4426950408889634 * torch.exp(torch.rand(heads, device="cuda"))).float().contiguous()
        got = ops.swinv2_qkv_fp8(a8, rs, w8, cs, bias, qs, out_dtype=torch.float16)
        h = ref.view(M, 3, heads, 32)
        n = h[:, :2] / h[:, :2].norm(dim=-1, keepdim=True).clamp_min(1e-12)
        want = torch.cat([n[:, :1] * qs.double()[None, None, :, None], n[:, 1:2], h[:, 2:]], 1).reshape(M, N)
        assert torch.isfinite(got).all()
        assert rel(got, want) <= 1e-3, rel(got, want)
        plain = ops.linear_fp8(a8, rs, w8, cs, bias, out_dtype=torch.float32)      # the same GEMM, fp32 output, plain epilogue
        assert torch.isfinite(plain).all()
        assert rel(plain, ref) <= 1e-5, rel(plain, ref)
    else:
        got = ops.linear_fp8(a8, rs, w8, cs, bias, act=ops.ACT_GELU, out_dtype=torch.float16)
        want = 0.5 * ref * (1.0 + torch.erf(ref / math.sqrt(2.0)))
        assert torch.isfinite(got).all()
        assert rel(got, want) <= 1e-3, rel(got, want)


def test_fp8_ops_reject_bad_operands():
    from cs_vit import ops
    a8, rs, w8, cs, bias, _ = _operands(64, 96, 64, seed=1)
    with pytest.raises(ValueError, match="float8"):
        ops.linear_fp8(a8.view(torch.uint8), rs, w8, cs)
    with pytest.raises(ValueError, match="scale"):
        ops.linear_fp8(a8, rs[:-1], w8, cs)
    with pytest.raises(ValueError, match="multiples of 16"):
        ops.linear_fp8(a8[:, :40], rs, w8[:, :40], cs)
    with pytest.raises(ValueError):
        ops.layernorm_post(torch.zeros(64, 64, device="cuda"), None, torch.ones(64, device="cuda"), torch.zeros(64, device="cuda"), 1e-5,
                           copy_mode=ops.COPY_MERGE2X2, copy_dtype=torch.float8_e4m3fn, geom=(8, 8, 1, 0))


# ---------------------------------------------------------------------------------------------------- layernorm_post copy
@pytest.mark.parametrize("C", [96, 128, 256, 512, 1024])
@pytest.mark.parametrize("mode", ["identity", "window"])
@pytest.mark.parametrize("with_resid", [False, True])
def test_layernorm_post_fp8_copy_is_bit_exact(C, mode, with_resid):
    from cs_vit import ops
    B, H, ws, shift = 2, 16, 8, 4
    rows = B * H * H
    g = torch.Generator(device="cuda").manual_seed(C + (7 if with_resid else 0))
    y = torch.randn(rows, C, device="cuda", generator=g) * 3.0
    gamma = 1.0 + 0.5 * torch.randn(C, device="cuda", generator=g)
    beta = 0.2 * torch.randn(C, device="cuda", generator=g)
    resid = 4.0 * torch.randn(rows, C, device="cuda", generator=g) if with_resid else None
    y[7] = 1.5                                # constant row: LN(y) = beta exactly; made an all-zero out row below
    if with_resid:
        resid[7] = -beta
    else:
        beta.zero_()
    cm = ops.COPY_IDENTITY if mode == "identity" else ops.COPY_WINDOW
    geom = (H, H, ws, shift) if mode == "window" else (0, 0, 0, 0)
    out, (copy, row_scale) = ops.layernorm_post(y, None if resid is None else resid.clone(), gamma, beta, 1e-5, copy_mode=cm,
                                                copy_dtype=torch.float8_e4m3fn, geom=geom)
    out16, copy16 = ops.layernorm_post(y, None if resid is None else resid.clone(), gamma, beta, 1e-5, copy_mode=cm,
                                       copy_dtype=torch.float16, geom=geom)
    assert torch.equal(out, out16), "the fp32 out must not depend on the copy format"
    assert (out[7] == 0).all()
    want_copy, want_scale = quant_rows(out)
    if mode == "window":
        idx = ops.window_index_map(H, H, ws, shift).long()
        want_copy = want_copy.view(B, H * H, C)[:, idx].reshape(rows, C)
        want_scale = want_scale.view(B, H * H)[:, idx].reshape(rows)
    assert torch.equal(copy.view(torch.uint8), want_copy.view(torch.uint8))
    assert torch.equal(row_scale, want_scale)
    assert torch.isfinite(row_scale).all() and torch.isfinite(copy.float()).all()
    assert (row_scale == 0).sum().item() == 1


# ---------------------------------------------------------------------------------------------------- backbone accuracy
def _emulated_forward(sd, px, depths, heads, window, return_stages=False):
    """The oracle restatement in fp32 with the fp8 mode's quantisation: the Q/K/V input (window order) and the fc1 input per row, the
    Q/K/V and fc1 weights per output channel.  Everything else stays exact fp32 (on CUDA tensors: with TF32 off)."""
    from cs_vit import ops
    from oracle import swinv2_restated as v2

    def deq_rows(x):
        shp = x.shape
        q, s = quant_rows(x.reshape(-1, shp[-1]))
        return (q.float() * s[:, None]).reshape(shp)

    def deq_w(w):
        w8, s = ops.quantize_weight_fp8(w)
        return w8.float() * s[:, None]

    sd = dict(sd)
    for k in list(sd):
        if k.endswith(("self.query.weight", "self.key.weight", "self.value.weight", "intermediate.dense.weight")):
            sd[k] = deq_w(sd[k])
    orig_attn, orig_lin = v2.cosine_window_attention, v2._lin
    v2.cosine_window_attention = lambda xw, *a, **kw: orig_attn(deq_rows(xw), *a, **kw)
    v2._lin = lambda x, sd_, p: orig_lin(deq_rows(x) if p.endswith("intermediate.dense") else x, sd_, p)
    try:
        return v2.swinv2_forward(px, sd, depths, heads, window=window, return_stages=return_stages)
    finally:
        v2.cosine_window_attention, v2._lin = orig_attn, orig_lin


# Measured on one B200 (1000 W): error against the fp32 mode, fp8 GPU vs its fp32 emulation (fp16 mode on swinv2_t_w16: 1.0e-3)
@pytest.mark.parametrize("name,attn8", [("swinv2_t_w16", False), ("swinv2_xs_w8", False), ("swinv2_xs_w8", True)])
def test_fp8_backbone_accuracy(name, attn8, tmp_path):
    from cs_vit.net.swinv2_b200 import load_backbone
    from cs_vit.synthetic import SWINV2_VARIANTS, make_random_backbone_dir
    from oracle import swinv2_restated as v2
    from test_swinv2_oracle import v2_case
    sd, px, _, case = v2_case(name)
    _, depths, heads = SWINV2_VARIANTS[case["variant"]]
    d = make_random_backbone_dir(str(tmp_path / name), case["variant"], seed=case["weight_seed"], image_size=case["image_size"],
                                 window_size=case["window"])
    model = load_backbone(d, precision="fp32").cuda()
    model._v2_tcgen05_8 = attn8
    out = {}
    with torch.no_grad():
        for prec in ("fp32", "fp16", "fp8"):
            model.precision = prec
            out[prec] = model.forward_features(px.cuda(), normalize=False).cpu()
        exact = v2.swinv2_forward(px, sd, depths, heads, window=case["window"])
        emu = _emulated_forward(sd, px, depths, heads, case["window"])
    assert torch.isfinite(out["fp8"]).all()
    err8, err16, err_emu = rel(out["fp8"], out["fp32"]), rel(out["fp16"], out["fp32"]), rel(emu, exact)
    print(f"{name} attn8={attn8}: fp8 {err8:.3e}  emulation {err_emu:.3e}  fp16 {err16:.3e}  (against the fp32 mode)")
    assert err8 <= 1.25 * err_emu + 1e-3


# ---------------------------------------------------------------------------------------------------- Poser and streams
@pytest.mark.parametrize("layer_type", ["encoder", "decoder"])
def test_fp8_poser_graphed_equals_eager(layer_type):
    from cs_vit.graph import KEYS, GraphedPredict
    from cs_vit.synthetic import make_inputs
    import test_stream_gpu as ts
    model = ts._realtime_poser("swinv2_xs", 256, layer_type, "fp8").cuda()
    inp = {k: v.cuda() for k, v in make_inputs(2, 3, 256, seed=11).items()}
    with torch.no_grad():
        eager = model.predict_batch(*(inp[k] for k in KEYS))
    graphed = GraphedPredict(model, inp)(*(inp[k] for k in KEYS))
    for k, v in eager.items():
        assert torch.isfinite(v.float()).all(), k
        assert torch.equal(v, graphed[k]), k


@pytest.mark.parametrize("layer_type", ["encoder", "decoder"])
def test_fp8_realtime_stream_matches_predict_batch(layer_type):
    import test_stream_gpu as ts
    ts.test_stream_matches_predict_batch("swinv2_xs", 256, layer_type, "fp8")


@pytest.mark.parametrize("layer_type", ["encoder", "decoder"])
def test_fp8_full_stream_matches_predict_batch(layer_type):
    import test_stream_full_gpu as tf
    tf.test_full_stream_matches_predict_batch("swinv2_xs", 256, layer_type, "fp8")


def test_fp8_refusals(tmp_path):
    import test_stream_gpu as ts
    from cs_vit.synthetic import make_inputs
    with pytest.raises(ValueError, match="swinv2 backbone only"):
        ts._realtime_poser("swin_xs", 224, "encoder", "fp8")
    model = ts._realtime_poser("swinv2_xs", 256, "encoder", "fp8").cuda()
    imgs = make_inputs(1, 1, 256, seed=2)["patches"].reshape(-1, 3, 256, 256).cuda()
    model.backbone.requires_grad_(True)
    with pytest.raises(ValueError, match="inference only"):
        model.backbone.forward_features(imgs, normalize=True).sum().backward()
