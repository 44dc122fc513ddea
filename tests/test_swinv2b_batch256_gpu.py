"""SwinV2-B inference at batch 256, the workload ``bench.py --variant swinv2_b`` times, against an fp64 restatement: image by image,
stage by stage and token by token, in every precision and attention-kernel mode.

At this size the forward takes paths the small goldens never reach: the CTA-pair GEMM (with its 16-warp GELU epilogue at K = 128 / 256,
its tail-split half tiles and the cosine-normalising Q/K/V epilogue), and, at 255 images, an odd 8 x 8 window count, a 64-row last GEMM
tile and a 192-row last CTA-pair row block at stage 3.  One relative error over the whole batch hides a fault in one image (it moves by
about 1/16 of that image's error), so every check here is localized:

* (a) every image's relative error on every stage output (and ``last_hidden_state``) is within the mode's bar;
* (b) the worst image is within ``IMG_SPREAD`` x the median image;
* (c) the worst token (relative row error) is within ``TOK_SPREAD`` x the median token.

The reference is ``oracle/swinv2_restated.py`` in fp64 on the GPU, computed once per checkpoint (window 16 and window 8).  The batch-256
path is also tied to the small-batch path (bit-identical in every mode), and the kernel checks at the end locate a failure
in the pair GEMM's cosine and GELU epilogues.  Outputs are NaN-filled before every kernel (``_nan_fill``) and must end finite.
"""
import math
import os

import pytest
import torch
import torch.nn.functional as F

from helpers import OUT_KEYS
from test_fp8_gpu import _emulated_forward, _nan_fill, rel  # noqa: F401  (_nan_fill: autouse fixture)

VARIANT = "swinv2_b"
BATCH = 256
SLOTS = (0, 37, 100, 101, 128, 200, 254, 255)     # the images of the batch-8 tie and of the fp8 emulation
CHUNK = 16                                        # images per fp64 reference call (stage 0 scores: ~34 MB per image)
STAGE_C = (128, 256, 512, 1024)
TOKENS = (4096, 1024, 256, 64)                    # per image and stage at 256^2
LABELS = ("stage0", "stage1", "stage2", "stage3", "final")

# (a) per-image bars.  Measured on one B200 (1000 W), worst image over every stage output and attention mode of both checkpoints:
# fp32 1.40e-6, fp16 1.26e-3, bf16 8.60e-3 (medians at stage 3: 1.3e-6 / 9.8e-4 / 7.7e-3 at window 16, 1.4e-6 / 1.2e-3 / 8.0e-3 at
# window 8).  fp8 takes its bar from the fp32 emulation of the fp8 mode (_Checkpoint.fp8_bars); measured at stage 3, worst image
# against that bar: 7.9e-2 / 9.8e-2 at window 16, 8.5e-2 / 1.02e-1 at window 8.
BAR = {"fp32": 3e-6, "fp16": 2e-3, "bf16": 1.2e-2}
# (b) worst image / median image, every mode and stage output.  Measured: at most 1.10.
IMG_SPREAD = 1.5
# (c) worst token / median token, per stage output (stage0 .. stage3, last_hidden_state), every mode.  Measured: at most 5.7 (stage 0,
# window 8, fp32; 2.9-5.2 in the other modes), 2.2, 1.4, 1.2, 1.2.
TOK_SPREAD = (8.0, 3.0, 2.0, 2.0, 2.0)

# attention kernels: (16 x 16 windows on tcgen05, 8 x 8 windows on tcgen05); otherwise the mma.sync kernels
ATTN = {"tc16": (True, False), "tc16+tc8": (True, True), "mma": (False, False), "mma8": (True, False), "tc8": (True, True)}
CASES = ([(16, p, a) for p in ("fp16", "bf16", "fp8") for a in ("tc16", "tc16+tc8", "mma")]
         + [(8, p, a) for p in ("fp16", "bf16", "fp8") for a in ("mma8", "tc8")]
         + [(16, "fp32", "tc16"), (8, "fp32", "mma8")])
RAGGED = [(ws, p, a) for ws, a16, a8 in ((16, "tc16", "tc16+tc8"), (8, "mma8", "tc8")) for p, a in (("fp16", a16), ("fp16", a8), ("fp8", a16))]


def _case_id(c):
    return f"w{c[0]}-{c[1]}-{c[2]}"


class _Checkpoint:
    """One random SwinV2-B backbone at 256^2, the model on the GPU, and the fp64 restatement of the 256 images through it."""

    def __init__(self, ws: int, root: str, images: torch.Tensor):
        from cs_vit.net.swinv2_b200 import load_backbone
        from cs_vit.synthetic import SWINV2_VARIANTS, make_random_backbone_dir
        from oracle import swinv2_restated as v2
        _, self.depths, self.heads = SWINV2_VARIANTS[VARIANT]
        self.ws = ws
        self.dir = make_random_backbone_dir(os.path.join(root, f"w{ws}"), VARIANT, seed=0 if ws == 16 else 1, image_size=256, window_size=ws)
        self.model = load_backbone(self.dir, precision="fp32").cuda()
        self.sd32 = {k: v.detach() for k, v in self.model.state_dict().items()}
        sd64 = {k: v.double() for k, v in self.sd32.items()}
        n = images.shape[0]
        self.stages = [torch.empty(n, t, c, dtype=torch.float64, device="cuda") for t, c in zip(TOKENS, STAGE_C)]
        self.final = torch.empty(n, TOKENS[3], STAGE_C[3], dtype=torch.float64, device="cuda")
        with torch.no_grad():
            for i in range(0, n, CHUNK):
                out, st = v2.swinv2_forward(images[i:i + CHUNK].double(), sd64, self.depths, self.heads, window=ws, return_stages=True)
                for s, t in enumerate(st):
                    self.stages[s][i:i + CHUNK] = t
                self.final[i:i + CHUNK] = out
        self.emu_bar = None

    def outputs(self):
        return self.stages + [self.final]

    def run(self, precision: str, attn: str, images: torch.Tensor):
        """forward_features at the given precision and attention kernels -> [stage0..stage3, last_hidden_state], fp32."""
        m = self.model
        m.precision = precision
        m._v2_tcgen05, m._v2_tcgen05_8 = ATTN[attn]
        with torch.no_grad():
            out, stages = m.forward_features(images, normalize=False, return_stages=True)
        return list(stages) + [out]

    def fp8_bars(self, images: torch.Tensor):
        """Per-output bars of the fp8 mode, as in test_fp8_backbone_accuracy: 1.25 x the error of the fp32 emulation of the fp8 mode (run on
        the SLOTS images, worst of them, against the fp64 reference) + 1e-3."""
        if self.emu_bar is None:
            slots = torch.tensor(SLOTS, device="cuda")
            with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
                assert not torch.backends.cuda.matmul.allow_tf32
                out, st = _emulated_forward(self.sd32, images[slots], self.depths, self.heads, self.ws, return_stages=True)
            emu = [image_errors(g, r[slots]) for g, r in zip(list(st) + [out], self.outputs())]
            print(f"w{self.ws} fp32 emulation of fp8, worst of {len(SLOTS)} images: " + "  ".join(f"{l} {e.max():.3e}" for l, e in zip(LABELS, emu)))
            self.emu_bar = [1.25 * e.max().item() + 1e-3 for e in emu]
        return self.emu_bar


@pytest.fixture(scope="module")
def images():
    g = torch.Generator().manual_seed(256)
    return torch.randn(BATCH, 3, 256, 256, generator=g).cuda()


@pytest.fixture(scope="module")
def ckpt(images, tmp_path_factory):
    cache = {}

    def get(ws: int) -> _Checkpoint:
        if ws not in cache:
            cache[ws] = _Checkpoint(ws, str(tmp_path_factory.mktemp("swinv2b")), images)
        return cache[ws]
    return get


# ---------------------------------------------------------------------------------------------------- localized metrics
def image_errors(got: torch.Tensor, ref: torch.Tensor) -> torch.Tensor:
    """[n, tokens, C] -> [n] relative error of each image."""
    d = got.double() - ref
    return d.flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1)


def token_errors(got: torch.Tensor, ref: torch.Tensor) -> torch.Tensor:
    """[n, tokens, C] -> [n, tokens] relative error of each token (row norm)."""
    return (got.double() - ref).norm(dim=-1) / ref.norm(dim=-1)


def check_localized(got, ref, rows, bars, what):
    """(a), (b), (c) on every output of one run; ``rows`` picks the reference images the outputs belong to."""
    for label, g, r, bar, tok_spread in zip(LABELS, got, ref, bars, TOK_SPREAD):
        r = r[rows]
        assert torch.isfinite(g).all(), f"{what} {label}: non-finite output"
        img, tok = image_errors(g, r), token_errors(g, r)
        i_med, i_max, i_arg = img.median().item(), img.max().item(), img.argmax().item()
        t_med, t_max, t_arg = tok.median().item(), tok.max().item(), tok.argmax().item()
        print(f"{what} {label}: image median {i_med:.3e} worst {i_max:.3e} (#{i_arg}), token median {t_med:.3e} worst {t_max:.3e} "
              f"(image {t_arg // tok.shape[1]} token {t_arg % tok.shape[1]}), batch {rel(g, r):.3e}")
        assert i_max <= bar, f"{what} {label}: image {i_arg} error {i_max:.3e} over the bar {bar:.1e}"
        assert i_max <= IMG_SPREAD * i_med, f"{what} {label}: image {i_arg} error {i_max:.3e} > {IMG_SPREAD} x median {i_med:.3e}"
        assert t_max <= tok_spread * t_med, (f"{what} {label}: image {t_arg // tok.shape[1]} token {t_arg % tok.shape[1]} error {t_max:.3e} "
                                             f"> {tok_spread} x median {t_med:.3e}")


def _bars(ck, precision, images):
    return ck.fp8_bars(images) if precision == "fp8" else [BAR[precision]] * len(LABELS)


# ---------------------------------------------------------------------------------------------------- the backbone at batch 256
def test_restatement_runs_in_fp64_on_cpu():
    """The restatement follows its state dict's dtype and device (the batch-256 reference below runs it in fp64 on the GPU): in fp64 on
    CPU tensors it matches the HF goldens of the three SwinV2 cases as closely as the fp32 restatement does."""
    from cs_vit.synthetic import SWINV2_VARIANTS
    from oracle import swinv2_restated as v2
    from test_swinv2_oracle import V2_CASES, v2_case
    for name in sorted(V2_CASES):
        sd, px, gold, case = v2_case(name)
        _, depths, heads = SWINV2_VARIANTS[case["variant"]]
        with torch.no_grad():
            out, stages = v2.swinv2_forward(px.double(), {k: v.double() for k, v in sd.items()}, depths, heads, window=case["window"],
                                            return_stages=True)
        assert out.dtype == torch.float64 and all(t.dtype == torch.float64 for t in stages)
        assert rel(out, torch.from_numpy(gold["last_hidden_state"])) < 2e-6, name
        for s, t in enumerate(stages):
            assert rel(t[:, ::case["stage_token_stride"]], torch.from_numpy(gold[f"stage{s}"])) < 2e-6, (name, s)


@pytest.mark.gpu
@pytest.mark.parametrize("ws,precision,attn", CASES, ids=[_case_id(c) for c in CASES])
def test_batch256_per_image_per_stage(ckpt, images, ws, precision, attn):
    ck = ckpt(ws)
    got = ck.run(precision, attn, images)
    check_localized(got, ck.outputs(), slice(None), _bars(ck, precision, images), _case_id((ws, precision, attn)))


@pytest.mark.gpu
@pytest.mark.parametrize("ws,precision,attn", RAGGED, ids=[_case_id(c) for c in RAGGED])
def test_ragged_batch255(ckpt, images, ws, precision, attn):
    """255 images: an odd 8 x 8 window count at stage 3, a 64-row last GEMM tile and a 192-row last CTA-pair row block there.  Images are
    independent, fp8 scales belong to one token and the pair and single-CTA GEMMs share one accumulation order, so the outputs equal
    rows 0-254 of the batch-256 run bit for bit."""
    ck = ckpt(ws)
    full = ck.run(precision, attn, images)
    got = ck.run(precision, attn, images[:BATCH - 1])
    check_localized(got, ck.outputs(), slice(0, BATCH - 1), _bars(ck, precision, images), "255 images " + _case_id((ws, precision, attn)))
    for label, a, b in zip(LABELS, got, full):
        assert torch.equal(a, b[:BATCH - 1]), f"{label}: batch 255 differs from rows 0-254 of batch 256 ({rel(a, b[:BATCH - 1]):.3e})"


@pytest.mark.gpu
@pytest.mark.parametrize("ws,precision,attn", CASES, ids=[_case_id(c) for c in CASES])
def test_tied_to_batch8(ckpt, images, ws, precision, attn):
    """The SLOTS images (0 and 255 among them) as their own batch of 8 equal their rows of the batch-256 run, bit for bit, in every mode.
    fp32 included: unlike Swin-v1's fused kernels, every SwinV2 fp32 op sums each output element in an order that does not depend on the
    number of rows (the SIMT GEMM runs one 64 x 64 tile per block over the whole K), and measured so on a B200."""
    ck = ckpt(ws)
    slots = torch.tensor(SLOTS, device="cuda")
    full = ck.run(precision, attn, images)
    small = ck.run(precision, attn, images[slots])
    for label, a, b in zip(LABELS, small, full):
        assert torch.equal(a, b[slots]), f"{label}: batch 8 differs from its rows of batch 256 ({rel(a, b[slots]):.3e})"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16", "fp8"])
def test_benched_poser_graphed_batch256_equals_eager_batch8(ckpt, precision):
    """The ``bench.py --variant swinv2_b`` model (encoder head, patch perspective decoration, 256^2, randomised head) replayed as a CUDA
    graph at batch 256 equals eager ``predict_batch`` on the SLOTS images, bit for bit, and is finite."""
    from cs_vit.graph import KEYS, GraphedPredict
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_inputs, randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO
    torch.manual_seed(0)
    model = Poser(ckpt(16).dir, image_size=256, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch",
                  precision=precision, temporal_supervision="full", temporal_init_method="zero")
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.SPATIAL)
    model.eval()
    model = model.cuda()
    dev = {k: v.cuda() for k, v in make_inputs(BATCH, 1, 256, seed=100).items()}
    slots = torch.tensor(SLOTS, device="cuda")
    graphed = {k: v.clone() for k, v in GraphedPredict(model, dev)(*(dev[k] for k in KEYS)).items()}
    with torch.no_grad():
        eager = model.predict_batch(*(dev[k][slots] for k in KEYS))
    for k in OUT_KEYS:
        assert torch.isfinite(graphed[k].float()).all() and torch.isfinite(eager[k].float()).all(), k
        assert torch.equal(graphed[k][slots], eager[k]), (k, rel(graphed[k][slots], eager[k]))


# ---------------------------------------------------------------------------------------------------- kernels at the batch-256 shapes
def _gemm_kernel() -> int:
    """The GEMM kernel the last launch of this thread chose: 1 CTA-pair, 2 single-CTA tcgen05, 3 SIMT."""
    from cs_vit import _lib
    return _lib.load().csvit_last_gemm_kernel()


def _pair_and_single(fn):
    """fn() with the automatic kernel choice (which must be the CTA pair) and with the pair kernel disabled."""
    from cs_vit import ops
    try:
        pair = fn()
        assert _gemm_kernel() == 1, "the CTA-pair kernel was not chosen at this shape"
        ops.set_gemm_tuning(pair=0)
        single = fn()
        assert _gemm_kernel() == 2
    finally:
        ops.set_gemm_tuning()
    return pair, single


UNIT = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}     # unit roundoff of the 16-bit output


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("stage,n_img", [(1, 256), (2, 256), (3, 256), (3, 255)])
def test_swinv2_qkv_pair_kernel_matches_fp64(stage, n_img, dt):
    """``ops.swinv2_qkv`` (F.normalize of every q and k head, q times its scale, v plain, in the GEMM epilogue) at the SwinV2-B Q/K/V shapes
    of batch 256 / 255.  Each 32-column head is one fp32 vector rounded once to 16 bit, so its relative error is at most the unit roundoff:
    checked head by head on every row.  Row ZERO is all-zero input: its k heads (no key bias) - and, at 255 images, where the q bias is zero
    too, its q heads - have norm 0, which F.normalize maps to 0."""
    from cs_vit import ops
    C = STAGE_C[stage]
    M, K, N, heads = n_img * TOKENS[stage], C, 3 * C, C // 32
    zero = M - 70                         # in the last GEMM tile / CTA-pair row block
    g = torch.Generator(device="cuda").manual_seed(100 * stage + n_img)
    a = torch.randn(M, K, device="cuda", generator=g).to(dt)
    a[zero] = 0
    w = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).to(dt)
    bias = 0.1 * torch.randn(N, device="cuda", generator=g)
    bias[C:2 * C] = 0                     # no key bias (V2:414)
    if n_img == 255:
        bias[:C] = 0
    qs = (1.4426950408889634 * torch.exp(torch.rand(heads, device="cuda", generator=g) * math.log(100.0))).contiguous()
    got, single = _pair_and_single(lambda: ops.swinv2_qkv(a, w, bias, qs))
    assert torch.isfinite(got).all()
    assert torch.equal(got, single), "CTA-pair and single-CTA kernels differ"
    h = (a.double() @ w.double().t() + bias.double()).view(M, 3, heads, 32)
    qk = F.normalize(h[:, :2], dim=-1)
    want = torch.cat([qk[:, :1] * qs.double()[:, None], qk[:, 1:], h[:, 2:]], 1)
    gh = got.double().view(M, 3, heads, 32)
    assert (gh[zero, 1] == 0).all() and (n_img == 256 or (gh[zero, 0] == 0).all()), "zero-norm heads must come out 0"
    norm = want.norm(dim=-1)
    err = (gh - want).norm(dim=-1) / norm.clamp_min(1e-300)
    err[norm == 0] = 0
    worst = err.amax(dim=(0, 2))          # [q, k, v]
    print(f"qkv stage {stage} M={M} {dt}: worst head error q {worst[0]:.3e} k {worst[1]:.3e} v {worst[2]:.3e} (unit roundoff {UNIT[dt]:.3e})")
    assert (worst <= 1.05 * UNIT[dt]).all(), worst.tolist()


def _gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


# Per-row relative error of the packed-fp16 GELU epilogue.  Measured on one B200 (1000 W), worst row of stages 0 and 1: fp16 4.6e-4
# (median 3.4e-4), bf16 2.3e-3 (median 1.7e-3)
GELU_ROW_BAR = {torch.float16: 8e-4, torch.bfloat16: 4e-3}


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("stage", [0, 1])
def test_fc1_gelu_pair_kernel_matches_fp64(stage, dt):
    """fc1 + GELU of SwinV2-B stages 0 / 1 at batch 256 (K = 128 / 256: the CTA-pair kernel's sixteen-warp GELU epilogue), row by row
    against fp64, and bit-identical to the single-CTA kernel."""
    from cs_vit import ops
    C = STAGE_C[stage]
    M, K, N = BATCH * TOKENS[stage], C, 4 * C
    g = torch.Generator(device="cuda").manual_seed(7 + stage)
    a = torch.randn(M, K, device="cuda", generator=g).to(dt)
    w = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).to(dt)
    b = 0.1 * torch.randn(N, device="cuda", generator=g)
    got, single = _pair_and_single(lambda: ops.linear(a, w, b, act=ops.ACT_GELU, out_dtype=dt))
    assert torch.isfinite(got).all()
    assert torch.equal(got, single), "CTA-pair and single-CTA kernels differ"
    errs = []
    for lo in range(0, M, 1 << 17):
        want = _gelu64(a[lo:lo + (1 << 17)].double() @ w.double().t() + b.double())
        errs.append((got[lo:lo + (1 << 17)].double() - want).norm(dim=1) / want.norm(dim=1))
    errs = torch.cat(errs)
    print(f"fc1 GELU stage {stage} M={M} {dt}: row error median {errs.median():.3e} worst {errs.max():.3e} (row {errs.argmax().item()})")
    assert errs.max() <= GELU_ROW_BAR[dt], (errs.max().item(), errs.argmax().item())
