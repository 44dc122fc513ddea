"""``autograd.Swinv2BlockFn`` (the CSVIT_V2_TRAIN_BLOCK=fused path) at SwinV2-B widths and batch, checked one quantity at a time.

Each case runs one block three ways on identical inputs: an fp64 restatement of ``Swinv2Layer`` (the truth), the same restatement on fp32
copies under ``torch.autocast`` (a plain PyTorch mixed-precision block: the comparator), and the block Function with the logit-scale and
bias tables built by ``swinv2_b200._attn_tables_log2``, as the backbone builds them.  Against the truth, the block's error must stay within
1.5x the comparator's for the output, ``dx`` and the gradient of every parameter, and in the worst (image, window) block of rows of the
output and ``dx`` (``logit_scale`` is compared with a variant that rounds its gradient where the kernels do, see the note at
``LOGIT_SCALE``).  The block runs with uninitialised allocations filled with NaN, so an element a kernel never writes cannot pass.
The restatement is pinned to ``oracle.swinv2_layer`` in fp64 on the CPU."""
import contextlib
import math
import time
import warnings

import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu

EPS = 1e-5
KEEP = 0.9                      # stochastic-depth keep probability of the drop-path cases
LN100 = math.log(100.0)
LOGIT_SCALE = "attention.self.logit_scale"
# logit_scale has its own comparator.  Its gradient is sum over (i, j) of dS_ij cos_ij, which cancels heavily because every row of the
# softmax gradient dS sums to zero.  The kernels round dq2 = dS k_hat to 16 bits and only then reduce q_hat . dq2
# (csvit_swinv2_cosnorm_bwd).  The plain comparator multiplies the scale into the fp32 scores, so it reduces dS cos without that rounding.
# Measured on a B200 (1000 W), fp16, w16 stage 0, shift 0, batch 3: e_blk 1.85e-3 against e_cmp 8.9e-4 (ratio 2.07).  The same restatement
# with the scale folded into q_hat before the q k^T product rounds that gradient where the kernels do: e_cmp 1.88e-3 (ratio 0.98).  Over all
# 30 cases the block's logit_scale error is 1.2-4.1e-3 in fp16 and 7e-3-3.4e-2 in bf16.  Against the folded comparator, the largest ratio is
# 1.42 (w8 stage 0, shift 4, bf16).  Against the plain one it is 2.07 in the case above and at most 1.27 in the rest.  So logit_scale is held
# to 1.5x the folded comparator; every other quantity is held to 1.5x the plain one.


# ---------------------------------------------------------------------------------------------------- the fp64 restatement


def _maps(H, ws, shift, device):
    """The oracle's index helpers (oracle/swin_restated.py, oracle/swinv2_restated.py), moved to ``device``."""
    from oracle.swin_restated import relative_position_index, shift_attention_mask, window_gather_index
    from oracle.swinv2_restated import relative_coords_table
    gather = window_gather_index(H, H, ws, shift)          # token read by (window, slot) after roll(-shift) + window_partition
    return {"gather": gather.to(device), "inv": torch.argsort(gather).to(device), "rel": relative_position_index(ws).reshape(-1).to(device),
            "mask": shift_attention_mask(H, H, ws, shift).to(device) if shift else None, "coords": relative_coords_table(ws).to(device)}


def _layer(x, p, m, B, H, heads, ws, s_a=None, s_m=None, fold_scale=False):
    """One Swinv2Layer (V2:662-715: cosine attention with continuous position bias, the shift mask added twice, res-post-norm) on the
    token-ordered ``x [B*H*H, C]``; ``p``: parameters by ``_BlockParamsV2`` name; ``s_a`` / ``s_m``: ``[B]`` stochastic-depth scales of the
    attention and MLP branches, or None.  Written without dtype casts, so it runs in fp64 as is and in mixed precision under autocast.
    ``fold_scale``: multiply the logit scale into q_hat before the q k^T product (as the kernels do) instead of into the scores (as HF does);
    under autocast the gradient of the scaled q is then rounded to 16 bits before the logit-scale reduction, where the kernels round it."""
    N, L = H * H, ws * ws
    nW, C = N // L, x.shape[1]
    d = C // heads
    xw = x.view(B, N, C)[:, m["gather"]].reshape(B * nW, L, C)

    def split(t):
        return t.reshape(B * nW, L, heads, d).transpose(1, 2)

    q = split(F.linear(xw, p["attention.self.query.weight"], p["attention.self.query.bias"]))
    k = split(F.linear(xw, p["attention.self.key.weight"]))
    v = split(F.linear(xw, p["attention.self.value.weight"], p["attention.self.value.bias"]))
    scale = torch.clamp(p["attention.self.logit_scale"], max=LN100).exp()
    if fold_scale:
        s = (F.normalize(q, dim=-1) * scale) @ F.normalize(k, dim=-1).transpose(-2, -1)
    else:
        s = (F.normalize(q, dim=-1) @ F.normalize(k, dim=-1).transpose(-2, -1)) * scale
    hid = F.relu(F.linear(m["coords"].to(x.dtype), p["attention.self.continuous_position_bias_mlp.0.weight"],
                          p["attention.self.continuous_position_bias_mlp.0.bias"]))
    table = F.linear(hid, p["attention.self.continuous_position_bias_mlp.2.weight"])                         # [(2ws-1)^2, heads]
    s = s + 16 * torch.sigmoid(table[m["rel"]].view(L, L, heads).permute(2, 0, 1))
    if m["mask"] is not None:
        s = (s.view(B, nW, heads, L, L) + 2 * m["mask"][None, :, None]).view(B * nW, heads, L, L)
    ctx = (s.softmax(-1) @ v).transpose(1, 2).reshape(B * nW, L, C)
    ya = F.linear(ctx, p["attention.output.dense.weight"], p["attention.output.dense.bias"]).reshape(B, N, C)[:, m["inv"]]
    a = F.layer_norm(ya, (C,), p["layernorm_before.weight"], p["layernorm_before.bias"], EPS)
    x1 = x.view(B, N, C) + (a if s_a is None else a * s_a.view(B, 1, 1))
    z = F.linear(F.gelu(F.linear(x1, p["intermediate.dense.weight"], p["intermediate.dense.bias"])), p["output.dense.weight"],
                 p["output.dense.bias"])
    b = F.layer_norm(z, (C,), p["layernorm_after.weight"], p["layernorm_after.bias"], EPS)
    return (x1 + (b if s_m is None else b * s_m.view(B, 1, 1))).reshape(B * N, C)


def _block_params(C, heads, seed):
    """A ``_BlockParamsV2`` with seeded weights: Linear weights of std 1 / sqrt(fan_in), random biases / LayerNorm affines / CPB-MLP, and
    logit scales around ln 10 with the last head above ln 100, so that its clamp is active."""
    from cs_vit.net.swinv2_b200 import _BlockParamsV2
    blk = _BlockParamsV2(C, heads, EPS)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, prm in blk.named_parameters():
            r = torch.randn(prm.shape, generator=g)
            if name.endswith("logit_scale"):
                r = math.log(10.0) + 0.3 * r
                r[-1] = math.log(150.0)
            elif name.endswith("continuous_position_bias_mlp.2.weight"):
                r = r * (2.0 / math.sqrt(prm.shape[1]))
            elif name.startswith("layernorm") and name.endswith("weight"):
                r = 1.0 + 0.2 * r
            elif name.endswith("bias"):
                r = 0.2 * r
            elif "continuous_position_bias_mlp" not in name:
                r = r / math.sqrt(prm.shape[1])
            prm.copy_(r)
    return blk


def test_restatement_matches_oracle_swinv2_layer(monkeypatch):
    """CPU, fp64: the restatement above equals ``oracle.swinv2_layer`` (roll / window_partition / mask added twice) to 1e-12."""
    import oracle.swinv2_restated as v2
    coords = v2.relative_coords_table
    monkeypatch.setattr(v2, "relative_coords_table", lambda ws, pws=0: coords(ws, pws).double())     # the oracle builds it in fp32
    B, H, C, heads, ws, shift = 2, 16, 64, 2, 8, 4
    blk = _block_params(C, heads, seed=1)
    sd = {"blk." + n: t.detach().double() for n, t in blk.named_parameters()}
    x = torch.randn(B * H * H, C, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    want = v2.swinv2_layer(x.view(B, H * H, C), sd, "blk", H, H, heads, ws, shift, EPS).reshape(B * H * H, C)
    got = _layer(x, {n: t.detach().double() for n, t in blk.named_parameters()}, _maps(H, ws, shift, "cpu"), B, H, heads, ws)
    assert ((got - want).norm() / want.norm()).item() <= 1e-12


# ---------------------------------------------------------------------------------------------------- the three runs


def _reference(blk, x, g2, m, geom, s_a, s_m, dtype=None, fold_scale=False):
    """(output, dx, {name: gradient}) of :func:`_layer`: in fp64 (``dtype`` None), or on fp32 copies under ``torch.autocast(dtype)``."""
    wd = torch.float64 if dtype is None else torch.float32
    p = {n: t.detach().to(wd).requires_grad_(True) for n, t in blk.named_parameters()}
    xx = x.detach().to(wd).requires_grad_(True)
    sa, sm = (None if s is None else s.to(wd) for s in (s_a, s_m))
    with torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
        out = _layer(xx, p, m, *geom, sa, sm, fold_scale)
    out.backward(g2.to(out.dtype))
    return out.detach().double(), xx.grad.double(), {n: t.grad.double() for n, t in p.items()}


def _block(blk, x, g2, geom, shift, s_a, s_m, act):
    """(output, dx, {name: gradient}) of ``autograd.swinv2_block`` with the backbone's table construction."""
    from cs_vit import autograd as ag
    from cs_vit.net.swinv2_b200 import _attn_tables_log2, relative_coords_table
    B, H, heads, ws = geom
    blk.zero_grad(set_to_none=True)
    xx = x.clone().requires_grad_(True)
    qs, bl2 = _attn_tables_log2(blk.attention.self, relative_coords_table(ws).to(x.device), ws, heads)
    out = ag.swinv2_block(xx, blk, qs, bl2, s_a, s_m, B, H, ws, shift, heads, EPS, act)
    out.backward(g2)
    return out.detach(), xx.grad, {n: t.grad.clone() for n, t in blk.named_parameters()}


@contextlib.contextmanager
def _poisoned():
    """Deterministic mode with ``fill_uninitialized_memory``: every ``torch.empty`` is NaN-filled, so an output element that a kernel
    leaves unwritten reads NaN.  (Warnings about ops without a deterministic implementation are beside the point here.)"""
    was, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            assert torch.utils.deterministic.fill_uninitialized_memory
            assert torch.isnan(torch.empty(4096, device="cuda")).all() and torch.isnan(torch.empty_like(torch.ones(8, device="cuda"))).all()
            yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)


def _rel(a, b):
    return ((a.double() - b).norm() / b.norm().clamp_min(1e-300)).item()


def _worst_window(got, want, B, H, ws, gather):
    """max over (image, window) of the relative error of that window's rows of the token-ordered ``[B*H*H, C]`` tensors."""
    C, L = want.shape[1], ws * ws
    blocks = lambda t: t.view(B, H * H, C)[:, gather].reshape(B, -1, L * C)      # noqa: E731
    num = blocks(got.double() - want).norm(dim=-1)
    return (num / blocks(want).norm(dim=-1).clamp_min(1e-300)).max().item()


def _fc1_dgrad_splits_k(rows, C):
    """Whether ``csvit_gemm_ex`` splits K in the block backward's fc1 input-gradient GEMM (``dh [rows, 4C] . w1 -> fp32 [rows, C]``,
    accumulated onto the gradient).  Mirrors launch_gemm_ex in gemm_ex.cu: 128 x 128 tiles, 64-wide k-blocks, and a split when the tiles
    fill at most half the SMs and there are at least 16 k-blocks, into min(SMs / tiles, k-blocks / 8) parts.  Split-K accumulates with
    atomics, so only an unsplit GEMM gives a bit-reproducible ``dx``."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = -(-rows // 128) * -(-C // 128)
    num_kb = -(-4 * C // 64)
    return tiles * 2 <= sms and num_kb >= 16 and min(sms // tiles, num_kb // 8) > 1


# ---------------------------------------------------------------------------------------------------- cases

# (checkpoint, stage, H, C, heads, ws, shift, batch, drop-path): SwinV2-B at 256^2 (embed 128, heads 4-32, window 16 or 8).  Batch 32 is the
# benchmarked batch; batch 3 gives the 8 x 8 core an odd window count at stage 3 (one window per image), so its last 128-row tile is half
# filled.  Batch 32 at stages 0 and 2 sends fc1 (N = 512 / 2048) to the CTA-pair GEMM.
CASES = [
    ("w16", 0, 64, 128, 4, 16, 0, 3, False),
    ("w16", 0, 64, 128, 4, 16, 8, 3, False),
    ("w16", 0, 64, 128, 4, 16, 8, 32, False),
    ("w16", 1, 32, 256, 8, 16, 0, 3, False),
    ("w16", 1, 32, 256, 8, 16, 8, 3, False),
    ("w16", 2, 16, 512, 16, 16, 0, 3, False),
    ("w16", 2, 16, 512, 16, 16, 0, 32, False),
    ("w16", 3, 8, 1024, 32, 8, 0, 3, False),
    ("w16", 3, 8, 1024, 32, 8, 0, 32, False),
    ("w8", 0, 64, 128, 4, 8, 0, 3, False),
    ("w8", 0, 64, 128, 4, 8, 4, 3, False),
    ("w8", 1, 32, 256, 8, 8, 4, 3, False),
    ("w8", 2, 16, 512, 16, 8, 4, 3, False),
    ("w16", 1, 32, 256, 8, 16, 8, 4, True),
    ("w8", 1, 32, 256, 8, 8, 4, 4, True),
]


def _case_id(c):
    ck, st, H, C, heads, ws, shift, B, dp = c
    return f"{ck}-stage{st}-ws{ws}-shift{shift}-b{B}" + ("-droppath" if dp else "")


def _drop_scales(B, device):
    """floor(keep + u) / keep per sample and branch: sample 0 dropped on the attention branch only, 1 on the MLP branch only, 2 on both,
    the rest kept (scaled by 1 / keep)."""
    u_a = torch.full((B,), 0.5)
    u_m = torch.full((B,), 0.5)
    u_a[0], u_m[1], u_a[2], u_m[2] = 0.03, 0.07, 0.01, 0.05
    return tuple((torch.floor(KEEP + u) / KEEP).to(device) for u in (u_a, u_m))


@gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_block_fn_against_fp64_swinv2_layer(case, dtype):
    """Per quantity (output, dx, every parameter's gradient): e_blk <= 1.5 e_cmp + 1e-5 against the fp64 truth, and the same bound on the
    worst (image, window) of the output and dx.  Run with NaN-filled allocations: everything finite.  Exact identities: a sample dropped on
    both branches passes x and g2 through unchanged, the clamped head's logit_scale gradient is 0, the forward is bit-reproducible, and so
    is dx when fc1's input-gradient GEMM does not split K.  At batch 32 of stages 0 and 2 the forward reaches the CTA-pair GEMM."""
    from cs_vit import ops
    ck, stage, H, C, heads, ws, shift, B, drop_path = case
    dev = torch.device("cuda")
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    blk = _block_params(C, heads, seed=1000 * stage + 10 * ws + shift + B).to(dev)
    g = torch.Generator(device=dev).manual_seed(7 + H + shift + B)
    x = torch.randn(B * H * H, C, device=dev, generator=g)
    g2 = torch.randn(B * H * H, C, device=dev, generator=g)
    s_a, s_m = _drop_scales(B, dev) if drop_path else (None, None)
    m = _maps(H, ws, shift, dev)
    geom = (B, H, heads, ws)

    truth = _reference(blk, x, g2, m, geom, s_a, s_m)
    cmp_ = _reference(blk, x, g2, m, geom, s_a, s_m, dtype)
    cmp_fold = _reference(blk, x, g2, m, geom, s_a, s_m, dtype, fold_scale=True)[2][LOGIT_SCALE]
    with _poisoned():
        out, dx, grads = _block(blk, x, g2, geom, shift, s_a, s_m, dtype)
        torch.cuda.synchronize()
    profile = (B == 32 and stage in (0, 2))
    if profile:
        ops.begin_profile("csvit_linear")
    try:
        out2, dx2, _ = _block(blk, x, g2, geom, shift, s_a, s_m, dtype)
    finally:
        prof = ops.end_profile() if profile else None

    failures = []
    names = ["output", "dx"] + list(grads)
    got = dict(output=out, dx=dx, **grads)
    want = dict(output=truth[0], dx=truth[1], **truth[2])
    cmpd = dict(output=cmp_[0], dx=cmp_[1], **cmp_[2])
    nonfinite = [n for n in names if not torch.isfinite(got[n]).all()]
    if nonfinite:
        rows = torch.nonzero(~torch.isfinite(dx).all(dim=1)).flatten()[:8].tolist() if "dx" in nonfinite else []
        failures.append(f"non-finite with NaN-filled allocations: {nonfinite} (first dx rows: {rows})")
    lines = [f"{_case_id(case)} {str(dtype)[6:]}", f"  {'quantity':<56} {'e_blk':>10} {'e_cmp':>10} {'ratio':>7}"]
    for n in names:
        eb, ec = _rel(got[n], want[n]), _rel(cmpd[n], want[n])
        lines.append(f"  {n:<56} {eb:10.3e} {ec:10.3e} {eb / max(ec, 1e-300):7.2f}")
        if n == LOGIT_SCALE:        # its own comparator: see the note at LOGIT_SCALE
            ec = _rel(cmp_fold, want[n])
            lines.append(f"  {n + ' (comparator, folded scale)':<56} {eb:10.3e} {ec:10.3e} {eb / max(ec, 1e-300):7.2f}")
        if not eb <= 1.5 * ec + 1e-5:
            failures.append(f"{n}: e_blk {eb:.3e} > 1.5 e_cmp {ec:.3e} + 1e-5")
    for n in ("output", "dx"):
        wb = _worst_window(got[n], want[n], B, H, ws, m["gather"])
        wc = _worst_window(cmpd[n], want[n], B, H, ws, m["gather"])
        lines.append(f"  {'worst window of ' + n:<56} {wb:10.3e} {wc:10.3e} {wb / max(wc, 1e-300):7.2f}")
        if not wb <= 1.5 * wc + 1e-5:
            failures.append(f"worst window of {n}: e_blk {wb:.3e} > 1.5 e_cmp {wc:.3e} + 1e-5")

    if drop_path:
        N = H * H
        both = [b for b in range(B) if s_a[b].item() == 0.0 and s_m[b].item() == 0.0]
        assert both, "the drop-path case must drop one sample on both branches"
        for b in both:
            r = slice(b * N, (b + 1) * N)
            if not torch.equal(out[r], x[r]):
                failures.append(f"sample {b} dropped on both branches: output rows differ from x")
            if not torch.equal(dx[r], g2[r]):
                failures.append(f"sample {b} dropped on both branches: dx rows differ from g2")
    ls = grads[LOGIT_SCALE].flatten()
    if ls[-1].item() != 0.0:
        failures.append(f"clamped head's logit_scale gradient {ls[-1].item()!r} != 0")
    if not torch.equal(out, out2):
        failures.append("forward output differs between two calls")
    split = _fc1_dgrad_splits_k(B * H * H, C)
    if not split and not torch.equal(dx, dx2):
        failures.append("dx differs between two calls although no GEMM on its path splits K")
    if profile and "kind1" not in prof:
        failures.append(f"no csvit_linear call took the CTA-pair kernel (kind 1): {sorted(k for k in prof if k.startswith('kind'))}")

    lines.append(f"  fc1 dgrad split-K: {split}; CTA-pair launches: {prof['kind1']['launches'] if prof and 'kind1' in prof else '-'}; "
                 f"peak memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB; {time.time() - t0:.1f} s")
    print("\n" + "\n".join(lines))
    assert not failures, "\n".join(failures)


# ---------------------------------------------------------------------------------------------------- row_scale_add


@gpu
@pytest.mark.parametrize("with_x", [True, False], ids=["x", "no-x"])
@pytest.mark.parametrize("rows,C,group_rows", [(37, 20, 1), (192, 36, 64), (768, 132, 256), (3 * 4096, 1024, 4096)])
def test_row_scale_add_matches_fp64(rows, C, group_rows, with_x):
    """``x + s[row // group_rows] * y`` against fp64: one fmaf per element, so within half an fp32 ulp, and exactly ``x`` (or 0) where the
    scale is 0.  185 and 1728 float4s are not a multiple of one 256-thread block; 3 x 4096 rows of 1024 take the capped grid's
    grid-stride loop.  NaN-filled allocations: every element of the output must be written."""
    from cs_vit import ops
    g = torch.Generator(device="cuda").manual_seed(rows + C)
    y = torch.randn(rows, C, device="cuda", generator=g)
    x = torch.randn(rows, C, device="cuda", generator=g) if with_x else None
    u = torch.rand(rows // group_rows, device="cuda", generator=g)
    u[0] = 0.0
    s = (torch.floor(0.8 + u) / 0.8).contiguous()
    with _poisoned():
        got = ops.row_scale_add(x, y, s, group_rows)
        torch.cuda.synchronize()
    sr = s.double().repeat_interleave(group_rows)[:, None]
    want = sr * y.double() + (x.double() if with_x else 0.0)
    assert ((got.double() - want).abs() <= want.abs() * 2.0 ** -24).all()
    dropped = (sr == 0).flatten()
    assert dropped.any()
    assert torch.equal(got[dropped], x[dropped] if with_x else torch.zeros_like(got[dropped]))


@gpu
def test_row_scale_add_rejects_bad_geometry():
    """C % 4 != 0 is refused by the library; rows % group_rows != 0 by ops and, called through the C ABI directly, by the library."""
    from cs_vit import ops
    from cs_vit._lib import CsvitError
    with pytest.raises(CsvitError):
        ops.row_scale_add(None, torch.randn(64, 6, device="cuda"), torch.ones(1, device="cuda"), 64)
    y = torch.randn(100, 8, device="cuda")
    s = torch.ones(2, device="cuda")
    with pytest.raises(ValueError):
        ops.row_scale_add(None, y, s, 64)
    out = torch.empty_like(y)
    with pytest.raises(CsvitError):
        ops._call("csvit_row_scale_add", None, y.data_ptr(), s.data_ptr(), out.data_ptr(), 100, 8, 64, ops._stream())
