"""CPU suite, part 1: the oracle restatement against the golden vectors produced by the live reference
(oracle/make_goldens.py), and the integer logic compiled into the kernels against HF's own maps."""
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, OUT_KEYS, build_product, head_options, manifest, rel

CASES = sorted(manifest()["cases"])


@pytest.mark.parametrize("name", CASES)
def test_restatement_matches_reference_goldens(name):
    from cs_vit.utils.mano_standin import SyntheticMANO
    from oracle import head_restated as head

    model, inputs, gold, case = build_product(name)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    opt = head_options(case)
    with torch.no_grad():
        flat = inputs["patches"].reshape(-1, 3, 224, 224)
        feats = head.backbone_features(flat, sd, opt)
        assert rel(feats, gold["features"]) < 1e-5
        # the head from the reference's own features: the backbone's fp32 round-off depends on the host (thread count, vector
        # ISA), and the decoder-query heads amplify a 2e-7 feature difference about 50x in the outputs
        ref_feats = torch.from_numpy(gold["features"])
        out = head.predict_batch(inputs, sd, opt, SyntheticMANO(), features_fn=lambda x: ref_feats, execute_all=False)
    for k in OUT_KEYS:
        assert out[k].shape == gold[k].shape
        assert rel(out[k], gold[k]) < 2e-5, (name, k, rel(out[k], gold[k]))


def test_swin_stage_outputs_match_hf_hidden_states():
    from oracle import head_restated as head
    from oracle import swin_restated as swin

    model, inputs, gold, case = build_product("swint_encoder_patch_spatial")
    opt = head_options(case)
    bsd = {k[len("backbone."):]: v.detach() for k, v in model.state_dict().items() if k.startswith("backbone.")}
    mean = torch.tensor(head.IMAGENET_MEAN)[None, :, None, None]
    std = torch.tensor(head.IMAGENET_STD)[None, :, None, None]
    with torch.no_grad():
        px = (inputs["patches"].reshape(-1, 3, 224, 224) - mean) / std
        emb = swin.patch_embed(px, bsd, 1e-5)
        assert rel(emb[:, :8], gold["hidden_0"]) < 1e-5
        _, stages = swin.swin_forward(px, bsd, opt.depths, opt.swin_heads, return_stages=True)
        # HF hidden_states[i+1] is stage i AFTER its patch merging; the last stage has none.
        assert rel(stages[-1][:, :8], gold[f"hidden_{len(stages)}"]) < 1e-5


INTS = dict(np.load(os.path.join(GOLDEN, "integer_maps.npz")))


@pytest.mark.parametrize("H,shift", [(56, 0), (56, 3), (28, 0), (28, 3), (14, 0), (14, 3), (7, 0)])
def test_integer_maps_oracle_and_kernel_host_code_bit_exact(H, shift):
    from cs_vit import ops
    from oracle import swin_restated as swin

    want = torch.from_numpy(INTS[f"gather_{H}_{shift}"])
    assert torch.equal(swin.window_gather_index(H, H, 7, shift).int(), want)
    idx, mask = ops.host_maps(H, H, 7, shift)
    assert torch.equal(idx, want)                                  # gather address == scatter address
    assert sorted(idx.tolist()) == list(range(H * H))              # a permutation: in-place residual is safe
    if shift:
        want_mask = torch.from_numpy(INTS[f"mask_{H}_{shift}"]).float() * -100.0
        assert torch.equal(swin.shift_attention_mask(H, H, 7, shift), want_mask)
        assert torch.equal(mask, want_mask)
    else:
        assert torch.count_nonzero(mask) == 0


def test_rel_index_and_merge_maps_bit_exact():
    from cs_vit import ops
    from oracle import swin_restated as swin

    assert torch.equal(ops.host_rel_pos_index(7), torch.from_numpy(INTS["rel_index_7"]))
    assert torch.equal(swin.relative_position_index(7).int(), torch.from_numpy(INTS["rel_index_7"]))
    for H in (56, 28, 14):
        want = torch.from_numpy(INTS[f"merge_{H}"])
        assert torch.equal(ops.host_merge_index_map(H, H), want)
        assert torch.equal(swin.merge_gather_index(H, H).int(), want)


def test_q2_only_last_encoder_layer_matters():
    """SURVEY Q2: the 'encoder' spatial head returns layers[-1](same input); earlier layers are dead code."""
    from cs_vit.utils.mano_standin import SyntheticMANO
    from oracle import head_restated as head

    model, inputs, gold, case = build_product("swint_encoder_patch_spatial")
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    for k in sd:
        if k.startswith("spatial_encoder.layers.0.") and sd[k].is_floating_point():
            sd[k] = torch.randn_like(sd[k])
    with torch.no_grad():
        out = head.predict_batch(inputs, sd, head_options(case), SyntheticMANO(), execute_all=True)
    assert rel(out["joint_cam"], gold["joint_cam"]) < 2e-5


def test_rotation_tail_backward_is_finite_at_clamped_entries():
    """matrix_to_quaternion takes sqrt of four terms that are exactly 0 (or round-off negative) for rotations whose quaternion
    has a zero component; the reference gives them a zero subgradient (ref:cs_vit/utils/geometry.py:150-161).  A NaN there
    poisons every gradient of the finetune step through clip_grad_norm_."""
    from cs_vit.utils.geometry import matrix_to_axis_angle, rotation_6d_to_matrix
    R = torch.stack([torch.diag(torch.tensor([1.0, -1.0, -1.0])), torch.eye(3), torch.diag(torch.tensor([-1.0, 1.0, -1.0]))])
    R = R.clone().requires_grad_(True)
    aa = matrix_to_axis_angle(R)
    aa.square().sum().backward()
    assert torch.isfinite(aa).all() and torch.isfinite(R.grad).all()
    d6 = torch.tensor([[1.0, 0.0, 0.0, 0.0, 1.0, 0.0], [0.3, -0.2, 0.9, 0.1, 0.8, -0.5]], requires_grad=True)
    matrix_to_axis_angle(rotation_6d_to_matrix(d6)).sum().backward()
    assert torch.isfinite(d6.grad).all()


def test_restated_stochastic_depth_matches_reference_autograd():
    """Train-mode Swin-T backbone with drop_path_rate 0.1 under the reference's recorded uniform draws: features and gradients of
    the restatement's autograd against the golden the unmodified HF modules produced (oracle/make_train_goldens.py)."""
    import numpy as np
    from helpers import GOLDEN, build_train_case
    from oracle import head_restated as head
    from oracle import swin_restated as swin
    model, batch, gold, case = build_train_case("train_backbone_swint_linear_droppath", "fp32")
    assert case["drop_path_rate"] == 0.1
    bsd = {k[len("backbone."):]: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()
           if k.startswith("backbone.") and v.is_floating_point()}
    imgs = batch["patches"].reshape(case["batch"], 3, 224, 224)
    mean = torch.tensor(head.IMAGENET_MEAN)[None, :, None, None]
    std = torch.tensor(head.IMAGENET_STD)[None, :, None, None]
    from cs_vit.synthetic import SWIN_VARIANTS
    _, depths, heads = SWIN_VARIANTS[case["variant"]]
    feats = swin.swin_forward((imgs - mean) / std, bsd, depths, heads, drop_path_rate=0.1, drop_draws=torch.from_numpy(gold["droppath_rand"]))
    ref = torch.from_numpy(gold["features"])
    assert ((feats.detach() - ref).norm() / ref.norm()).item() < 1e-5
    # the dropped samples make this differ from the plain forward: the masks really act
    plain = np.load(os.path.join(GOLDEN, "train_backbone_swint_linear.npz"))["features"]
    assert np.abs(plain - gold["features"]).max() > 1e-2
    R = torch.randn(feats.shape, generator=torch.Generator().manual_seed(case["linear_loss_seed"]))
    (feats * R).sum().backward()
    checked = 0
    for key in gold:
        if key.startswith("grad/"):
            g, want = bsd[key[5:]].grad, torch.from_numpy(gold[key])
            assert ((g - want).norm() / want.norm().clamp_min(1e-12)).item() < 2e-4, key
            checked += 1
    assert checked > 100
