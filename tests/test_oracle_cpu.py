"""Pins oracle/restate.py against the committed golden vectors (produced by executing the unmodified
reference, oracle/make_golden.py)."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import restate

GOLD = Path(__file__).parent / "golden"


# d=64 / per-frame mask;  d=88, mlp 48/11, tube mask, 1+2 taps;  train mode: injected DropPath draw + tanh GELU
FIXTURES = ["pretrain_tiny", "pretrain_d88", "pretrain_dp"]


def fixture_kwargs(z, name):
    """Extra restatement arguments a fixture needs (pretrain_dp: stochastic-depth factors, FusedMLP's tanh GELU)."""
    if name == "pretrain_dp":
        return dict(gelu_mode="tanh", drop_path=torch.from_numpy(z["drop_path_factors"]))
    return {}


def load_tiny(name="pretrain_tiny"):
    z = np.load(GOLD / f"{name}.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    p = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w/")}
    g = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("g/")}
    return z, cfg, p, g


def restate_cfg(cfg):
    depth = cfg["depth"]
    return dict(depth=depth, num_heads=cfg["num_heads"], attn_pool_num_heads=cfg["attn_pool_num_heads"],
                patch_size=cfg["patch_size"], tubelet_size=1,
                clip_return_index=[depth - 1 - i for i in range(cfg["clip_return_layer"])],
                mae_return_index=[depth - 1 - i for i in range(cfg["mae_return_layer"])])


@pytest.mark.parametrize("fixture", FIXTURES)
def test_forward_matches_golden(fixture):
    z, cfg, p, _ = load_tiny(fixture)
    rc = restate_cfg(cfg)
    out = restate.forward_pretrain(p, rc, torch.from_numpy(z["x"]), torch.from_numpy(z["mask"]), **fixture_kwargs(z, fixture))
    # the reference appends taps in block order; clip_return_index is stored descending but taps are
    # collected ascending (internvideo2_pretrain.py:664-683) -> same order as ours.
    for o, name in zip(out, ("x_clip_align", "x_align", "x_mae_align")):
        ref = torch.from_numpy(z[name])
        assert o.shape == ref.shape
        assert torch.allclose(o, ref, atol=2e-5, rtol=1e-4), (name, (o - ref).abs().max())


@pytest.mark.parametrize("fixture", FIXTURES)
def test_losses_and_grads_match_golden(fixture):
    z, cfg, p, g = load_tiny(fixture)
    p = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in p.items()}
    out = restate.forward_pretrain(p, restate_cfg(cfg), torch.from_numpy(z["x"]), torch.from_numpy(z["mask"]),
                                   **fixture_kwargs(z, fixture))
    ls = [restate.align_loss(o, torch.from_numpy(z[t])) for o, t in zip(out, ("tgt_clip", "tgt_final", "tgt_mae"))]
    for l, name in zip(ls, ("loss_clip", "loss_final", "loss_mae")):
        assert abs(float(l) - float(z[name])) < 1e-5
    sum(ls).backward()
    for k, ref in g.items():
        got = p[k].grad
        assert got is not None, k
        assert torch.allclose(got, ref, atol=3e-6, rtol=2e-3), (k, (got - ref).abs().max())


@pytest.mark.parametrize("fixture", FIXTURES)
def test_visible_indices_bit_exact(fixture):
    z, cfg, p, _ = load_tiny(fixture)
    mask = torch.from_numpy(z["mask"])
    idx = restate.visible_indices(mask)
    B, N = mask.shape
    ar = torch.arange(N).expand(B, N)
    assert torch.equal(idx, ar[~mask].reshape(B, -1))          # == x[~mask] ordering (:659)
    assert idx.dtype == torch.int64 and bool((idx[:, 0] == 0).all())


def test_block_cfg2_matches_golden():
    """One Block at the 1B model's real size (D=1408, 16x88, hidden 6144, n=417, B=2): the restatement against
    the rows/norms the unmodified reference Block produced (weights regenerated from the fixture's seed)."""
    from oracle.make_golden import block_cfg2_inputs
    z = np.load(GOLD / "block_cfg2.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    sd, x, dy = block_cfg2_inputs(cfg)
    p = {"blocks.0." + k: v.clone().requires_grad_(True) for k, v in sd.items()}
    x = x.clone().requires_grad_(True)
    y = restate.block(p, 0, x, cfg["num_heads"])
    y.backward(dy)
    rows = torch.from_numpy(z["rows"]).long()
    D = cfg["dim"]
    assert torch.allclose(y.detach().reshape(-1, D)[rows], torch.from_numpy(z["y_rows"]).float(), atol=2e-2, rtol=2e-3)
    assert abs(float(y.detach().double().norm()) - float(z["y_norm"])) < 1e-4 * float(z["y_norm"])
    assert torch.allclose(x.grad.reshape(-1, D)[rows], torch.from_numpy(z["dx_rows"]).float(), atol=1e-3, rtol=2e-3)
    assert abs(float(x.grad.double().norm()) - float(z["dx_norm"])) < 1e-4 * float(z["dx_norm"])
    for k in sd:
        g = p["blocks.0." + k].grad
        ref = torch.from_numpy(z["g/" + k])
        got = g[::64] if g.ndim == 2 else g
        assert torch.allclose(got, ref, atol=1e-4 * float(ref.abs().max()), rtol=2e-3), k
        assert abs(float(g.double().norm()) - float(z["gn/" + k])) < 1e-4 * float(z["gn/" + k]), k


def test_clip_small_matches_golden():
    """cfg-3 surface: unmasked tower -> vision_align -> vtc_loss (learnable temperature, duplicate caption)."""
    z = np.load(GOLD / "clip_small.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    p = {k[2:]: torch.from_numpy(z[k]).clone().requires_grad_(True) for k in z.files if k.startswith("w/")}
    rc = dict(depth=cfg["depth"], num_heads=cfg["num_heads"], attn_pool_num_heads=cfg["attn_pool_num_heads"],
              patch_size=cfg["patch_size"], tubelet_size=1, num_frames=cfg["num_frames"])
    image = torch.from_numpy(z["image"])
    v = restate.clip_small_embed(p, rc, image)
    assert torch.allclose(v, torch.from_numpy(z["vision_embeds"]), atol=2e-5, rtol=1e-4)
    temp = torch.tensor(float(z["temp"]), requires_grad=True)
    loss = restate.vtc_loss(v, torch.from_numpy(z["text"]), torch.from_numpy(z["idx"]), temp)
    assert abs(float(loss) - float(z["loss"])) < 1e-5
    loss.backward()
    assert abs(float(temp.grad) - float(z["g/temp"])) < 1e-3 * abs(float(z["g/temp"]))
    for k in z.files:
        if k.startswith("g/") and k != "g/temp":
            assert torch.allclose(p[k[2:]].grad, torch.from_numpy(z[k]), atol=3e-6, rtol=2e-3), k
    with torch.no_grad():
        vi = restate.clip_small_embed(p, rc, image[:, :1], use_image=True)
    assert torch.allclose(vi, torch.from_numpy(z["vision_embeds_image"]), atol=2e-5, rtol=1e-4)


def test_teachers_and_mask_match_golden():
    """Frozen teachers + attention-guided mask (SURVEY §8f-1): restatement vs outputs of the unmodified reference."""
    z = np.load(GOLD / "teachers.npz")
    ccfg = json.loads(bytes(z["clip_cfg"]).decode()); mcfg = json.loads(bytes(z["mae_cfg"]).decode())
    pc = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("wc/")}
    pm = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("wm/")}
    depth = ccfg["depth"]
    rc = dict(depth=depth, num_heads=ccfg["num_heads"], attn_pool_num_heads=ccfg["attn_pool_num_heads"],
              patch_size=ccfg["patch_size"], return_index=[depth - 1 - i for i in range(ccfg["clip_return_layer"])])
    with torch.no_grad():
        zz, x, attn = restate.internvl_clip_forward(pc, rc, torch.from_numpy(z["clip_video"]))
    assert torch.allclose(zz, torch.from_numpy(z["z"]), atol=2e-5, rtol=1e-4)
    assert torch.allclose(x, torch.from_numpy(z["x"]), atol=2e-5, rtol=1e-4)
    assert torch.allclose(attn, torch.from_numpy(z["attn"]), atol=1e-6, rtol=1e-4)
    from internvideo_b200.teachers import get_sinusoid_encoding_table
    md = mcfg["depth"]
    rm = dict(depth=md, num_heads=mcfg["num_heads"], patch_size=mcfg["patch_size"], tubelet_size=mcfg["tubelet_size"],
              return_index=[md - 1 - i for i in range(mcfg["mae_return_layer"])], eps=1e-6)
    pos = get_sinusoid_encoding_table(2048, mcfg["embed_dim"])
    with torch.no_grad():
        zm = restate.videomae_teacher_forward(pm, rm, torch.from_numpy(z["mae_video"]).float(), pos)
    assert torch.allclose(zm, torch.from_numpy(z["zm"]).float(), atol=2e-3, rtol=2e-3)     # stored as fp16
    # the standard token-axis attention is NOT what the reference computes (videomae.py:94-97)
    with torch.no_grad():
        zs = restate.videomae_teacher_forward(pm, rm, torch.from_numpy(z["mae_video"]).float(), pos, head_axis_attention=False)
    assert (zs - torch.from_numpy(z["zm"]).float()).abs().max() > 1e-2
    imp = torch.from_numpy(z["importance"])
    mask = restate.attention_guided_mask(torch.from_numpy(z["attn"]), 2, 0.75, imp)
    assert torch.equal(mask, torch.from_numpy(z["mask"]))                                    # bit-exact
    zt = torch.from_numpy(z["z"])
    vis = zt[~mask.unsqueeze(0).repeat(zt.shape[0], 1, 1)].reshape(zt.shape[0], 2, -1, zt.shape[-1])
    assert torch.equal(vis, torch.from_numpy(z["targets_clip_middle_vis"]))


def test_vtc_matches_golden():
    z = np.load(GOLD / "vtc.npz")
    v = [torch.from_numpy(z[f"v{r}"]).requires_grad_(True) for r in range(2)]
    t = [torch.from_numpy(z[f"t{r}"]).requires_grad_(True) for r in range(2)]
    idx = [torch.from_numpy(z[f"idx{r}"]) for r in range(2)]
    for rank in range(2):
        # what rank `rank` computes: gathered tensors where only its own rows carry grad
        va = restate.allgather_rows([x if r == rank else x.detach() for r, x in enumerate(v)])
        ta = restate.allgather_rows([x if r == rank else x.detach() for r, x in enumerate(t)])
        loss = restate.vtc_loss(va, ta, restate.allgather_rows(idx), float(z["temp"]))
        assert abs(float(loss) - float(z[f"loss{rank}"])) < 1e-5
        gv, gt = torch.autograd.grad(loss, [v[rank], t[rank]])
        assert torch.allclose(gv, torch.from_numpy(z[f"gv{rank}"]), atol=1e-6, rtol=1e-4)
        assert torch.allclose(gt, torch.from_numpy(z[f"gt{rank}"]), atol=1e-6, rtol=1e-4)
    m = restate.get_mask(restate.allgather_rows(idx))
    assert torch.allclose(m.sum(1), torch.ones(16))
    assert m[3, 8] > 0 and m[3, 13] > 0 and abs(float(m[3, 3]) - 1 / 3) < 1e-6   # soft targets on duplicates


def test_pixel_target_matches_golden():
    z = np.load(GOLD / "pixel_target.npz")
    im, mask = torch.from_numpy(z["images"]), torch.from_numpy(z["mask"])
    assert torch.allclose(restate.pixel_targets(im, mask, 16, 2, True), torch.from_numpy(z["labels"]), atol=1e-5, rtol=1e-5)
    assert torch.allclose(restate.pixel_targets(im, mask, 16, 2, False), torch.from_numpy(z["labels_raw"]), atol=1e-6)


def test_restatement_vs_live_reference_sdims():
    """BASELINE cfg-1: InternVideo2-S dims, 2 clips x 4 frames x 224^2, CPU eager, seeded weights: a seeded sample and
    the norm of every output against the reference's (tests/golden/ref_checks.npz)."""
    from oracle.make_golden import SDIMS_SEED, sample_flat, sdims_inputs, seeded_state
    ref = np.load(GOLD / "ref_checks.npz")
    p = seeded_state(json.loads(bytes(ref["sdims/layout"]).decode()), SDIMS_SEED)
    x, mask = sdims_inputs()
    with torch.no_grad():
        rc = dict(depth=12, num_heads=6, attn_pool_num_heads=16, patch_size=14, tubelet_size=1,
                  clip_return_index=[11], mae_return_index=[11])
        out = restate.forward_pretrain(p, rc, x, mask)
    assert [tuple(o.shape) for o in out] == [(1, 2, 209, 3200), (2, 768), (1, 2, 208, 1408)]
    for i, o in enumerate(out):
        assert tuple(o.shape) == tuple(ref[f"sdims/shape{i}"])
        o_s, r_s = sample_flat(o, 4096, 100 + i), torch.from_numpy(ref[f"sdims/sample{i}"])
        assert torch.allclose(o_s, r_s, atol=3e-5, rtol=1e-4), (o_s - r_s).abs().max()
        assert abs(float(o.double().norm()) - float(ref[f"sdims/norm{i}"])) <= 1e-4 * float(ref[f"sdims/norm{i}"])


def test_stage2_tower_restatement_matches_golden():
    """oracle/restate.forward_stage2_tower against the reference-generated fixture (SURVEY §8 f-3)."""
    z = np.load(GOLD / "stage2.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    p = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w/")}
    depth = cfg["depth"]
    rc = dict(depth=depth, num_heads=cfg["num_heads"], attn_pool_num_heads=cfg["attn_pool_num_heads"],
              patch_size=cfg["patch_size"], tubelet_size=cfg["tubelet_size"], num_frames=cfg["num_frames"],
              return_index=[depth - 1 - i * cfg["clip_student_return_interval"] for i in range(cfg["clip_return_layer"])])
    video = torch.from_numpy(z["video"]); mask = torch.from_numpy(z["mask"])
    names = ("x_vis", "x_pool_vis", "x_clip_align", "x_align")
    for tag, out in (("a", restate.forward_stage2_tower(p, rc, video)),
                     ("b", restate.forward_stage2_tower(p, rc, video, mask)),
                     ("c", restate.forward_stage2_tower(p, rc, video[:, :, :1], None, True))):
        for nm, t in zip(names, out):
            assert torch.allclose(t, torch.from_numpy(z[f"{tag}/{nm}"]), atol=3e-5, rtol=1e-4), (tag, nm)
    d = restate.forward_stage2_tower(p, rc, video, mask, False, -2, True)
    assert torch.allclose(d, torch.from_numpy(z["d/x_vis"]), atol=3e-5, rtol=1e-4)
    pe = dict(p, img_pos_embed=torch.from_numpy(z["e/img_pos_embed"]), clip_img_pos_embed=torch.from_numpy(z["e/clip_img_pos_embed"]))
    for nm, t in zip(names, restate.forward_stage2_tower(pe, rc, video[:, :, :1], None, True)):
        assert torch.allclose(t, torch.from_numpy(z[f"e/{nm}"]), atol=3e-5, rtol=1e-4), ("e", nm)


def test_iv1_videomae_restatement_matches_golden():
    """oracle/restate.forward_iv1_videomae + pixel_targets + mse_loss against the reference-generated fixture (§8 a15 / f-4)."""
    z = np.load(GOLD / "iv1_videomae.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    p = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w/")}
    rc = dict(encoder_depth=cfg["encoder_depth"], encoder_num_heads=cfg["encoder_num_heads"], decoder_depth=cfg["decoder_depth"],
              decoder_num_heads=cfg["decoder_num_heads"], patch_size=cfg["patch_size"], tubelet_size=cfg["tubelet_size"], eps=1e-6)
    images = torch.from_numpy(z["images"]); mask = torch.from_numpy(z["mask"])
    out = restate.forward_iv1_videomae(p, rc, images, mask)
    assert torch.allclose(out, torch.from_numpy(z["out"]), atol=5e-5, rtol=1e-4)
    enc = restate.forward_iv1_videomae(p, rc, images, mask, return_encoder=True)
    assert torch.allclose(enc, torch.from_numpy(z["enc_out"]), atol=5e-5, rtol=1e-4)
    labels = restate.pixel_targets(images, mask, cfg["patch_size"], cfg["tubelet_size"], True)
    assert torch.allclose(labels, torch.from_numpy(z["labels"]), atol=1e-5, rtol=1e-5)
    assert abs(float(restate.mse_loss(out, labels)) - float(z["loss"])) < 1e-5
