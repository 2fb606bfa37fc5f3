"""TEST INFRASTRUCTURE ONLY — generate tests/golden/*.npz by EXECUTING the unmodified reference.

Run in the build container (where /root/reference is mounted):  python oracle/make_golden.py
The GPU box has no /root/reference; it only reads the committed .npz files.

Fixtures
  pretrain_tiny.npz  PretrainInternVideo2 (reference ctor, naive path) D=128, 2 heads (d=64), depth 2,
                     2 frames of 56x56: weights (bf16-representable), input, mask, the three outputs,
                     hidden states, the 2-2cos losses against seeded targets and d(loss)/d(param).
  pretrain_d88.npz   same, D=176 with 2 heads of d=88 (the 1B model's head_dim), mlp_ratio 48/11, 1 CLIP + 2 MAE
                     taps, B=3, tube mask.
  pretrain_dp.npz    TRAIN mode, D=176 / d=88, depth 3, stochastic depth 0.4 with the per-sample draw stored and
                     injected, tanh GELU (FusedMLP's activation), B=4, 2+2 taps: the path bench.py runs.
  block_cfg2.npz     one reference Block at the 1B model's real size (D=1408, 16x88, hidden 6144, n=417, B=2):
                     output / input-gradient rows and parameter-gradient rows + norms; weights come from a seed.
  clip_small.npz     cfg-3 surface: the reference's unmasked InternVideo2 tower -> vision_align -> vtc_loss with a
                     learnable temperature and a duplicate caption; outputs, loss, every gradient; use_image forward.
  teachers.npz       frozen teachers (InternVL_CLIP per-frame ViT; VideoMAE ViT at the recipe geometry) + the
                     attention-guided mask / target selection of engine_for_pretraining.py:105-125 with the draw injected.
  vtc.npz            VTC_VTM_Loss.vtc_loss on 2 gloo ranks through the reference AllGather: inputs per
                     rank, loss, and the per-rank input gradients (local-slice backward semantics).
  pixel_target.npz   IV1 VideoMAE target construction: the reference's own statements
                     (engine_for_pretraining.py:66-98) exec'd on a seeded clip.
  ref_checks.npz     small results of reference functions and modules that the CPU tests check host code against:
                     mask generators, position tables and interpolation, a reference-built model's attributes, an
                     InternVideo2-S forward on seeded weights (sampled), stage-2 criterions, recall@k, IV1 init digests.
"""
from __future__ import annotations

import json
import os
from functools import partial
import sys
import textwrap
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle import ref_shim  # noqa: E402

GOLD = ROOT / "tests" / "golden"


def bf16_round(t):
    return t.to(torch.bfloat16).to(torch.float32)


TINY_CFG = dict(embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, num_frames=2, img_size=56,
                patch_size=14, drop_path_rate=0.0, attn_pool_num_heads=2, clip_embed_dim=96,
                clip_teacher_embed_dim=160, clip_teacher_final_dim=96, mae_teacher_embed_dim=128,
                clip_return_layer=2, mae_return_layer=1, init_values=0.1)


def make_pretrain_tiny():
    torch.manual_seed(1234)
    model = ref_shim.build_reference_model(**TINY_CFG).eval()
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for name, p in model.named_parameters():
            # make every term matter: perturb zero-init biases / unit norm weights / LayerScale
            if name.endswith("bias") or name.endswith("_bias"):
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
            elif "norm" in name and name.endswith("weight"):
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith("gamma"):
                p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
            elif name == "cls_token":
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            p.copy_(bf16_round(p))
    B, T, L = 2, TINY_CFG["num_frames"], (TINY_CFG["img_size"] // TINY_CFG["patch_size"]) ** 2
    x = bf16_round(torch.randn(B, 3, T, 56, 56, generator=g))
    mask = torch.ones(B, 1 + T * L, dtype=torch.bool)
    mask[:, 0] = False
    for b in range(B):
        for t in range(T):
            keep = torch.randperm(L, generator=g)[:6]
            mask[b, 1 + t * L + keep] = False
    out = model(x, mask)
    # seeded, L2-normalised stand-ins for the teacher targets (engine_for_pretraining.py:118-125)
    tg = [torch.nn.functional.normalize(torch.randn(o.shape, generator=g), dim=-1) for o in out]
    # losses: engine_for_pretraining.py:131-136,148
    losses = [(2 - 2 * (o * t).sum(dim=-1)).mean() for o, t in zip(out, tg)]
    loss = losses[0] + losses[1] + losses[2]
    model.zero_grad()
    loss.backward()
    blob = {"cfg": np.frombuffer(json.dumps(TINY_CFG).encode(), dtype=np.uint8),
            "x": x.numpy(), "mask": mask.numpy(),
            "x_clip_align": out[0].detach().numpy(), "x_align": out[1].detach().numpy(),
            "x_mae_align": out[2].detach().numpy(),
            "tgt_clip": tg[0].numpy(), "tgt_final": tg[1].numpy(), "tgt_mae": tg[2].numpy(),
            "loss_clip": losses[0].detach().numpy(), "loss_final": losses[1].detach().numpy(),
            "loss_mae": losses[2].detach().numpy()}
    for k, v in model.state_dict().items():
        blob["w/" + k] = v.numpy()
    for k, p in model.named_parameters():
        blob["g/" + k] = p.grad.numpy()
    np.savez_compressed(GOLD / "pretrain_tiny.npz", **blob)
    print("pretrain_tiny:", [tuple(o.shape) for o in out], float(loss))


D88_CFG = dict(embed_dim=176, depth=2, num_heads=2, mlp_ratio=48 / 11, num_frames=2, img_size=56,
               patch_size=14, drop_path_rate=0.0, attn_pool_num_heads=2, clip_embed_dim=64,
               clip_teacher_embed_dim=96, clip_teacher_final_dim=64, mae_teacher_embed_dim=176,
               clip_return_layer=1, mae_return_layer=2, init_values=0.05)


def make_pretrain_d88():
    """Second model fixture: the 1B model's odd head_dim (88 = 1408/16, zero-padded to 96 columns inside the
    attention kernels), its non-integer mlp_ratio 48/11, 1 CLIP tap + 2 MAE taps, and a TUBE mask (the same
    kept patches in every frame — datasets/masking_generator.py:4-25) with a different keep count."""
    torch.manual_seed(4321)
    model = ref_shim.build_reference_model(**D88_CFG).eval()
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("bias") or name.endswith("_bias"):
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
            elif "norm" in name and name.endswith("weight"):
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith("gamma"):
                p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
            elif name == "cls_token":
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            p.copy_(bf16_round(p))
    B, T, L = 3, D88_CFG["num_frames"], (D88_CFG["img_size"] // D88_CFG["patch_size"]) ** 2
    x = bf16_round(torch.randn(B, 3, T, 56, 56, generator=g))
    mask = torch.ones(B, 1 + T * L, dtype=torch.bool)
    mask[:, 0] = False
    for b in range(B):
        keep = torch.randperm(L, generator=g)[:5]          # tube: same patches in every frame
        for t in range(T):
            mask[b, 1 + t * L + keep] = False
    out = model(x, mask)
    tg = [torch.nn.functional.normalize(torch.randn(o.shape, generator=g), dim=-1) for o in out]
    losses = [(2 - 2 * (o * t).sum(dim=-1)).mean() for o, t in zip(out, tg)]
    loss = losses[0] + losses[1] + losses[2]
    model.zero_grad()
    loss.backward()
    blob = {"cfg": np.frombuffer(json.dumps(D88_CFG).encode(), dtype=np.uint8),
            "x": x.numpy(), "mask": mask.numpy(),
            "x_clip_align": out[0].detach().numpy(), "x_align": out[1].detach().numpy(),
            "x_mae_align": out[2].detach().numpy(),
            "tgt_clip": tg[0].numpy(), "tgt_final": tg[1].numpy(), "tgt_mae": tg[2].numpy(),
            "loss_clip": losses[0].detach().numpy(), "loss_final": losses[1].detach().numpy(),
            "loss_mae": losses[2].detach().numpy()}
    for k, v in model.state_dict().items():
        blob["w/" + k] = v.numpy()
    for k, p in model.named_parameters():
        blob["g/" + k] = p.grad.numpy()
    np.savez_compressed(GOLD / "pretrain_d88.npz", **blob)
    print("pretrain_d88:", [tuple(o.shape) for o in out], float(loss))


DP_CFG = dict(embed_dim=176, depth=3, num_heads=2, mlp_ratio=48 / 11, num_frames=2, img_size=56,
              patch_size=14, drop_path_rate=0.4, attn_pool_num_heads=2, clip_embed_dim=64,
              clip_teacher_embed_dim=96, clip_teacher_final_dim=64, mae_teacher_embed_dim=176,
              clip_return_layer=2, mae_return_layer=2, init_values=0.08)


class _InjectedDropPath(torch.nn.Module):
    """timm DropPath with the Bernoulli draw made beforehand: x * factor[b] (factor = keep_mask / keep_prob).
    Replaces the stub DropPath instances of the reference Block (timm itself is not installed) so that the
    draw can be stored in the fixture and injected into the CUDA path (SURVEY App.B-16)."""

    def __init__(self, factor):
        super().__init__()
        self.factor = factor

    def forward(self, x):
        return x * self.factor.view(-1, *([1] * (x.ndim - 1)))


def make_pretrain_dp():
    """Third model fixture — the path bench.py actually runs: TRAIN mode with stochastic depth (per-sample
    DropPath factors injected: exercises the `rowscale` of the residual GEMM epilogues and of layerscale_bwd)
    and the tanh GELU of FA2's FusedMLP (`use_fused_mlp=True` in the recipes; the extension is absent here, so the
    reference Mlp's activation is swapped for nn.GELU(approximate='tanh') — the same math FusedMLP documents)."""
    torch.manual_seed(2468)
    model = ref_shim.build_reference_model(**DP_CFG).train()
    g = torch.Generator().manual_seed(13)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("bias") or name.endswith("_bias"):
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
            elif "norm" in name and name.endswith("weight"):
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith("gamma"):
                p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
            elif name == "cls_token":
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            p.copy_(bf16_round(p))
    B, T, L = 4, DP_CFG["num_frames"], (DP_CFG["img_size"] // DP_CFG["patch_size"]) ** 2
    depth = DP_CFG["depth"]
    rates = [DP_CFG["drop_path_rate"] * i / (depth - 1) for i in range(depth)]
    factors = torch.ones(2 * depth, B)
    for i, blk in enumerate(model.blocks):
        blk.mlp.act = torch.nn.GELU(approximate="tanh")
        for j, attr in enumerate(("drop_path1", "drop_path2")):
            keep = 1.0 - rates[i]
            f = torch.bernoulli(torch.full((B,), keep), generator=g) / keep
            if i == depth - 1 and j == 0:
                f[1] = 0.0                                  # make sure a dropped sample is in the fixture
            factors[2 * i + j] = f
            if rates[i] > 0:
                setattr(blk, attr, _InjectedDropPath(factors[2 * i + j]))
            else:
                factors[2 * i + j] = 1.0
    x = bf16_round(torch.randn(B, 3, T, 56, 56, generator=g))
    mask = torch.ones(B, 1 + T * L, dtype=torch.bool)
    mask[:, 0] = False
    for b in range(B):
        for t in range(T):
            mask[b, 1 + t * L + torch.randperm(L, generator=g)[:7]] = False
    out = model(x, mask)
    tg = [torch.nn.functional.normalize(torch.randn(o.shape, generator=g), dim=-1) for o in out]
    losses = [(2 - 2 * (o * t).sum(dim=-1)).mean() for o, t in zip(out, tg)]
    loss = losses[0] + losses[1] + losses[2]
    model.zero_grad()
    loss.backward()
    blob = {"cfg": np.frombuffer(json.dumps(DP_CFG).encode(), dtype=np.uint8),
            "x": x.numpy(), "mask": mask.numpy(), "drop_path_factors": factors.numpy(),
            "x_clip_align": out[0].detach().numpy(), "x_align": out[1].detach().numpy(),
            "x_mae_align": out[2].detach().numpy(),
            "tgt_clip": tg[0].numpy(), "tgt_final": tg[1].numpy(), "tgt_mae": tg[2].numpy(),
            "loss_clip": losses[0].detach().numpy(), "loss_final": losses[1].detach().numpy(),
            "loss_mae": losses[2].detach().numpy()}
    for k, v in model.state_dict().items():
        blob["w/" + k] = v.numpy()
    for k, p in model.named_parameters():
        blob["g/" + k] = p.grad.numpy()
    np.savez_compressed(GOLD / "pretrain_dp.npz", **blob)
    print("pretrain_dp:", [tuple(o.shape) for o in out], float(loss), "factors", factors.tolist())


BLOCK_CFG2 = dict(dim=1408, num_heads=16, mlp_ratio=48 / 11, init_values=0.1, B=2, n=417, seed=97)


def block_cfg2_inputs(cfg=BLOCK_CFG2):
    """Seeded weights / input / upstream gradient of the cfg-2-size Block fixture (25 M weights: regenerated
    from the seed wherever the fixture is used instead of being stored).  torch's CPU generator is
    deterministic for a given torch build, and the GPU box runs this same image."""
    D, H = cfg["dim"], cfg["num_heads"]
    Hd = int(D * cfg["mlp_ratio"])
    g = torch.Generator().manual_seed(cfg["seed"])
    r = lambda *s, std=1.0: bf16_round(torch.randn(*s, generator=g) * std)
    sd = {"norm1.weight": 1 + r(D, std=0.1), "attn.qkv.weight": r(3 * D, D, std=0.03),
          "attn.q_norm.weight": 1 + r(D, std=0.1), "attn.k_norm.weight": 1 + r(D, std=0.1),
          "attn.proj.weight": r(D, D, std=0.03), "attn.proj.bias": r(D, std=0.05),
          "ls1.gamma": cfg["init_values"] * (1 + r(D, std=0.3)), "norm2.weight": 1 + r(D, std=0.1),
          "mlp.fc1.weight": r(Hd, D, std=0.03), "mlp.fc1.bias": r(Hd, std=0.05),
          "mlp.fc2.weight": r(D, Hd, std=0.02), "mlp.fc2.bias": r(D, std=0.05),
          "ls2.gamma": cfg["init_values"] * (1 + r(D, std=0.3))}
    sd = {k: bf16_round(v) for k, v in sd.items()}
    x = r(cfg["B"], cfg["n"], D)
    dy = r(cfg["B"], cfg["n"], D, std=0.05)
    return sd, x, dy


def block_cfg2_rows(cfg=BLOCK_CFG2):
    """Token rows of the flattened [B*n, D] output / input-gradient that the fixture stores: every other row plus
    the complete tail tile; weight gradients are stored as every 64th row plus their full norm."""
    M = cfg["B"] * cfg["n"]
    return sorted(set(range(0, M, 2)) | set(range(M - 40, M)))


def make_block_cfg2():
    """ONE reference Block at the 1B model's real dimensions (D=1408, 16 heads of 88, hidden 6144, n=417
    visible tokens, 2 clips): forward output, input gradient and parameter gradients of the unmodified
    reference module (internvideo2_pretrain.py:247-297, naive path, fp32 on the host cores)."""
    cfg = BLOCK_CFG2
    mod = ref_shim.import_single_modality()
    blk = mod.Block(cfg["dim"], cfg["num_heads"], cfg["mlp_ratio"], qkv_bias=False, init_values=cfg["init_values"],
                    drop_path=0.0, norm_layer=mod.RMSNorm, use_flash_attn=False, use_fused_mlp=False,
                    qk_normalization=True, use_fused_rmsnorm=False)
    sd, x, dy = block_cfg2_inputs(cfg)
    blk.load_state_dict(sd, strict=True)
    x = x.clone().requires_grad_(True)
    y = blk(x)
    y.backward(dy)
    rows = block_cfg2_rows(cfg)
    D = cfg["dim"]
    blob = {"cfg": np.frombuffer(json.dumps(cfg).encode(), dtype=np.uint8), "rows": np.asarray(rows, dtype=np.int32),
            "y_rows": y.detach().reshape(-1, D)[rows].numpy().astype(np.float16),
            "dx_rows": x.grad.reshape(-1, D)[rows].numpy().astype(np.float16),
            "y_norm": np.float64(y.detach().double().norm()), "dx_norm": np.float64(x.grad.double().norm())}
    for k, p in blk.named_parameters():
        gk = p.grad
        blob["gn/" + k] = np.float64(gk.double().norm())
        blob["g/" + k] = (gk[::64] if gk.ndim == 2 else gk).numpy()
    np.savez_compressed(GOLD / "block_cfg2.npz", **blob)
    print("block_cfg2: y", tuple(y.shape), float(y.norm()), "dx", float(x.grad.norm()))


CLIP_CFG = dict(embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, num_frames=2, img_size=56, patch_size=14,
                drop_path_rate=0.0, attn_pool_num_heads=2, clip_embed_dim=96, init_values=0.1,
                layerscale_no_force_fp32=True, qk_normalization=True)
CLIP_ALIGN_DIM = 64


def make_clip_small():
    """BASELINE cfg-3 surface at toy size: the reference's unmasked `InternVideo2` tower
    (internvideo2_clip_vision.py:340-548, naive path) -> vision_align (LayerNorm + Linear, internvideo2_clip_small.py:35-41)
    -> VTC_VTM_Loss.vtc_loss against seeded text embeddings with a learnable temperature; outputs, loss and the
    gradient of every parameter; plus the single-image (`use_image=True`, temporal-mean position table) forward."""
    mod = ref_shim.import_clip_vision()
    crit, _ = ref_shim.import_criterions()
    torch.manual_seed(1357)
    tower = mod.InternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **CLIP_CFG).eval()
    align = torch.nn.Sequential(torch.nn.LayerNorm(CLIP_CFG["clip_embed_dim"]),
                                torch.nn.Linear(CLIP_CFG["clip_embed_dim"], CLIP_ALIGN_DIM))
    temp = torch.nn.Parameter(torch.ones([]) * 0.07)
    g = torch.Generator().manual_seed(17)
    with torch.no_grad():
        for name, p in list(tower.named_parameters()) + list(align.named_parameters()):
            if name.endswith("bias") or name.endswith("_bias"):
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
            elif ("norm" in name or name.startswith("0.")) and name.endswith("weight"):
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith("gamma"):
                p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
            elif name == "cls_token":
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            p.copy_(bf16_round(p))
        temp.copy_(bf16_round(temp))
    B, T = 4, CLIP_CFG["num_frames"]
    image = bf16_round(torch.randn(B, T, 3, 56, 56, generator=g))            # [B,T,C,H,W] as the dataloader gives it
    text = torch.randn(B, CLIP_ALIGN_DIM, generator=g)
    idx = torch.tensor([5, 9, 5, 2])                                          # one duplicate caption -> soft targets
    v_tok = tower(image.permute(0, 2, 1, 3, 4), use_image=False)
    v = align(v_tok)
    loss = crit.VTC_VTM_Loss(False).vtc_loss(v, text, idx, temp, all_gather=False)
    loss.backward()
    with torch.no_grad():
        v_img = align(tower(image[:, :1].permute(0, 2, 1, 3, 4), use_image=True))
    blob = {"cfg": np.frombuffer(json.dumps(dict(CLIP_CFG, align_dim=CLIP_ALIGN_DIM)).encode(), dtype=np.uint8),
            "image": image.numpy(), "text": text.numpy(), "idx": idx.numpy(), "temp": temp.detach().numpy(),
            "vision_tokens": v_tok.detach().numpy(), "vision_embeds": v.detach().numpy(),
            "vision_embeds_image": v_img.numpy(), "loss": loss.detach().numpy(), "g/temp": temp.grad.numpy()}
    for k, t in tower.state_dict().items():
        blob["w/vision_encoder." + k] = t.numpy()
    for k, t in align.state_dict().items():
        blob["w/vision_align." + k] = t.numpy()
    for k, p in tower.named_parameters():
        blob["g/vision_encoder." + k] = p.grad.numpy()
    for k, p in align.named_parameters():
        blob["g/vision_align." + k] = p.grad.numpy()
    np.savez_compressed(GOLD / "clip_small.npz", **blob)
    print("clip_small: tokens", tuple(v_tok.shape), "embeds", tuple(v.shape), "loss", float(loss), "dtemp", float(temp.grad))


STAGE2_CFG = dict(embed_dim=128, depth=3, num_heads=2, mlp_ratio=4, num_frames=2, img_size=56, patch_size=14,
                  drop_path_rate=0.0, attn_pool_num_heads=2, clip_embed_dim=96, init_values=0.1, qk_normalization=True,
                  clip_teacher_embed_dim=80, clip_teacher_final_dim=48, clip_return_layer=2,
                  clip_student_return_interval=1, tubelet_size=1)


def make_stage2():
    """SURVEY §8 f-3: the stage-2 form of the tower (multi_modality/.../internvideo2.py:380-668, naive path) at toy size,
    executed unmodified: (a) video, no mask; (b) video with a per-clip random mask; (c) single image through the temporal
    mean of the position tables; (d) x_vis_only with an early exit (x_vis_return_idx=-2); (e) the same weights in a model
    with separate image tables (sep_image_video_pos_embed).  Forward outputs + parameter gradients of (b)."""
    mod = ref_shim.import_stage2_tower()
    import contextlib, io
    g = torch.Generator().manual_seed(29)

    def build(sep):
        torch.manual_seed(2468)
        with contextlib.redirect_stdout(io.StringIO()):
            m = mod.PretrainInternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False,
                                         sep_image_video_pos_embed=sep, **STAGE2_CFG).eval()
        return m

    tower = build(False)
    with torch.no_grad():
        for name, p in tower.named_parameters():
            if name.endswith("bias") or name.endswith("_bias"):
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
            elif "norm" in name and name.endswith("weight"):
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith("gamma"):
                p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
            elif name == "cls_token":
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            p.copy_(bf16_round(p))
    B, T = 3, STAGE2_CFG["num_frames"]
    L = (STAGE2_CFG["img_size"] // STAGE2_CFG["patch_size"]) ** 2
    video = bf16_round(torch.randn(B, 3, T, 56, 56, generator=g))
    keep = 11                                                     # visible patch tokens per clip (+ cls)
    mask = torch.ones(B, 1 + T * L, dtype=torch.bool)
    mask[:, 0] = False
    for b in range(B):
        mask[b, 1 + torch.randperm(T * L, generator=g)[:keep]] = False
    blob = {"cfg": np.frombuffer(json.dumps(STAGE2_CFG).encode(), dtype=np.uint8), "video": video.numpy(),
            "mask": mask.numpy()}
    with torch.no_grad():
        for tag, out in (("a", tower(video)), ("c", tower(video[:, :, :1], None, True))):
            for nm, t in zip(("x_vis", "x_pool_vis", "x_clip_align", "x_align"), out):
                blob[f"{tag}/{nm}"] = t.numpy()
        blob["d/x_vis"] = tower(video, mask, False, -2, True).numpy()
    out = tower(video, mask)
    for nm, t in zip(("x_vis", "x_pool_vis", "x_clip_align", "x_align"), out):
        blob[f"b/{nm}"] = t.detach().numpy()
    wt = [torch.randn(t.shape, generator=g) for t in out]
    loss = sum((t * w).sum() for t, w in zip(out, wt))
    loss.backward()
    for nm, w in zip(("x_vis", "x_pool_vis", "x_clip_align", "x_align"), wt):
        blob[f"b/w_{nm}"] = w.numpy()
    for k, t in tower.state_dict().items():
        blob["w/" + k] = t.numpy()
    for k, p in tower.named_parameters():
        blob["g/" + k] = p.grad.numpy() if p.grad is not None else np.zeros(tuple(p.shape), np.float32)
    sep = build(True)
    sd = tower.state_dict()
    with torch.no_grad():
        img_tab = bf16_round(torch.randn(1, L + 1, STAGE2_CFG["embed_dim"], generator=g) * 0.5)
        cimg_tab = bf16_round(torch.randn(1, L + 1, STAGE2_CFG["embed_dim"], generator=g) * 0.5)
    sd["img_pos_embed"], sd["clip_img_pos_embed"] = img_tab, cimg_tab
    sep.load_state_dict(sd, strict=True)
    with torch.no_grad():
        oe = sep(video[:, :, :1], None, True)
    blob["e/img_pos_embed"], blob["e/clip_img_pos_embed"] = img_tab.numpy(), cimg_tab.numpy()
    for nm, t in zip(("x_vis", "x_pool_vis", "x_clip_align", "x_align"), oe):
        blob[f"e/{nm}"] = t.numpy()
    np.savez_compressed(GOLD / "stage2.npz", **blob)
    print("stage2: x_vis", tuple(blob["a/x_vis"].shape), "masked", tuple(blob["b/x_vis"].shape), "image",
          tuple(blob["c/x_vis"].shape), "early", tuple(blob["d/x_vis"].shape), "clip_align", tuple(blob["b/x_clip_align"].shape))


CLIP_T_CFG = dict(embed_dim=128, depth=3, num_heads=2, mlp_ratio=4, img_size=56, patch_size=14, init_values=0.1,
                  attn_pool_num_heads=2, clip_embed_dim=64, clip_return_layer=2, clip_return_interval=1,
                  layerscale_no_force_fp32=False, drop_path_rate=0.0)
MAE_T_CFG = dict(img_size=224, patch_size=14, embed_dim=64, depth=2, num_heads=2, mlp_ratio=4, qkv_bias=True,
                 init_values=0.0, all_frames=16, tubelet_size=2, mae_return_layer=2, mae_return_interval=1)


def make_teachers():
    """Frozen teachers + attention-guided mask (SURVEY §8f-1) at toy size, from the unmodified reference modules:
      * InternVL_CLIP (internvl_clip_vision.py:336-465, naive path): per-frame ViT, taps of the last 2 blocks with the cls
        tokens averaged over time, pooled feature, pooling attention map;
      * VideoMAE teacher VisionTransformer (videomae.py:207-313) at the recipe geometry (16 frames, tubelet 2, 16x16
        patches of 14 px -> 2048 tokens).  Its Attention calls flash_attn_func on [B,H,N,d] tensors (FA2's layout is
        [B,N,H,d]) — executed here with a CPU stand-in that does exactly what FA2 does with such inputs;
      * the mask-building statements of engine_for_pretraining.py:105-116 exec'd verbatim with torch.multinomial replaced by
        a stored permutation, and the target selection :118-125."""
    ivl, mae = ref_shim.import_teachers()
    import contextlib, io
    torch.manual_seed(8642)
    with contextlib.redirect_stdout(io.StringIO()):
        clip_t = ivl.InternVL_CLIP(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **CLIP_T_CFG).eval()
        mae_t = mae.VisionTransformer(norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), **MAE_T_CFG).eval()
    g = torch.Generator().manual_seed(23)
    with torch.no_grad():
        for model in (clip_t, mae_t):
            for name, p in model.named_parameters():
                if name == "pos_embed":
                    p.copy_(torch.randn(p.shape, generator=g) * 0.1)
                elif name.endswith("bias") or name.endswith("_bias"):
                    p.add_(torch.randn(p.shape, generator=g) * 0.05)
                elif "norm" in name and name.endswith("weight"):
                    p.add_(torch.randn(p.shape, generator=g) * 0.1)
                elif name.endswith("gamma"):
                    p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
                elif name == "cls_token":
                    p.add_(torch.randn(p.shape, generator=g) * 0.1)
                p.copy_(bf16_round(p))
    B, T = 2, 2
    clip_video = bf16_round(torch.randn(B, 3, T, 56, 56, generator=g))
    mae_video = bf16_round(torch.randn(1, 3, 16, 224, 224, generator=g))
    with torch.no_grad():
        z, x, attn = clip_t(clip_video)
        zm = mae_t(mae_video)
    # mask statements of the engine, verbatim, with the multinomial draw injected
    src = Path(ref_shim.IV2_SM, "engines", "engine_for_pretraining.py").read_text().splitlines()
    start = next(i for i, l in enumerate(src) if "BT, N = attn.shape" in l)
    end = next(i for i, l in enumerate(src) if "targets_mae_vis = norm_mae[~mae_bool_masked_pos]" in l)
    snippet = textwrap.dedent("\n".join(src[start:end + 1]))
    BT, N = attn.shape
    importance = torch.stack([torch.randperm(N, generator=g) for _ in range(BT)])

    class _T:        # torch with multinomial replaced by the stored draw
        def __getattr__(self, k):
            return (lambda a, n: importance) if k == "multinomial" else getattr(torch, k)
    norm_mae_small = torch.nn.functional.normalize(torch.randn(2, B, T * N, 24, generator=g), dim=-1)
    env = dict(torch=_T(), attn=attn, mask_ratio=0.75, mask_type="attention", B=B, norm_clip_middle=z,
               norm_clip_final=x, norm_mae=norm_mae_small, bool_masked_pos=None)
    exec(snippet, env)
    blob = {"clip_cfg": np.frombuffer(json.dumps(CLIP_T_CFG).encode(), dtype=np.uint8),
            "mae_cfg": np.frombuffer(json.dumps(MAE_T_CFG).encode(), dtype=np.uint8),
            "clip_video": clip_video.numpy(), "mae_video": mae_video.numpy().astype(np.float16),
            "z": z.numpy(), "x": x.numpy(), "attn": attn.numpy(), "zm": zm.numpy().astype(np.float16),
            "importance": importance.numpy(), "mask": env["bool_masked_pos"].numpy(),
            "norm_mae_small": norm_mae_small.numpy(),
            "targets_clip_middle_vis": env["targets_clip_middle_vis"].numpy(),
            "targets_mae_vis": env["targets_mae_vis"].numpy()}
    for k, v in clip_t.state_dict().items():
        blob["wc/" + k] = v.numpy()
    for k, v in mae_t.state_dict().items():
        blob["wm/" + k] = v.numpy()
    np.savez_compressed(GOLD / "teachers.npz", **blob)
    print("teachers: z", tuple(z.shape), "x", tuple(x.shape), "attn", tuple(attn.shape), "zm", tuple(zm.shape),
          "mask", tuple(env["bool_masked_pos"].shape), "vis", tuple(env["targets_clip_middle_vis"].shape))


def _vtc_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    crit, mutils = ref_shim.import_criterions()
    g = torch.Generator().manual_seed(100 + rank)
    Bl, Cc = 8, 64
    v = torch.randn(Bl, Cc, generator=g).requires_grad_(True)
    t = torch.randn(Bl, Cc, generator=g).requires_grad_(True)
    idx = torch.arange(rank * Bl, (rank + 1) * Bl)
    if rank == 1:
        idx[0] = 3   # duplicate of a rank-0 sample -> soft targets
        idx[5] = 3
    loss = crit.VTC_VTM_Loss(False).vtc_loss(v, t, idx, temp=0.07, all_gather=True)
    loss.backward()
    q.put((rank, v.detach().numpy(), t.detach().numpy(), idx.numpy(), float(loss),
           v.grad.numpy(), t.grad.numpy()))
    dist.barrier()
    dist.destroy_process_group()


def make_vtc():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_vtc_worker, args=(r, 2, 29731, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted([q.get() for _ in range(2)], key=lambda r: r[0])
    [p.join() for p in procs]
    blob = {"temp": np.float32(0.07)}
    for r, v, t, idx, loss, gv, gt in res:
        blob.update({f"v{r}": v, f"t{r}": t, f"idx{r}": idx, f"loss{r}": np.float32(loss),
                     f"gv{r}": gv, f"gt{r}": gt})
    np.savez_compressed(GOLD / "vtc.npz", **blob)
    print("vtc: loss per rank", [r[4] for r in res])


def make_pixel_target():
    src = Path(ref_shim.IV1_MAE, "engine_for_pretraining.py").read_text().splitlines()
    # the reference's own statements, engine_for_pretraining.py:66-98 (inside `with torch.no_grad():`)
    start = next(i for i, l in enumerate(src) if "calculate the predict label" in l)
    end = next(i for i, l in enumerate(src) if "labels = images_patch[bool_masked_pos]" in l)
    snippet = textwrap.dedent("\n".join(src[start:end + 1]))
    from einops import rearrange
    g = torch.Generator().manual_seed(5)
    images = torch.randn(2, 3, 4, 32, 32, generator=g)
    mask = torch.zeros(2, 8, dtype=torch.bool)
    mask[0, [0, 3, 4, 6]] = True
    mask[1, [1, 2, 5, 7]] = True
    env = dict(torch=torch, rearrange=rearrange, images=images, bool_masked_pos=mask,
               device=torch.device("cpu"), normlize_target=True, patch_size=16,
               IMAGENET_DEFAULT_MEAN=(0.485, 0.456, 0.406), IMAGENET_DEFAULT_STD=(0.229, 0.224, 0.225))
    exec(snippet, env)
    labels = env["labels"]
    env2 = dict(env, normlize_target=False)
    exec(snippet, env2)
    np.savez_compressed(GOLD / "pixel_target.npz", images=images.numpy(), mask=mask.numpy(),
                        labels=labels.numpy(), labels_raw=env2["labels"].numpy())
    print("pixel_target:", tuple(labels.shape))


IV1_CFG = dict(img_size=32, patch_size=16, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2,
               decoder_num_classes=1536, decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=1, mlp_ratio=4,
               qkv_bias=True, init_values=0.1, tubelet_size=2)


def make_iv1_videomae():
    """SURVEY §8 a15 / f-4: InternVideo1's VideoMAE pre-training model (modeling_pretrain.py:269-387, unmodified) at toy
    size, with the reference's own label statements (engine_for_pretraining.py:66-98) and nn.MSELoss: prediction of the
    masked tubelets, loss, gradient of every parameter."""
    mod = ref_shim.import_iv1_videomae()
    from functools import partial
    from einops import rearrange
    torch.manual_seed(4321)
    net = mod.PretrainVisionTransformer(norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), **IV1_CFG).train()
    g = torch.Generator().manual_seed(31)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.endswith("bias") or name.endswith("_bias"):
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
            elif "norm" in name and name.endswith("weight"):
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            elif "gamma" in name:
                p.mul_(1 + torch.randn(p.shape, generator=g) * 0.3)
            p.copy_(bf16_round(p))
    B, T = 3, 16
    N = net.encoder.patch_embed.num_patches                     # 2 x 2 x 8 = 32 tubelets
    images = bf16_round(torch.randn(B, 3, T, 32, 32, generator=g))
    mask = torch.zeros(B, N, dtype=torch.bool)
    for b in range(B):
        mask[b, torch.randperm(N, generator=g)[:20]] = True     # 20 masked, 12 visible per clip
    src = Path(ref_shim.IV1_MAE, "engine_for_pretraining.py").read_text().splitlines()
    start = next(i for i, l in enumerate(src) if "calculate the predict label" in l)
    end = next(i for i, l in enumerate(src) if "labels = images_patch[bool_masked_pos]" in l)
    env = dict(torch=torch, rearrange=rearrange, images=images, bool_masked_pos=mask, device=torch.device("cpu"),
               normlize_target=True, patch_size=16, IMAGENET_DEFAULT_MEAN=(0.485, 0.456, 0.406),
               IMAGENET_DEFAULT_STD=(0.229, 0.224, 0.225))
    exec(textwrap.dedent("\n".join(src[start:end + 1])), env)
    labels = env["labels"]
    out = net(images, mask)
    loss = torch.nn.MSELoss()(input=out, target=labels)
    loss.backward()
    blob = {"cfg": np.frombuffer(json.dumps(IV1_CFG).encode(), dtype=np.uint8), "images": images.numpy(),
            "mask": mask.numpy(), "labels": labels.numpy(), "out": out.detach().numpy(), "loss": loss.detach().numpy()}
    for k, t in net.state_dict().items():
        blob["w/" + k] = t.numpy()
    for k, p in net.named_parameters():
        blob["g/" + k] = p.grad.numpy() if p.grad is not None else np.zeros(tuple(p.shape), np.float32)
    with torch.no_grad():
        blob["enc_out"] = net.encoder(images, mask).numpy()
    np.savez_compressed(GOLD / "iv1_videomae.npz", **blob)
    print("iv1_videomae: out", tuple(out.shape), "loss", float(loss), "enc", tuple(blob["enc_out"].shape))


def _json(obj):
    return np.frombuffer(json.dumps(obj).encode(), dtype=np.uint8)


def seeded_state(layout, seed):
    """Seeded weights for a state_dict layout [(key, shape), ...] that is too large to store: LayerScale around 0.1,
    norm weights around 1, small biases, every other tensor N(0, 0.02).  Regenerated wherever the fixture is used."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shape in layout:
        t = torch.randn(tuple(shape), generator=g)
        if k.endswith("gamma"):
            t = 0.1 * (1 + 0.3 * t)
        elif "norm" in k and k.endswith("weight"):
            t = 1 + 0.1 * t
        elif k.endswith("bias"):
            t = 0.05 * t
        else:
            t = 0.02 * t
        sd[k] = t
    return sd


def describe_module(model, exact_max_numel=4096):
    """What code that reads hyper-parameters off a built module can see, without the module's source: per submodule its
    kind (list or not), its plain attributes, and its parameters and buffers (None where registered as None).  Tensors of
    up to `exact_max_numel` elements are stored exactly, larger ones only as a (key, shape) layout for seeded_state(layout, 0)."""
    def plain(v):
        if v is None or isinstance(v, (bool, int, float, str)):
            return True
        return isinstance(v, (list, tuple)) and all(plain(x) for x in v)

    mods, exact, layout = [], {}, []
    for name, m in model.named_modules():
        tensors = []
        for kind, store in (("p", m._parameters), ("b", m._buffers)):
            for k, t in store.items():
                full = f"{name}.{k}" if name else k
                persistent = kind == "p" or k not in m._non_persistent_buffers_set
                tensors.append([kind, k, None if t is None else list(t.shape), persistent])
                if t is None:
                    continue
                if t.numel() <= exact_max_numel:
                    exact[full] = t.detach().numpy().copy()
                else:
                    layout.append((full, list(t.shape)))
        mods.append(dict(name=name, is_list=isinstance(m, (torch.nn.ModuleList, torch.nn.Sequential)),
                         attrs={k: v for k, v in vars(m).items() if not k.startswith("_") and plain(v)}, tensors=tensors))
    return dict(modules=mods, seeded_layout=layout), exact


def sample_flat(t, n, seed):
    """A fixed, seeded sample of n elements of t (flattened), in index order."""
    flat = t.detach().reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return flat[idx]


SDIMS_CFG = dict(embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, num_frames=4, drop_path_rate=0.0,
                 clip_return_layer=1, mae_return_layer=1, attn_pool_num_heads=16, init_values=0.1)
SDIMS_SEED = 2025
FROM_REF_CFG = dict(embed_dim=176, depth=3, num_heads=2, mlp_ratio=48 / 11, num_frames=2, img_size=56, patch_size=14,
                    drop_path_rate=0.3, attn_pool_num_heads=2, clip_embed_dim=64, clip_teacher_embed_dim=96,
                    clip_teacher_final_dim=64, mae_teacher_embed_dim=176, clip_return_layer=2, mae_return_layer=2,
                    clip_student_return_interval=1, init_values=0.08)
SEP_POS_CFG = dict(sep_pos_embed=True, embed_dim=64, depth=1, num_heads=2, num_frames=2, img_size=28,
                   clip_teacher_embed_dim=32, clip_teacher_final_dim=16, mae_teacher_embed_dim=64, attn_pool_num_heads=2,
                   clip_embed_dim=16)
IV1_INIT_CFG = dict(img_size=32, patch_size=16, encoder_embed_dim=128, encoder_depth=1, encoder_num_heads=2,
                    decoder_num_classes=1536, decoder_embed_dim=64, decoder_depth=1, decoder_num_heads=1, qkv_bias=True,
                    init_values=0.1)


def sdims_inputs():
    """Input clips and mask of the InternVideo2-S restatement check (BASELINE cfg-1: 2 clips x 4 frames x 224^2)."""
    g = torch.Generator().manual_seed(SDIMS_SEED + 1)
    x = torch.randn(2, 3, 4, 224, 224, generator=g)
    g = torch.Generator().manual_seed(3)
    mask = torch.ones(2, 1 + 4 * 256, dtype=torch.bool)
    mask[:, 0] = False
    for b in range(2):
        for t in range(4):
            mask[b, 1 + t * 256 + torch.randperm(256, generator=g)[:52]] = False
    return x, mask


def make_ref_checks():
    """Small results of the unmodified reference that the CPU tests compare the project's host code against, one entry
    group per check (tests/test_masking_cpu.py, test_modules_cpu.py, test_oracle_cpu.py, test_stage2_cpu.py,
    test_videomae_v1_cpu.py).  Inputs are regenerated from the same seeds in the tests."""
    import contextlib, hashlib, importlib, io, types
    import importlib.util
    blob = {}

    def load(path, name):
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    # batch mask generators (multi_modality/models/mask.py) under fixed numpy seeds
    mm_mask = load(os.path.join(ref_shim.IV2_MM, "models", "mask.py"), "_ivref_mm_mask")
    for i, (size, ratio, B) in enumerate((((8, 16, 16), 0.8, 4), ((1, 14, 14), 0.5, 3), ((4, 16, 16), 0.9, 2))):
        np.random.seed(11); blob[f"mask/tube{i}"] = mm_mask.TubeMaskingGenerator(size, ratio, B, device="cpu").numpy()
        np.random.seed(12); blob[f"mask/random{i}"] = mm_mask.RandomMaskingGenerator(size, ratio, B, device="cpu").numpy()
    # per-clip mask generators (single_modality/datasets/masking_generator.py)
    sm_mask = load(os.path.join(ref_shim.IV2_SM, "datasets", "masking_generator.py"), "_ivref_sm_maskgen")
    for i, (size, ratio) in enumerate((((8, 14, 14), 0.9), ((4, 16, 16), 0.8))):
        np.random.seed(5); blob[f"clipmask/tube{i}"] = np.stack([sm_mask.TubeMaskingGenerator(size, ratio)() for _ in range(3)])
        blob[f"clipmask/tube_repr{i}"] = _json(repr(sm_mask.TubeMaskingGenerator(size, ratio)))
        np.random.seed(6); blob[f"clipmask/random{i}"] = np.stack([sm_mask.RandomMaskingGenerator(size, ratio)() for _ in range(3)])

    # 3-D sin-cos table, separable position tables and pos-embed interpolation
    sm = ref_shim.import_single_modality()
    blob["pos/sincos_64_4_2_cls"] = np.asarray(sm.get_3d_sincos_pos_embed(64, 4, 2, cls_token=True))
    ref = ref_shim.build_reference_model(**SEP_POS_CFG)
    rs = ref.state_dict()
    blob["seppos/keys"] = _json(list(rs))
    for k, t in rs.items():
        if "pos_embed" in k:
            blob["seppos/" + k] = t.numpy()
    ref_shim.import_clip_vision()
    pe = importlib.import_module("_ivref_mm_backbone.pos_embed")
    from internvideo_b200.clip_modules import InternVideo2
    tower = InternVideo2(embed_dim=64, depth=1, num_heads=2, num_frames=8, img_size=112, attn_pool_num_heads=2,
                         clip_embed_dim=16, use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False)
    ck = {"vision_encoder.pos_embed": torch.randn(1, 1 + 4 * 16, 64, generator=torch.Generator().manual_seed(0))}
    with contextlib.redirect_stdout(io.StringIO()):
        pe.interpolate_pos_embed(ck, tower, orig_t_size=4)
    out = ck["vision_encoder.pos_embed"]
    blob["interp/shape"] = np.asarray(out.shape, dtype=np.int64)
    blob["interp/sample"], blob["interp/norm"] = sample_flat(out, 4096, 99).numpy(), np.float64(out.double().norm())

    # a reference-built PretrainInternVideo2 as patch.from_reference sees it
    desc, exact = describe_module(ref_shim.build_reference_model(**FROM_REF_CFG).train())
    blob["fromref/desc"] = _json(desc)
    for k, t in exact.items():
        blob["fromref/t/" + k] = t

    # InternVideo2-S student forward (naive path, fp32) on seeded weights: a seeded sample of every output + its norm
    model = ref_shim.build_reference_model(**SDIMS_CFG).eval()
    layout = [(k, list(t.shape)) for k, t in model.state_dict().items()]
    model.load_state_dict(seeded_state(layout, SDIMS_SEED), strict=True)
    x, mask = sdims_inputs()
    with torch.no_grad():
        outs = model(x, mask)
    blob["sdims/layout"] = _json(layout)
    for i, o in enumerate(outs):
        blob[f"sdims/shape{i}"] = np.asarray(o.shape, dtype=np.int64)
        blob[f"sdims/sample{i}"] = sample_flat(o, 4096, 100 + i).numpy()
        blob[f"sdims/norm{i}"] = np.float64(o.double().norm())

    # stage-2 criterions: the triplets vtm_loss hands its fusion encoder, uta_loss, get_sim
    crit, _ = ref_shim.import_criterions()
    for hard in (True, False):
        g = torch.Generator().manual_seed(3)
        B, Lv, Lt, C = 12, 5, 4, 16
        vis = torch.randn(B, Lv, C, generator=g); txt = torch.randn(B, Lt, C, generator=g)
        vp = torch.randn(B, C, generator=g); tp = torch.randn(B, C, generator=g)
        atts = (torch.rand(B, Lt, generator=g) > 0.3).long()
        idx = torch.arange(B); idx[7] = 2
        seen = {}

        def encoder(encoder_embeds, attention_mask, encoder_hidden_states, encoder_attention_mask, return_dict, mode):
            seen.update(text=encoder_embeds, atts=attention_mask, vision=encoder_hidden_states)
            return types.SimpleNamespace(last_hidden_state=encoder_embeds)

        head = torch.nn.Linear(C, 2)
        torch.manual_seed(77)
        crit.VTC_VTM_Loss(hard).vtm_loss(encoder, head, 0.07, vis, txt, vp, tp, atts, idx)
        for k, t in seen.items():
            blob[f"vtm/{int(hard)}/{k}"] = t.detach().numpy()
    g = torch.Generator().manual_seed(9)
    s = torch.randn(2, 3, 7, 20, generator=g); c = torch.randn(2, 3, 7, 20, generator=g)
    for norm in ("l2", "none"):
        for kind in ("l2", "mse", "smooth_l1"):
            blob[f"uta/{norm}/{kind}"] = crit.UTA_Loss(norm, kind).uta_loss(s, c).numpy()
    v = torch.randn(6, 16, generator=g); t = torch.randn(5, 16, generator=g)
    blob["sim/2d/v2t"], blob["sim/2d/t2v"] = (a.numpy() for a in crit.get_sim(v, t, 0.07))
    v3 = torch.randn(6, 4, 16, generator=g)
    for agg in ("mean", "max"):
        blob[f"sim/v3/{agg}/v2t"], blob[f"sim/v3/{agg}/t2v"] = (a.numpy() for a in crit.get_sim(v3, t, 0.07, agg))
    t3 = torch.randn(5, 3, 16, generator=g)
    for agg in ("mean", "max"):
        blob[f"sim/t3/{agg}/v2t"], blob[f"sim/t3/{agg}/t2v"] = (a.numpy() for a in crit.get_sim(v, t3, 0.07, agg))
    # recall@k of tasks_clip/retrieval_utils.py::itm_eval (the function alone: its module imports the whole project)
    path = os.path.join(ref_shim.IV2_MM, "tasks_clip", "retrieval_utils.py")
    src = open(path).read()
    start = src.index("def itm_eval(")
    ns = {"np": np}
    exec(compile(src[start:src.index("\n\n\n", start)] if "\n\n\n" in src[start:] else src[start:], path, "exec"), ns)
    rg = np.random.default_rng(4)
    s = rg.standard_normal((9, 13)).astype(np.float32)
    txt2img = [int(x) for x in rg.integers(0, 9, 13)]
    img2txt = [[j for j in range(13) if txt2img[j] == i] or [0] for i in range(9)]
    blob["itm_eval"] = _json({k: float(v) for k, v in ns["itm_eval"](s, s.T.copy(), txt2img, img2txt).items()})

    # InternVideo1 VideoMAE: fixed sinusoid tables, key order, and a digest of every initial tensor under one seed
    iv1 = ref_shim.import_iv1_videomae()
    torch.manual_seed(3)
    net = iv1.PretrainVisionTransformer(**IV1_INIT_CFG)
    blob["iv1/pos_embed"] = net.pos_embed.numpy()
    blob["iv1/encoder_pos_embed"] = net.encoder.pos_embed.numpy()
    blob["iv1/init_sha256"] = _json([[k, list(t.shape), hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()]
                                     for k, t in net.state_dict().items()])

    np.savez_compressed(GOLD / "ref_checks.npz", **blob)
    print("ref_checks:", len(blob), "entries,", os.path.getsize(GOLD / "ref_checks.npz"), "bytes")


if __name__ == "__main__":
    assert ref_shim.available(), "reference not mounted"
    GOLD.mkdir(parents=True, exist_ok=True)
    which = sys.argv[1:] or ["pretrain_tiny", "pretrain_d88", "pretrain_dp", "block_cfg2", "clip_small", "teachers", "vtc",
                             "pixel_target", "stage2", "iv1_videomae", "ref_checks"]
    makers = {"pretrain_tiny": make_pretrain_tiny, "pretrain_d88": make_pretrain_d88, "vtc": make_vtc,
              "pixel_target": make_pixel_target, "pretrain_dp": make_pretrain_dp, "block_cfg2": make_block_cfg2,
              "clip_small": make_clip_small, "teachers": make_teachers, "stage2": make_stage2, "iv1_videomae": make_iv1_videomae,
              "ref_checks": make_ref_checks}
    for w in which:      # e.g. `python oracle/make_golden.py pretrain_d88` regenerates one fixture only
        makers[w]()
