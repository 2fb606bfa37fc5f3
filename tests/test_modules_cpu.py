"""Host-side contract of the nn.Module mirror: state_dict keys == the reference's, ctor kwargs accepted,
and no CPU execution path (cfg-1 plumbing: the oracle runs on CPU, the product refuses to).  What the reference computed
for these checks is stored in tests/golden/ref_checks.npz (oracle/make_golden.py::make_ref_checks)."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from internvideo_b200 import _lib
from internvideo_b200.modules import PretrainInternVideo2, get_3d_sincos_pos_embed
from oracle.make_golden import FROM_REF_CFG, SEP_POS_CFG, sample_flat, seeded_state

GOLD = Path(__file__).parent / "golden"
REF = np.load(GOLD / "ref_checks.npz")


def test_state_dict_keys_match_reference_golden():
    z = np.load(GOLD / "pretrain_tiny.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    ref_keys = {k[2:]: z[k].shape for k in z.files if k.startswith("w/")}
    model = PretrainInternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **cfg)
    sd = model.state_dict()
    assert set(sd.keys()) == set(ref_keys.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(ref_keys[k]), k
    model.load_state_dict({k: torch.from_numpy(z["w/" + k]) for k in ref_keys}, strict=True)


def test_no_cpu_execution_path():
    z = np.load(GOLD / "pretrain_tiny.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    model = PretrainInternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **cfg).bfloat16()
    with pytest.raises(_lib.IvbError):
        model(torch.from_numpy(z["x"]).to(torch.bfloat16), torch.from_numpy(z["mask"]))


def test_init_matches_reference_init_statistics():
    ref = REF["pos/sincos_64_4_2_cls"]
    assert np.allclose(get_3d_sincos_pos_embed(64, 4, 2, cls_token=True), ref, atol=1e-6)


def test_clip_tower_state_dict_keys_match_reference_golden():
    """InternVideo2 (unmasked tower) + InternVideo2_CLIP_small: key set / shapes == the instantiated reference's
    (tests/golden/clip_small.npz stores the reference state_dict), strict load works."""
    from internvideo_b200.clip_modules import InternVideo2, InternVideo2_CLIP_small
    z = np.load(GOLD / "clip_small.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    align_dim = cfg.pop("align_dim")
    ref = {k[len("w/vision_encoder."):]: z[k].shape for k in z.files if k.startswith("w/vision_encoder.")}
    tower = InternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **cfg)
    sd = tower.state_dict()
    assert set(sd) == set(ref)
    assert all(tuple(sd[k].shape) == tuple(ref[k]) for k in sd)
    ve = dict(cfg, align_dim=align_dim, use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False)
    wrap = InternVideo2_CLIP_small(dict(model=dict(vision_encoder=ve, temp=0.01, temp_min=0.01, freeze_vision=True,
                                                   open_vision_clip_projector=True, freeze_text=True)))
    want = {k[2:] for k in z.files if k.startswith("w/")} | {"temp"}
    assert set(wrap.state_dict()) == want
    # freezing: only the attention-pooling projector, vision_align and temp train (scripts/pretraining/clip/L14/config.py)
    trainable = {n for n, p in wrap.named_parameters() if p.requires_grad}
    assert all(n.startswith(("vision_encoder.clip_projector", "vision_align", "temp")) for n in trainable) and "temp" in trainable
    assert wrap.no_weight_decay() >= {"temp", "vision_encoder.pos_embed", "vision_encoder.cls_token"}


def test_stage1_checkpoint_remap_and_sep_pos_embed_keys():
    """Checkpoint interop (internvideo2_clip_small.py:207-231): a stage-1 PretrainInternVideo2 state_dict wrapped the
    DeepSpeed way ({'module': ...}) loads into the CLIP wrapper's tower: decoders and decoder position tables are
    dropped, every tower key is prefixed.  sep_pos_embed=True exposes the reference's separable tables."""
    from internvideo_b200.clip_modules import InternVideo2_CLIP_small, remap_vision_checkpoint
    z = np.load(GOLD / "pretrain_tiny.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    stage1 = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w/")}
    ve = dict(embed_dim=cfg["embed_dim"], depth=cfg["depth"], num_heads=cfg["num_heads"], mlp_ratio=cfg["mlp_ratio"],
              num_frames=cfg["num_frames"], img_size=cfg["img_size"], patch_size=cfg["patch_size"], drop_path_rate=0.0,
              attn_pool_num_heads=cfg["attn_pool_num_heads"], clip_embed_dim=cfg["clip_embed_dim"],
              init_values=cfg["init_values"], align_dim=32, use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False)
    wrap = InternVideo2_CLIP_small(dict(model=dict(vision_encoder=ve, temp=0.01, temp_min=0.01)))
    new = remap_vision_checkpoint({"module": stage1}, wrap.vision_encoder)
    assert not any("decoder" in k or "clip_pos_embed" in k or "mae_pos_embed" in k for k in new)
    msg = wrap.load_state_dict(new, strict=False)
    assert not msg.unexpected_keys and all(k.startswith(("vision_align", "temp")) for k in msg.missing_keys)
    assert torch.equal(wrap.vision_encoder.blocks[1].mlp.fc2.weight, stage1["blocks.1.mlp.fc2.weight"])
    m = PretrainInternVideo2(sep_pos_embed=True, embed_dim=64, depth=1, num_heads=2, num_frames=2, img_size=28,
                             clip_teacher_embed_dim=32, clip_teacher_final_dim=16, mae_teacher_embed_dim=64,
                             attn_pool_num_heads=2, clip_embed_dim=16, use_flash_attn=False, use_fused_rmsnorm=False,
                             use_fused_mlp=False)
    keys = set(m.state_dict())
    assert {"pos_embed_spatial", "pos_embed_temporal", "pos_embed_cls", "clip_pos_embed_spatial", "clip_pos_embed_temporal",
            "clip_pos_embed_cls", "mae_pos_embed_spatial", "mae_pos_embed_temporal"} <= keys and "pos_embed" not in keys
    assert tuple(m._pos_table("").shape) == (1, 1 + 2 * 4, 64) and tuple(m._pos_table("mae_").shape) == (1, 8, 64)


def test_sep_pos_embed_and_interpolation_match_reference():
    """sep_pos_embed: same keys and the same initial separable tables as the reference model; pos-embed interpolation
    (4 -> 8 frames, 4x4 -> 8x8 grid) equals the reference's interpolate_pos_embed (pos_embed.py:137-182) on a seeded
    sample of its output and in norm."""
    from internvideo_b200.clip_modules import InternVideo2, interpolate_pos_embed
    ours = PretrainInternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **SEP_POS_CFG)
    rs_keys, os_ = json.loads(bytes(REF["seppos/keys"]).decode()), ours.state_dict()
    assert set(rs_keys) == set(os_)
    for k in rs_keys:
        if "pos_embed" in k:
            assert torch.allclose(torch.from_numpy(REF["seppos/" + k]), os_[k], atol=1e-6), k
    tower = InternVideo2(embed_dim=64, depth=1, num_heads=2, num_frames=8, img_size=112, attn_pool_num_heads=2,
                         clip_embed_dim=16, use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False)
    g = torch.Generator().manual_seed(0)
    b = {"vision_encoder.pos_embed": torch.randn(1, 1 + 4 * 16, 64, generator=g)}
    interpolate_pos_embed(b, tower, orig_t_size=4)
    out = b["vision_encoder.pos_embed"]
    assert tuple(REF["interp/shape"]) == out.shape == (1, 1 + 8 * 64, 64)
    assert torch.allclose(torch.from_numpy(REF["interp/sample"]), sample_flat(out, 4096, 99), atol=1e-6)
    assert abs(float(out.double().norm()) - float(REF["interp/norm"])) < 1e-6 * float(REF["interp/norm"])


def _reference_built_model():
    """The reference-built PretrainInternVideo2 of FROM_REF_CFG as stored by oracle/make_golden.py::describe_module: the
    same module tree, plain attributes, parameters and buffers (small tensors exact, large ones regenerated from the
    seeded layout; from_reference copies whatever values they hold)."""
    desc = json.loads(bytes(REF["fromref/desc"]).decode())
    seeded = seeded_state(desc["seeded_layout"], 0)
    mods = {}
    for d in desc["modules"]:
        m = torch.nn.ModuleList() if d["is_list"] else torch.nn.Module()
        for k, v in d["attrs"].items():
            setattr(m, k, v)
        for kind, k, shape, persistent in d["tensors"]:
            full = f"{d['name']}.{k}" if d["name"] else k
            t = None if shape is None else torch.from_numpy(REF["fromref/t/" + full]) if "fromref/t/" + full in REF \
                else seeded[full]
            if kind == "p":
                m.register_parameter(k, None if t is None else torch.nn.Parameter(t, requires_grad=False))
            else:
                m.register_buffer(k, t, persistent=persistent)
        if d["name"]:
            parent, _, leaf = d["name"].rpartition(".")
            mods[parent].add_module(leaf, m)
        mods[d["name"]] = m
    return mods[""]


def test_from_reference_rebuilds_config_and_weights():
    """patch.from_reference: hyper-parameters are read off a reference-BUILT model and the weights load strictly."""
    from internvideo_b200 import patch
    kw = FROM_REF_CFG
    ref = _reference_built_model()
    cfg = patch.reference_config(ref)
    for k in ("embed_dim", "depth", "num_heads", "num_frames", "img_size", "patch_size", "attn_pool_num_heads",
              "clip_embed_dim", "clip_teacher_embed_dim", "clip_teacher_final_dim", "mae_teacher_embed_dim",
              "clip_return_layer", "mae_return_layer"):
        assert cfg[k] == kw[k], k
    assert abs(cfg["mlp_ratio"] - kw["mlp_ratio"]) < 1e-2 and abs(cfg["drop_path_rate"] - 0.3) < 1e-6
    ours = patch.from_reference(ref, dtype=torch.float32, device=None)
    assert ours.training and ours.clip_return_index == ref.clip_return_index and ours.mae_return_index == ref.mae_return_index
    rs, os_ = ref.state_dict(), ours.state_dict()
    assert set(rs) == set(os_) and all(torch.equal(rs[k], os_[k]) for k in rs)
    assert [b.drop_path1.drop_prob if hasattr(b.drop_path1, "drop_prob") else 0.0 for b in ours.blocks] == \
           pytest.approx([getattr(b.drop_path1, "drop_prob", 0.0) for b in ref.blocks])
    # the attention seam refuses what the pre-training path never uses, like the reference's asserts do
    fa = patch.FlashAttention(attention_dropout=0.0)
    with pytest.raises(AssertionError):
        fa(torch.zeros(1, 4, 3, 2, 8))                      # fp32 / CPU
