"""Host logic of internvideo_b200/stage2.py (no kernels): the hard-negative sampler of the video-text matching loss, the
unmasked-teacher alignment loss, dual-softmax retrieval scores and recall@k — against what the unmodified reference
functions return for the same inputs (tests/golden/ref_checks.npz, oracle/make_golden.py::make_ref_checks) and against
hand-checked cases."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from internvideo_b200 import stage2

REF = np.load(Path(__file__).parent / "golden" / "ref_checks.npz")


def test_state_dict_keys_match_reference_tower():
    """No MAE branch, optional image tables — the key set of multi_modality/.../internvideo2.py (golden fixture keys)."""
    import json
    from pathlib import Path
    z = np.load(Path(__file__).parent / "golden" / "stage2.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    m = stage2.PretrainInternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, **cfg)
    ref_keys = {k[2:] for k in z.files if k.startswith("w/")}
    assert set(m.state_dict().keys()) == ref_keys
    m2 = stage2.PretrainInternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False,
                                     sep_image_video_pos_embed=True, **cfg)
    assert set(m2.state_dict().keys()) == ref_keys | {"img_pos_embed", "clip_img_pos_embed"}
    assert m2.img_pos_embed.shape == (1, 17, cfg["embed_dim"])
    with pytest.raises(Exception):
        m(torch.zeros(1, 3, 2, 56, 56))            # CPU input / fp32 parameters: no CPU path


def test_vtm_negatives_never_pick_positives():
    g = torch.Generator().manual_seed(0)
    sim = torch.randn(16, 16, generator=g)
    idx = torch.tensor([0, 1, 2, 3, 0, 5, 6, 7, 8, 9, 10, 11, 12, 3, 14, 15])
    for hard in (True, False):
        torch.manual_seed(1)
        vneg, tneg = stage2.vtm_negatives(sim, sim.T.contiguous(), idx, hard=hard)
        assert vneg.shape == tneg.shape == (16,)
        assert (idx[vneg] != idx).all() and (idx[tneg] != idx).all()
    vneg, tneg = stage2.vtm_negatives(sim, sim.T.contiguous(), None, hard=True)
    assert (vneg != torch.arange(16)).all() and (tneg != torch.arange(16)).all()


@pytest.mark.parametrize("hard", [True, False])
def test_vtm_negatives_match_reference_draws(hard):
    """Same RNG state -> the reference's vtm_loss hands its fusion encoder exactly the triplets built here."""
    g = torch.Generator().manual_seed(3)
    B, Lv, Lt, C = 12, 5, 4, 16
    vis = torch.randn(B, Lv, C, generator=g); txt = torch.randn(B, Lt, C, generator=g)
    vp = torch.randn(B, C, generator=g); tp = torch.randn(B, C, generator=g)
    atts = (torch.rand(B, Lt, generator=g) > 0.3).long()
    idx = torch.arange(B); idx[7] = 2
    seen = {k: torch.from_numpy(REF[f"vtm/{int(hard)}/{k}"]) for k in ("text", "atts", "vision")}
    torch.manual_seed(77)
    sim_v2t, sim_t2v = stage2.get_sim(vp, tp, 0.07)
    vneg, tneg = stage2.vtm_negatives(sim_v2t, sim_t2v, idx, hard=hard)
    vision_all, text_all, atts_all, labels = stage2.vtm_triplets(vis, txt, atts, vneg, tneg)
    assert torch.equal(vision_all, seen["vision"]) and torch.equal(text_all, seen["text"]) and torch.equal(atts_all, seen["atts"])
    assert labels.tolist() == [1] * B + [0] * (2 * B)


def test_uta_loss_and_get_sim_match_reference():
    def ref(key):
        return torch.from_numpy(REF[key])

    def ref_sim(key):
        return ref(key + "/v2t"), ref(key + "/t2v")

    g = torch.Generator().manual_seed(9)
    s = torch.randn(2, 3, 7, 20, generator=g); c = torch.randn(2, 3, 7, 20, generator=g)
    for norm in ("l2", "none"):
        for kind in ("l2", "mse", "smooth_l1"):
            got = stage2.UTA_Loss(norm, kind).uta_loss(s, c)
            assert torch.allclose(ref(f"uta/{norm}/{kind}"), got, rtol=1e-6, atol=1e-7), (norm, kind)
    v = torch.randn(6, 16, generator=g); t = torch.randn(5, 16, generator=g)
    for a, b in zip(ref_sim("sim/2d"), stage2.get_sim(v, t, 0.07)):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)
    v3 = torch.randn(6, 4, 16, generator=g)
    for agg in ("mean", "max"):
        for a, b in zip(ref_sim(f"sim/v3/{agg}"), stage2.get_sim(v3, t, 0.07, agg)):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)
    t3 = torch.randn(5, 3, 16, generator=g)
    for agg in ("mean", "max"):
        for a, b in zip(ref_sim(f"sim/t3/{agg}"), stage2.get_sim(v, t3, 0.07, agg)):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)


def test_retrieval_scores_and_recall():
    # 4 videos, 6 captions: captions 2k, 2k+1 describe video k for k < 2; videos 2, 3 have one caption each
    v = torch.eye(4, 8)
    t = torch.zeros(6, 8)
    owner = [0, 0, 1, 1, 2, 3]
    for j, k in enumerate(owner):
        t[j, k] = 1.0
        t[j, 4 + (j % 4)] = 0.3
    dsl, dsl_t, i2t, t2i = stage2.retrieval_scores(v, t)
    assert i2t.shape == (4, 6) and t2i.shape == (6, 4) and torch.equal(t2i, i2t.T)
    assert torch.allclose(dsl, i2t * i2t.softmax(dim=0)) and torch.allclose(dsl_t, i2t.T * i2t.T.softmax(dim=0))
    img2txt = [[0, 1], [2, 3], 4, 5]
    r = stage2.recall_at_k(i2t, t2i, owner, img2txt)
    assert r["txt_r1"] == 100.0 and r["img_r1"] == 100.0 and r["r_mean"] == 100.0
    bad = i2t.clone(); bad[0] = bad[0].flip(0)       # video 0 now prefers the wrong captions
    r = stage2.recall_at_k(bad, bad.T, owner, img2txt)
    assert r["txt_r1"] == 75.0
    s = torch.tensor([[1.0, 2.0], [3.0, 0.0]])
    assert torch.equal(stage2.ensemble_clip_scores(s, "mean"), torch.tensor([2.0, 1.0]))
    assert torch.equal(stage2.ensemble_clip_scores(s, "max"), torch.tensor([3.0, 2.0]))
    assert torch.allclose(stage2.ensemble_clip_scores(s, "lse"), torch.logsumexp(s, 0))
    with pytest.raises(ValueError):
        stage2.ensemble_clip_scores(s, "median")


def test_recall_matches_reference_itm_eval():
    g = np.random.default_rng(4)
    s = g.standard_normal((9, 13)).astype(np.float32)
    txt2img = [int(x) for x in g.integers(0, 9, 13)]
    img2txt = [[j for j in range(13) if txt2img[j] == i] or [0] for i in range(9)]
    ref = json.loads(bytes(REF["itm_eval"]).decode())
    got = stage2.recall_at_k(torch.from_numpy(s), torch.from_numpy(s.T.copy()), txt2img, img2txt)
    assert ref == got
