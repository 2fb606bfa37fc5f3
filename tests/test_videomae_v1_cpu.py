"""Host side of internvideo_b200/videomae_v1.py: constructor surface, state_dict keys and the fixed sinusoid tables of the
InternVideo1 VideoMAE model against the reference module (tables and initial-tensor digests stored in
tests/golden/ref_checks.npz) and the committed golden fixture."""
import hashlib
import json
from functools import partial
from pathlib import Path

import numpy as np
import pytest
import torch

from internvideo_b200 import videomae_v1 as v1
from oracle.make_golden import IV1_INIT_CFG

GOLD = Path(__file__).parent / "golden"


def test_state_dict_keys_match_the_golden_fixture():
    z = np.load(GOLD / "iv1_videomae.npz")
    cfg = json.loads(bytes(z["cfg"]).decode())
    m = v1.PretrainVisionTransformer(norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), **cfg)
    assert set(m.state_dict()) == {k[2:] for k in z.files if k.startswith("w/")}
    assert m.encoder.patch_embed.num_patches == 32 and tuple(m.pos_embed.shape) == (1, 32, cfg["decoder_embed_dim"])
    assert not isinstance(m.pos_embed, torch.nn.Parameter)          # fixed table, like the reference
    with pytest.raises(Exception):
        m(torch.zeros(1, 3, 16, 32, 32), torch.zeros(1, 32, dtype=torch.bool))     # fp32 / CPU: no CPU path


def test_factories_have_the_published_sizes():
    for fn, enc, dec, p in ((v1.pretrain_mae_small_patch16_224, 384, 192, 16), (v1.pretrain_mae_base_patch16_224, 768, 384, 16)):
        m = fn(decoder_depth=4)
        assert m.encoder.embed_dim == enc and m.decoder.embed_dim == dec and m.decoder.num_classes == 3 * 2 * p * p
        assert m.encoder.blocks[0].attn.q_bias is not None and m.encoder.blocks[0].gamma_1 is None
        assert m.encoder.patch_embed.num_patches == 14 * 14 * 8


def test_tables_and_init_match_reference():
    ref = np.load(GOLD / "ref_checks.npz")
    torch.manual_seed(3); mine = v1.PretrainVisionTransformer(**IV1_INIT_CFG)
    assert torch.equal(torch.from_numpy(ref["iv1/pos_embed"]), mine.pos_embed)
    assert torch.equal(torch.from_numpy(ref["iv1/encoder_pos_embed"]), mine.encoder.pos_embed)
    sd_r, sd_m = json.loads(bytes(ref["iv1/init_sha256"]).decode()), mine.state_dict()
    assert [k for k, _, _ in sd_r] == list(sd_m)                  # same keys in the same registration order
    for k, shape, digest in sd_r:                                 # same init draws (xavier / trunc-normal under one seed)
        assert tuple(shape) == tuple(sd_m[k].shape), k
        if "mask_token" not in k:
            assert hashlib.sha256(sd_m[k].contiguous().numpy().tobytes()).hexdigest() == digest, k
    assert float(mine.mask_token.abs().max()) <= 0.02 + 1e-6
