"""internvideo_b200/masking.py against the reference generators under the same numpy seed (bit-exact; their masks are
stored in tests/golden/ref_checks.npz, oracle/make_golden.py::make_ref_checks), and the structural properties the student
relies on (fixed number of visible tokens per clip, tube = same spatial mask in every frame)."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from internvideo_b200 import masking

REF = np.load(Path(__file__).parent / "golden" / "ref_checks.npz")


def test_tube_and_random_structure():
    np.random.seed(0)
    m = masking.tube_mask((4, 16, 16), 0.8, 3, device="cpu")
    assert m.shape == (3, 4 * 256) and m.dtype == torch.bool
    f = m.view(3, 4, 256)
    assert (f == f[:, :1]).all()                                   # the same spatial mask in every frame
    assert (f[:, 0].sum(1) == int(0.8 * 256)).all()
    r = masking.random_mask((4, 16, 16), 0.8, 3, device="cpu")
    assert (r.sum(1) == int(0.8 * 1024)).all()
    s = masking.student_mask("tube", (4, 16, 16), 0.8, 3, device="cpu")
    assert s.shape == (3, 1 + 1024) and not s[:, 0].any()          # cls visible
    assert masking.student_mask("none", (4, 16, 16), 0.8, 3, device="cpu") is None
    with pytest.raises(NotImplementedError):
        masking.student_mask("block", (4, 16, 16), 0.8, 3, device="cpu")


def test_attention_mask_keeps_the_injected_draw():
    B, T, N = 2, 3, 16
    g = torch.Generator().manual_seed(1)
    attn = torch.rand(B * T, N, generator=g)
    imp = torch.stack([torch.randperm(N, generator=g) for _ in range(B * T)])
    m = masking.student_mask("attention", None, 0.75, B, device="cpu", attn=attn, importance=imp)
    assert m.shape == (B, 1 + T * N) and not m[:, 0].any()
    vis = (~m[:, 1:]).view(B * T, N)
    assert (vis.sum(1) == N - int(N * 0.75)).all()
    for r in range(B * T):
        assert set(torch.nonzero(vis[r]).flatten().tolist()) == set(imp[r, :N - int(N * 0.75)].tolist())


def test_batch_generators_match_reference_bit_exact():
    for i, (size, ratio, B) in enumerate((((8, 16, 16), 0.8, 4), ((1, 14, 14), 0.5, 3), ((4, 16, 16), 0.9, 2))):
        np.random.seed(11); b = masking.tube_mask(size, ratio, B, device="cpu")
        assert torch.equal(torch.from_numpy(REF[f"mask/tube{i}"]), b)
        np.random.seed(12); b = masking.random_mask(size, ratio, B, device="cpu")
        assert torch.equal(torch.from_numpy(REF[f"mask/random{i}"]), b)


def test_clip_generators_match_reference_bit_exact():
    for i, (size, ratio) in enumerate((((8, 14, 14), 0.9), ((4, 16, 16), 0.8))):
        np.random.seed(5); g = masking.TubeMaskingGenerator(size, ratio); b = [g() for _ in range(3)]
        a = REF[f"clipmask/tube{i}"]
        assert len(a) == 3 and all(np.array_equal(x, y) for x, y in zip(a, b))
        assert json.loads(bytes(REF[f"clipmask/tube_repr{i}"]).decode()) == repr(g)
        np.random.seed(6); g = masking.RandomMaskingGenerator(size, ratio); b = [g() for _ in range(3)]
        a = REF[f"clipmask/random{i}"]
        assert len(a) == 3 and all(np.array_equal(x, y) for x, y in zip(a, b))
