"""Shared helpers for the parity tests (the oracle is imported here as the checker only)."""
import hashlib
from pathlib import Path

import numpy as np
import torch

BF16 = torch.bfloat16


def load_image_golden() -> dict:
    """tests/golden/image_golden.npz with every input image rebuilt from its stored (h, w, k) test-card recipe
    (`<key>_card`) and checked against the digest of the card the outputs were minted from (`<key>_sha256`)."""
    from oracle.image_oracle import card
    g = dict(np.load(Path(__file__).resolve().parent / "golden" / "image_golden.npz"))
    for key in [k[: -len("_card")] for k in g if k.endswith("_card")]:
        img = card(*g.pop(key + "_card").tolist())
        assert hashlib.sha256(img.tobytes()).hexdigest() == str(g.pop(key + "_sha256")), f"{key}: test card differs"
        g[key] = img
    return g


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(BF16).to(torch.float32)


def randn(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return bf16_round(torch.randn(shape, generator=g) * scale)


def to_dev(t: torch.Tensor) -> torch.Tensor:
    return t.to(device="cuda", dtype=BF16).contiguous()


def assert_close(got: torch.Tensor, want: torch.Tensor, rel=1.6e-2, what=""):
    """bf16 tolerance: max |got - want| <= rel * max|want| (fp32 accumulate, one or two bf16 roundings)."""
    got = got.detach().float().cpu()
    want = want.detach().float().cpu()
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    assert torch.isfinite(got).all(), f"{what}: non-finite values"
    err = (got - want).abs().max().item()
    ref = want.abs().max().item()
    assert err <= rel * max(ref, 1e-6), f"{what}: max err {err:.4e} vs max|ref| {ref:.4e} (rel {err / max(ref, 1e-6):.3e})"
    return err / max(ref, 1e-6)
