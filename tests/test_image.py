"""Image front end, CPU side: the numpy restatement of Pillow's 8-bit bicubic resampler + the reference's tiling + the
CLIP normalisation (oracle/image_oracle.py) against the golden digests minted from the reference's own
`dynamic_preprocess`, Pillow and transformers (oracle/make_golden_image.py) -- bit for bit -- and the host-side
coefficient tables / lookup table of vita_b200.image_frontend against the oracle's."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import image_oracle as O
from tests.util import load_image_golden

GOLD = load_image_golden()
CASES = ["wide", "tall", "square", "tiny", "pano"]


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_reference_tiles_and_pixels(name):
    img = GOLD[name + "_image"]
    tiles = O.dynamic_preprocess(img)
    assert tiles.shape[0] == int(GOLD[name + "_n_tiles"])
    assert np.array_equal(tiles[0, :32, :32], GOLD[name + "_tile0_crop"])
    assert sha(tiles) == str(GOLD[name + "_tiles_sha256"]), "uint8 tiles differ from Pillow / the reference's tiling"
    px = torch.from_numpy(O.normalize_tiles(tiles)).to(torch.bfloat16)
    assert sha(px.view(torch.int16).numpy()) == str(GOLD[name + "_pixels_bf16_sha256"])


def test_grid_choice_matches_reference_cases():
    # (width, height) -> (columns, rows) as find_closest_aspect_ratio returns them (golden run)
    assert O.closest_grid(500, 300) == (3, 2)
    assert O.closest_grid(700, 1000) == (2, 3)
    assert O.closest_grid(448, 448) == (1, 1)
    assert O.closest_grid(2400, 600) == (4, 1)
    assert O.closest_grid(333, 901) == (2, 5)


def test_frontend_tables_equal_the_oracle():
    from vita_b200 import image_frontend as I
    for in_size, out_size in [(500, 1344), (300, 896), (901, 2240), (37, 896), (3000, 448), (448, 449), (1900, 1792)]:
        ksize, bounds, kk = O.precompute_coeffs(in_size, out_size)
        k2, b2, kk2 = I.resample_tables(in_size, out_size)
        assert k2 == ksize
        assert np.array_equal(b2, bounds.astype(np.int32)) and np.array_equal(kk2, kk.astype(np.int32)), (in_size, out_size)
    for w, h in [(500, 300), (700, 1000), (448, 448), (2400, 600), (333, 901), (61, 37), (950, 120)]:
        assert I.closest_grid(w, h) == O.closest_grid(w, h)
    lut = I.normalize_lut()                         # [3, 256] bf16
    assert np.array_equal(lut.view(torch.int16).numpy(), GOLD["lut_bf16_bits"])


FRAMES = ["landscape", "portrait", "sq"]


@pytest.mark.parametrize("name", FRAMES)
@pytest.mark.parametrize("pad", [True, False])
def test_oracle_reproduces_video_frame_preprocessing(name, pad):
    """expand2square + CLIP preprocess (PIL backend = transformers 4.41 behaviour) on video frames, bit for bit."""
    px = torch.from_numpy(O.preprocess_frames([GOLD["frame_" + name]], pad=pad)).to(torch.bfloat16)
    assert sha(px.view(torch.int16).numpy()) == str(GOLD[f"frame_{name}_pad{int(pad)}_pixels_bf16_sha256"])


class NumpyBackend:
    """Stand-in for the two byte kernels so that the host-side geometry of vita_b200.image_frontend (grid choice,
    coefficient tables, padding, crop offsets, tile order) can be checked without a GPU.  Test infrastructure."""

    def resample(self, img, axis, out_size, kk, bounds):
        src = np.moveaxis(img.numpy().astype(np.int64), 0 if axis == 0 else 1, 0)
        kk, bounds = kk.numpy().astype(np.int64), bounds.numpy()
        out = np.empty((out_size,) + src.shape[1:], dtype=np.uint8)
        for o in range(out_size):
            xmin, xmax = bounds[o]
            acc = (1 << 21) + np.tensordot(kk[o, :xmax], src[xmin:xmin + xmax], axes=(0, 0))
            out[o] = np.clip(acc >> 22, 0, 255)
        return torch.from_numpy(np.ascontiguousarray(np.moveaxis(out, 0, 0 if axis == 0 else 1)))

    def tiles_lut(self, img, lut, out, gi, gj, T, tile0):
        a = img.numpy()
        for t in range(gi * gj):
            tile = a[(t // gi) * T:(t // gi + 1) * T, (t % gi) * T:(t % gi + 1) * T]
            for c in range(3):
                out[tile0 + t, c] = lut[c][torch.from_numpy(tile[..., c].astype(np.int64))]


def _host_proc():
    from vita_b200.image_frontend import ImageProcessor
    return ImageProcessor("cpu", backend=NumpyBackend())


@pytest.mark.parametrize("name", ["wide", "tiny"])
def test_frontend_geometry_on_host_matches_reference(name):
    px, n = _host_proc().preprocess(GOLD[name + "_image"])
    assert n == int(GOLD[name + "_n_tiles"])
    assert sha(px.view(torch.int16).numpy()) == str(GOLD[name + "_pixels_bf16_sha256"])


@pytest.mark.parametrize("name", FRAMES)
@pytest.mark.parametrize("pad", [True, False])
def test_frontend_frame_geometry_on_host_matches_reference(name, pad):
    px = _host_proc().preprocess_frames([GOLD["frame_" + name]], pad=pad)
    assert sha(px.view(torch.int16).numpy()) == str(GOLD[f"frame_{name}_pad{int(pad)}_pixels_bf16_sha256"])


def test_frame_sampling_positions():
    from vita_b200.image_frontend import sample_frame_positions as P
    # 10 s at 30 fps, 1 frame per second, at most 16: positions 0, 30, ..., 270
    assert P(300, 30.0, 16) == list(range(0, 300, 30))
    # 60 s: 60 candidates thinned to 16 with linspace(dtype=int)
    assert P(1800, 30.0, 16) == [list(range(0, 1800, 30))[i] for i in np.linspace(0, 59, num=16, dtype=int)]
    # 2 s clip: 2 candidates repeated up to min_frames = 4
    assert P(60, 30.0, 16) == [0, 0, 0, 30]      # linspace(0, 1, 4, dtype=int) = 0, 0, 0, 1
    for n, fps, mx, s, e in [(300, 30.0, 16, None, None), (1800, 29.97, 8, 3, 41), (500, 25.0, 4, 7, 7), (90, 24.0, 16, 9, 2),
                             (1000, 60.0, 16, 0, 1000), (10, 30.0, 16, None, None), (5000, 23.976, 16, 12.7, 80.2)]:
        assert P(n, fps, mx, s=s, e=e) == O.sample_frame_positions(n, fps, mx, s=s, e=e), (n, fps, mx, s, e)
