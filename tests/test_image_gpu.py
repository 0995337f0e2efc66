"""csrc/image.cu through vita_b200.image_frontend against the golden digests (reference dynamic_preprocess + Pillow +
CLIPImageProcessor, minted by oracle/make_golden_image.py) and against the numpy oracle: integer / byte work, so the bar
is bit-exact."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import image_oracle as O
from tests.util import load_image_golden

pytestmark = pytest.mark.gpu
GOLD = load_image_golden()


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def proc():
    from vita_b200.image_frontend import ImageProcessor
    return ImageProcessor("cuda")


@pytest.mark.parametrize("name", ["wide", "tall", "square", "tiny", "pano"])
def test_pipeline_reproduces_reference_bits(proc, name):
    img = GOLD[name + "_image"]
    big, thumb, (gi, gj) = proc.dynamic_tiles_u8(img)
    T = 448
    b = big.cpu().numpy()
    tiles = [b[(t // gi) * T:(t // gi + 1) * T, (t % gi) * T:(t % gi + 1) * T] for t in range(gi * gj)]
    if thumb is not None:
        tiles.append(thumb.cpu().numpy())
    tiles = np.stack(tiles)
    assert tiles.shape[0] == int(GOLD[name + "_n_tiles"])
    assert sha(tiles) == str(GOLD[name + "_tiles_sha256"]), "resized bytes differ from Pillow"
    px, n = proc.preprocess(img)
    assert n == tiles.shape[0] and px.dtype == torch.bfloat16 and tuple(px.shape) == (n, 3, T, T)
    assert sha(px.cpu().view(torch.int16).numpy()) == str(GOLD[name + "_pixels_bf16_sha256"])


@pytest.mark.parametrize("h,w,tw,th", [(2000, 3000, 1344, 896), (123, 77, 448, 448), (448, 600, 448, 448),
                                       (50, 40, 55, 41), (700, 448, 448, 1792), (5, 3, 448, 448)])
def test_resize_equals_oracle(proc, h, w, tw, th):
    """Down- and up-scaling, one-axis-only resizes, tiny inputs (windows clipped at both borders)."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.int64)
    img = np.stack([(xx * 7 + yy * 3) % 256, (xx * xx // 5 + yy) % 256, (255 - (xx + 2 * yy) % 256)], -1).astype(np.uint8)
    got = proc.resize(torch.from_numpy(img).cuda(), tw, th).cpu().numpy()
    want = O.resize_bicubic(img, tw, th)
    assert got.shape == want.shape == (th, tw, 3)
    assert np.array_equal(got, want)


def test_process_images_and_model_entry_points(proc):
    """The reference's two-step API: tiles cut on the host -> model.process_images(...) -> the same bits; and the
    result feeds encode_images."""
    from vita_b200 import weights as W
    from vita_b200.config import VitaConfig
    from vita_b200.model.vita_mixtral import VITAMixtralForCausalLM
    img = GOLD["wide_image"]
    tiles = O.dynamic_preprocess(img)
    cfg = VitaConfig.tiny()
    model = VITAMixtralForCausalLM(cfg, W.pack(W.synthetic_state(cfg, 0), cfg, "cuda"), "cuda", max_seq_len=256,
                                   max_new_tokens=8)
    px = model.process_images([t for t in tiles], model.config)
    assert sha(px.cpu().view(torch.int16).numpy()) == str(GOLD["wide_pixels_bf16_sha256"])
    px2, n = model.preprocess_image(img)
    assert torch.equal(px, px2) and n == tiles.shape[0]
    with pytest.raises(ValueError):
        model.process_images([img], model.config)          # not a 448 x 448 tile


@pytest.mark.parametrize("name", ["landscape", "portrait", "sq"])
@pytest.mark.parametrize("pad", [True, False])
def test_video_frames_reproduce_reference_bits(proc, name, pad):
    """video_audio_demo.py:83-110: expand2square + CLIP preprocess (transformers 4.41 = PIL backend) per frame."""
    px = proc.preprocess_frames([GOLD["frame_" + name]], pad=pad)
    assert px.is_cuda and tuple(px.shape) == (1, 3, 448, 448)
    assert sha(px.cpu().view(torch.int16).numpy()) == str(GOLD[f"frame_{name}_pad{int(pad)}_pixels_bf16_sha256"])


def test_video_frame_batch(proc):
    frames = [GOLD["frame_landscape"], GOLD["frame_portrait"], GOLD["frame_sq"], GOLD["frame_landscape"]]
    px = proc.preprocess_frames(frames)
    want = torch.from_numpy(O.preprocess_frames(frames)).to(torch.bfloat16)
    assert torch.equal(px.cpu(), want)
