"""TEST INFRASTRUCTURE ONLY: CPU restatement of the image preprocessing in front of InternViT.

Reference path (video_audio_demo.py:214-221 -> vita/util/data_utils_video_audio_neg_patch.py:1197-1255 ->
vita/util/mm_utils.py:30-43 -> transformers CLIPImageProcessor with the constants of
web_demo/vllm_tools/model_weight_file/preprocessor_config.json):
  1. `dynamic_preprocess`: choose the tile grid (i, j) closest in aspect ratio, `image.resize((448 i, 448 j))`
     (PIL default = bicubic), cut 448 x 448 tiles row-major, append a 448 x 448 thumbnail when there is more than one.
  2. per tile: rescale by 1/255, normalise with mean (0.485, 0.456, 0.406) / std (0.229, 0.224, 0.225)
     (resize-to-448 and centre crop are identities on 448 x 448 tiles).
The resize arithmetic lives in the third-party dependency Pillow (unpinned in the reference; 12.2.0 installed here):
src/libImaging/Resample.c, 8-bit path -- double-precision separable coefficients, normalised, rounded to 22-bit fixed
point, horizontal pass then vertical pass with a uint8 intermediate, each output = clip8((2^21 + sum p*k) >> 22).
Restated below in numpy and pinned against PIL itself (oracle/make_golden_image.py -> tests/golden/image_golden.npz,
checked bit-for-bit by tests/test_image.py).
"""
import math

import numpy as np

PRECISION_BITS = 32 - 8 - 2
IMAGE_SIZE = 448
MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)


def _bicubic(x: float) -> float:
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def precompute_coeffs(in_size: int, out_size: int):
    """Resample.c `precompute_coeffs` + `normalize_coeffs_8bpc` for the full box [0, in_size): (ksize, bounds, kk)."""
    scale = filterscale = float(in_size) / out_size
    if filterscale < 1.0:
        filterscale = 1.0
    support = 2.0 * filterscale
    ksize = int(math.ceil(support)) * 2 + 1
    bounds = np.zeros((out_size, 2), dtype=np.int64)
    kk = np.zeros((out_size, ksize), dtype=np.int64)
    for xx in range(out_size):
        center = 0 + (xx + 0.5) * scale
        ww = 0.0
        ss = 1.0 / filterscale
        xmin = int(center - support + 0.5)
        if xmin < 0:
            xmin = 0
        xmax = int(center + support + 0.5)
        if xmax > in_size:
            xmax = in_size
        xmax -= xmin
        k = [0.0] * ksize
        for x in range(xmax):
            w = _bicubic((x + xmin - center + 0.5) * ss)
            k[x] = w
            ww += w
        for x in range(xmax):
            if ww != 0.0:
                k[x] /= ww
        for x in range(ksize):
            v = k[x]
            kk[xx, x] = int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
        bounds[xx] = (xmin, xmax)
    return ksize, bounds, kk


def _pass(img: np.ndarray, out_size: int, axis: int) -> np.ndarray:
    """One separable pass over `axis` of an [H, W, C] uint8 image."""
    src = np.moveaxis(img, axis, 0).astype(np.int64)          # [in, other, C]
    _, bounds, kk = precompute_coeffs(src.shape[0], out_size)
    out = np.empty((out_size,) + src.shape[1:], dtype=np.uint8)
    for xx in range(out_size):
        xmin, xmax = bounds[xx]
        acc = np.full(src.shape[1:], 1 << (PRECISION_BITS - 1), dtype=np.int64)
        acc += np.tensordot(kk[xx, :xmax], src[xmin:xmin + xmax], axes=(0, 0))
        out[xx] = np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)
    return np.moveaxis(out, 0, axis)


def resize_bicubic(img: np.ndarray, width: int, height: int) -> np.ndarray:
    """PIL `Image.resize((width, height))` on an RGB image given as [H, W, 3] uint8 (horizontal pass first)."""
    h, w, _ = img.shape
    out = img
    if width != w:
        out = _pass(out, width, axis=1)
    if height != h:
        out = _pass(out, height, axis=0)
    return out.copy() if out is img else out


def closest_grid(width: int, height: int, min_num: int = 1, max_num: int = 12, image_size: int = IMAGE_SIZE):
    """`find_closest_aspect_ratio` over the grids `dynamic_preprocess` enumerates (data_utils...:1197-1231)."""
    ratios = sorted({(i, j) for n in range(min_num, max_num + 1) for i in range(1, n + 1) for j in range(1, n + 1)
                     if min_num <= i * j <= max_num}, key=lambda r: r[0] * r[1])
    aspect = width / height
    best, best_diff = (1, 1), float("inf")
    for r in ratios:
        diff = abs(aspect - r[0] / r[1])
        if diff < best_diff:
            best_diff, best = diff, r
        elif diff == best_diff and width * height > 0.5 * image_size * image_size * r[0] * r[1]:
            best = r
    return best


def dynamic_preprocess(img: np.ndarray, min_num: int = 1, max_num: int = 12, use_thumbnail: bool = True):
    """[H, W, 3] uint8 -> [N, 448, 448, 3] uint8 tiles in the reference's order (+ thumbnail)."""
    h, w, _ = img.shape
    gi, gj = closest_grid(w, h, min_num, max_num)
    big = resize_bicubic(img, IMAGE_SIZE * gi, IMAGE_SIZE * gj)
    tiles = [big[(t // gi) * IMAGE_SIZE:(t // gi + 1) * IMAGE_SIZE, (t % gi) * IMAGE_SIZE:(t % gi + 1) * IMAGE_SIZE]
             for t in range(gi * gj)]
    if use_thumbnail and len(tiles) != 1:
        tiles.append(resize_bicubic(img, IMAGE_SIZE, IMAGE_SIZE))
    return np.stack(tiles)


def normalize_tiles(tiles_u8: np.ndarray) -> np.ndarray:
    """CLIPImageProcessor rescale + normalise (transformers image_transforms: `image.astype(float64) * (1/255)` cast to
    float32, then `(image - mean) / std` in float32): [N, 448, 448, 3] uint8 -> [N, 3, 448, 448] float32."""
    x = (tiles_u8.astype(np.float64) * (1 / 255)).astype(np.float32)
    mean = np.asarray(MEAN, dtype=np.float32)
    std = np.asarray(STD, dtype=np.float32)
    x = (x - mean) / std
    return np.ascontiguousarray(x.transpose(0, 3, 1, 2)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ video frames
def expand2square(img: np.ndarray, background) -> np.ndarray:
    """mm_utils.py:16-28 / video_audio_demo.py:86-97: pad the short side with the background colour, image centred."""
    h, w, _ = img.shape
    if w == h:
        return img
    s = max(w, h)
    out = np.empty((s, s, 3), dtype=np.uint8)
    out[...] = np.asarray(background, dtype=np.uint8)
    if w > h:
        out[(w - h) // 2:(w - h) // 2 + h, :] = img
    else:
        out[:, (h - w) // 2:(h - w) // 2 + w] = img
    return out


def clip_resize_crop(img: np.ndarray, size: int = IMAGE_SIZE) -> np.ndarray:
    """CLIPImageProcessor of transformers 4.41 (the reference's pin; PIL backend): shortest edge -> `size` with the long
    edge int(size * long / short), PIL bicubic, then centre crop size x size (top = (h - size) // 2)."""
    h, w, _ = img.shape
    short, long = (w, h) if w <= h else (h, w)
    new_long = int(size * long / short)
    nh, nw = (new_long, size) if w <= h else (size, new_long)
    r = resize_bicubic(img, nw, nh)
    top, left = (nh - size) // 2, (nw - size) // 2
    return np.ascontiguousarray(r[top:top + size, left:left + size])


def preprocess_frames(frames, pad: bool = True) -> np.ndarray:
    """video_audio_demo.py:83-110: (expand2square with int(mean * 255)) -> CLIP preprocess: [T, 3, 448, 448] float32."""
    bg = tuple(int(x * 255) for x in MEAN)
    tiles = [clip_resize_crop(expand2square(f, bg) if pad else f) for f in frames]
    return normalize_tiles(np.stack(tiles))


def sample_frame_positions(n_frames: int, fps: float, max_frames: int, min_frames: int = 4, video_framerate: int = 1,
                           s=None, e=None):
    """Index arithmetic of `_get_rawvideo_dec` (video_audio_demo.py:43-81): which decoded frames are kept."""
    if s is None:
        start_time, end_time = None, None
    else:
        start_time, end_time = int(s), int(e)
        start_time = start_time if start_time >= 0.0 else 0.0
        end_time = end_time if end_time >= 0.0 else 0.0
        if start_time > end_time:
            start_time, end_time = end_time, start_time
        elif start_time == end_time:
            end_time = start_time + 1
    f_start = 0 if start_time is None else int(start_time * fps)
    f_end = int(min(1000000000 if end_time is None else end_time * fps, n_frames - 1))
    if f_end - f_start + 1 <= 0:
        return []
    t_stride = int(round(float(fps) / int(video_framerate)))
    all_pos = list(range(f_start, f_end + 1, t_stride))
    if len(all_pos) > max_frames:
        return [all_pos[i] for i in np.linspace(0, len(all_pos) - 1, num=max_frames, dtype=int)]
    if len(all_pos) < min_frames:
        return [all_pos[i] for i in np.linspace(0, len(all_pos) - 1, num=min_frames, dtype=int)]
    return all_pos


# ------------------------------------------------------------------------------------------------ golden inputs
def card(h: int, w: int, k: int) -> np.ndarray:
    """Deterministic integer test card: gradients, a checkerboard patch, hard-edged boxes (no libm, no RNG).  The image
    golden stores (h, w, k) and a digest of each card rather than its pixels."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.int64)
    img = np.stack([(xx * 255 // max(w - 1, 1) + k * 17) % 256, (yy * 255 // max(h - 1, 1) + k * 29) % 256,
                    ((xx + yy) * 3 + k * 41) % 256], -1)
    cb = ((xx // 7 + yy // 5) % 2 == 0) & (xx > w // 2) & (yy < h // 2)
    img[cb] = 255 - img[cb]
    img[h // 3: h // 3 + max(h // 9, 2), w // 4: w // 4 + max(w // 5, 2)] = (250, 10, 128)
    img[(yy - h // 2) ** 2 + (xx - w // 3) ** 2 < (min(h, w) // 6) ** 2] = (5, 240, 60)
    return img.astype(np.uint8)
