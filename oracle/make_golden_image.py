"""Mints tests/golden/image_golden.npz in the build container from the real thing:
  * tiles: the reference's own `dynamic_preprocess` (vita/util/data_utils_video_audio_neg_patch.py:1197-1255, its two
    functions are compiled from the reference source without importing the training module) driving Pillow's resize;
  * pixel values: transformers' CLIPImageProcessor with the reference's preprocessor_config.json constants, cast to
    bf16 as `model.process_images(...).to(dtype=model.dtype)` does (video_audio_demo.py:219-221).
Inputs are oracle.image_oracle.card test cards, stored as their (h, w, k) and a SHA-256 digest; outputs are stored as
SHA-256 digests plus a small crop (the numpy oracle reproduces them bit for bit, tests/test_image.py).
Run: python oracle/make_golden_image.py"""
import ast
import hashlib
import os
import sys

import numpy as np
import torch
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.image_oracle import card  # noqa: E402

REF = "/root/reference/vita/util/data_utils_video_audio_neg_patch.py"


def reference_functions():
    ns = {}
    for node in ast.parse(open(REF).read()).body:
        if isinstance(node, ast.FunctionDef) and node.name in ("find_closest_aspect_ratio", "dynamic_preprocess"):
            exec(compile(ast.Module([node], []), REF, "exec"), ns)
    return ns["dynamic_preprocess"]


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    from transformers import CLIPImageProcessor
    dyn = reference_functions()
    ip = CLIPImageProcessor(crop_size=448, do_center_crop=True, do_normalize=True, do_resize=True,
                            image_mean=[0.485, 0.456, 0.406], image_std=[0.229, 0.224, 0.225], resample=3, size=448)
    out = {}
    cases = {"wide": (300, 500, 1), "tall": (451, 167, 2), "square": (448, 448, 3), "tiny": (37, 61, 4), "pano": (120, 950, 5)}
    for name, (h, w, k) in cases.items():
        img = card(h, w, k)
        tiles, n = dyn(Image.fromarray(img), min_num=1, max_num=12, image_size=448, use_thumbnail=True)
        t = np.stack([np.asarray(x) for x in tiles])
        pv = ip.preprocess(list(tiles), return_tensors="pt")["pixel_values"].to(torch.bfloat16)
        out[name + "_image_card"] = np.array([h, w, k])
        out[name + "_image_sha256"] = np.array(sha(img))
        out[name + "_tiles_sha256"] = np.array(sha(t))
        out[name + "_pixels_bf16_sha256"] = np.array(sha(pv.view(torch.int16).numpy()))
        out[name + "_n_tiles"] = np.array(n[0])
        out[name + "_tile0_crop"] = t[0, :32, :32].copy()
        print(name, img.shape, "->", t.shape, sha(t)[:12], sha(pv.view(torch.int16).numpy())[:12])
    # video frames (video_audio_demo.py:83-110): expand2square with int(mean * 255) + CLIP preprocess.  The reference
    # pins transformers 4.41.1, whose CLIPImageProcessor resizes through PIL; in the installed 5.x that behaviour is
    # CLIPImageProcessorPil (the default class moved to a torchvision backend that is not bit-compatible).
    from transformers.models.clip import CLIPImageProcessorPil
    ipp = CLIPImageProcessorPil(crop_size=448, do_center_crop=True, do_normalize=True, do_resize=True,
                                image_mean=[0.485, 0.456, 0.406], image_std=[0.229, 0.224, 0.225], resample=3, size=448)

    def expand2square(pil_img, background_color):          # as the demo defines it inline
        width, height = pil_img.size
        if width == height:
            return pil_img
        side = max(width, height)
        result = Image.new(pil_img.mode, (side, side), background_color)
        result.paste(pil_img, (0, (width - height) // 2) if width > height else ((height - width) // 2, 0))
        return result

    frames = {"landscape": (180, 320, 6), "portrait": (321, 179, 7), "sq": (200, 200, 8)}
    bg = tuple(int(x * 255) for x in ipp.image_mean)
    for name, (h, w, k) in frames.items():
        img = card(h, w, k)
        out["frame_" + name + "_card"] = np.array([h, w, k])
        out["frame_" + name + "_sha256"] = np.array(sha(img))
        for pad in (True, False):
            pil = Image.fromarray(img)
            pv = ipp.preprocess(expand2square(pil, bg) if pad else pil, return_tensors="pt")["pixel_values"].to(torch.bfloat16)
            out[f"frame_{name}_pad{int(pad)}_pixels_bf16_sha256"] = np.array(sha(pv.view(torch.int16).numpy()))
            print("frame", name, "pad" if pad else "nopad", tuple(pv.shape), sha(pv.view(torch.int16).numpy())[:12])
    # every uint8 value through the processor: the 3 x 256 table the GPU path indexes
    ramp = np.tile(np.arange(256, dtype=np.uint8)[None, :, None], (448, 2, 3))[:, :448]
    pv = ip.preprocess([Image.fromarray(ramp)], return_tensors="pt")["pixel_values"][0].to(torch.bfloat16)
    out["lut_bf16_bits"] = pv[:, 0, :256].contiguous().view(torch.int16).numpy()
    path = os.path.join(HERE, "..", "tests", "golden", "image_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", os.path.normpath(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
