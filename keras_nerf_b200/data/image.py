"""ImageLoader (reference: keras_nerf/data/image.py) -- PNG decode on the host, everything after it in one
libknerf kernel (`knerf_image_prepare`: uint8 -> float, antialiased bilinear resize, alpha composite, clip)."""
from __future__ import annotations

import io
import os

import numpy as np
import torch

from .. import _lib


def decode_image_rgba(source) -> np.ndarray:
    """tf.io.read_file + tf.io.decode_image(channels=4, expand_animations=False) (image.py:19-20):
    path / bytes -> [H,W,4] uint8.  Decoding (zlib inflate + PNG unfiltering) is host library work (Pillow)."""
    from PIL import Image
    if isinstance(source, (bytes, bytearray)):
        source = io.BytesIO(source)
    elif isinstance(source, (str, os.PathLike)) and not os.path.exists(source):
        raise FileNotFoundError(source)
    with Image.open(source) as im:
        im.seek(0)                                         # expand_animations=False: first frame only
        return np.array(im.convert("RGBA"), dtype=np.uint8)   # a writable copy


def as_rgba_uint8(image) -> torch.Tensor:
    """path / encoded bytes / decoded [H,W,3|4] uint8 array or tensor -> [H,W,4] uint8 tensor (opaque alpha added)"""
    if torch.is_tensor(image) or isinstance(image, np.ndarray):
        rgba = torch.as_tensor(image)
        if rgba.dtype != torch.uint8 or rgba.dim() != 3 or rgba.shape[-1] not in (3, 4):
            raise ValueError("decoded images must be [H,W,3|4] uint8")
        if rgba.shape[-1] == 3:                         # decode_image(channels=4) gives opaque alpha
            rgba = torch.cat([rgba, torch.full_like(rgba[..., :1], 255)], dim=-1)
        return rgba
    return torch.from_numpy(decode_image_rgba(image))


def prepare_image(image, out_h: int, out_w: int, white_background: bool = False, device=None) -> torch.Tensor:
    """`knerf_image_prepare` on one image: -> float32 CUDA tensor [out_h, out_w, 4] (antialiased bilinear resize,
    rgb composited on the background, alpha).  `image` as `as_rgba_uint8` takes it."""
    device = device or _lib.default_device()
    rgba = as_rgba_uint8(image).contiguous().to(device, non_blocking=True)
    in_h, in_w = int(rgba.shape[0]), int(rgba.shape[1])
    with torch.cuda.device(device):
        out = torch.empty((int(out_h), int(out_w), 4), dtype=torch.float32, device=device)
        _lib.call("knerf_image_prepare", _lib.ptr(rgba, torch.uint8), in_h, in_w, int(out_h), int(out_w),
                  int(white_background), _lib.ptr(out), _lib.stream())
    return out


class ImageLoader:
    """Same constructor and call signature as keras_nerf/data/image.py:4-35.

    `__call__(image_path)` -> float32 CUDA tensor [image_width, image_height, 4] (rgb composited on the
    background, alpha), i.e. the reference's axis order: it hands (image_width, image_height) to
    tf.image.resize as (height, width) (image.py:22-23); identical for the square images of nerf_synthetic.
    Also accepts encoded bytes or an already decoded [H,W,3|4] uint8 array / tensor.  `prepare_image` takes
    (out_h, out_w) in the usual order.
    """

    def __init__(self, image_width: int, image_height: int, white_background: bool = False, device=None, **kwargs):
        self.image_width = int(image_width)
        self.image_height = int(image_height)
        self.white_background = bool(white_background)
        self.device = torch.device(device) if device is not None else None

    def __call__(self, image_path) -> torch.Tensor:
        # (sic) image.py:22-23: out_h, out_w = image_width, image_height
        return prepare_image(image_path, self.image_width, self.image_height, self.white_background, self.device)
