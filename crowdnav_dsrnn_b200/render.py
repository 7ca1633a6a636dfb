"""Host-side pieces of `render(mode="rgb_array")`: argument checks, baselines' `tile_images` layout and a PNG writer.

The frames themselves are drawn on the GPU by `cn_env_render` (csrc/render.cu) through `CrowdEngine.render`.  Only the
gym-standard "rgb_array" mode exists; the reference's interactive matplotlib window ("human") is not reproduced.
"""
import struct
import zlib

import numpy as np

from . import abi

MODES = ("rgb_array",)


def check_mode(mode):
    if mode not in MODES:
        raise NotImplementedError("render(mode=%r): only mode='rgb_array' is supported (frames are drawn on the GPU); "
                                  "the interactive matplotlib window is out of scope" % (mode,))


def check_size(size):
    """Frame side in pixels: an int in [32, 2048] divisible by 16 (the limits of cn_env_render)."""
    if isinstance(size, bool) or not isinstance(size, (int, np.integer)):
        raise TypeError("size must be an int, got %r" % (size,))
    size = int(size)
    if not (abi.RENDER_MIN_SIZE <= size <= abi.RENDER_MAX_SIZE) or size % abi.RENDER_SIZE_MULTIPLE:
        raise ValueError("size %d must be a multiple of %d in %d..%d" % (size, abi.RENDER_SIZE_MULTIPLE, abi.RENDER_MIN_SIZE,
                                                                          abi.RENDER_MAX_SIZE))
    return size


def tile_images(frames):
    """baselines.common.tile_images: k frames [k, h, w, c] -> one [rows * h, cols * w, c] image, rows = ceil(sqrt(k)),
    cols = ceil(k / rows), row-major, the unused cells zero."""
    frames = np.asarray(frames)
    k, h, w, c = frames.shape
    rows = int(np.ceil(np.sqrt(k)))
    cols = int(np.ceil(float(k) / rows))
    grid = np.concatenate([frames, np.zeros((rows * cols - k, h, w, c), dtype=frames.dtype)], axis=0)
    return grid.reshape(rows, cols, h, w, c).transpose(0, 2, 1, 3, 4).reshape(rows * h, cols * w, c)


def write_png(path, rgb):
    """An [h, w, 3] uint8 array as an 8-bit RGB PNG (stdlib zlib only)."""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, c = rgb.shape
    if c != 3:
        raise ValueError("write_png needs [h, w, 3], got %r" % (rgb.shape,))
    raw = np.concatenate([np.zeros((h, 1), dtype=np.uint8), rgb.reshape(h, w * 3)], axis=1).tobytes()  # filter 0 per row

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n")
        f.write(chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)))
        f.write(chunk(b"IDAT", zlib.compress(raw, 6)))
        f.write(chunk(b"IEND", b""))
