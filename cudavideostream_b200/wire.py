"""Opt-in compact wire format CVW1 (include/cvs_b200.h): ctypes view of the C ABI plus a host-side parser.

The reference's format (server/src/threads.cpp:229-231, client/opencv.cpp:52-66) is u32 pos, i32 xs[pos], u8 diff[pos];
CVW1 carries the same ascending indices as per-tile counts + one-byte offsets.  `parse` is a host decoder in a few
lines of numpy that refuses every inconsistent frame the device decoder refuses, and a buffer too short for its frame.
"""
from __future__ import annotations

import struct

import numpy as np

from .api import _check, load_library

TILE = 192
MAGIC = 0x31575643
HEADER = 16


def _pad16(v: int) -> int:
    return (v + 15) & ~15


def bound(width: int, height: int) -> int:
    return int(load_library().cvs_wire_bound(width, height))


def ntiles(width: int, height: int) -> int:
    return (3 * width * height + TILE - 1) // TILE


def scratch_words(width: int, height: int) -> int:
    return ntiles(width, height) + 2


def size_of(wire: np.ndarray) -> int:
    """Total bytes of the encoded frame at the start of `wire` (from its header)."""
    magic, pos, nt, tile = struct.unpack_from("<4I", wire, 0)
    if magic != MAGIC or tile != TILE:
        raise ValueError("not a CVW1 frame")
    return HEADER + _pad16(nt) + _pad16(pos) + pos


def parse(wire: np.ndarray, geometry: tuple[int, int] | None = None):
    """Returns (pos, xs[pos] int32 ascending, diff[pos] uint8) of one CVW1 frame in host memory.

    Raises ValueError, before anything is decoded, unless the buffer holds the whole frame, the header is CVW1 with
    tile 192 (and, given the frame's geometry (width, height), its ntiles), no tile counts more entries than it has
    bytes, the counts add up to pos, and inside each tile the offsets are strictly ascending and below the tile's
    length.  Without a geometry every tile counts as 192 bytes long, the last one included."""
    wire = np.ascontiguousarray(wire, dtype=np.uint8).reshape(-1)
    if wire.size < HEADER:
        raise ValueError("shorter than a CVW1 header")
    magic, pos, nt, tile = struct.unpack_from("<4I", wire, 0)
    if magic != MAGIC or tile != TILE:
        raise ValueError("not a CVW1 frame")
    last = TILE
    if geometry is not None:
        n = 3 * geometry[0] * geometry[1]
        if nt != ntiles(*geometry):
            raise ValueError(f"ntiles {nt} is not the {ntiles(*geometry)} of a {geometry[0]}x{geometry[1]} frame")
        last = n - TILE * (nt - 1)
    o0 = HEADER + _pad16(nt)
    d0 = o0 + _pad16(pos)
    if wire.size < d0 + pos:
        raise ValueError(f"buffer of {wire.size} bytes, frame of {d0 + pos}")
    counts = wire[HEADER:HEADER + nt].astype(np.int64)
    lens = np.full(nt, TILE, dtype=np.int64)
    lens[-1:] = last
    if (counts > lens).any():
        raise ValueError("a tile counts more entries than it has bytes")
    if int(counts.sum()) != pos:
        raise ValueError("tile counts do not add up to pos")
    tile_of = np.repeat(np.arange(nt, dtype=np.int64), counts)
    off = wire[o0:o0 + pos].astype(np.int64)
    if (off >= lens[tile_of]).any():
        raise ValueError("an offset lies past its tile")
    xs = tile_of * TILE + off
    if (np.diff(xs) <= 0).any():  # with every offset inside its tile: ascending inside each tile
        raise ValueError("offsets are not strictly ascending inside a tile")
    return pos, xs.astype(np.int32), wire[d0:d0 + pos].copy()


def encode_device(d_xs: int, d_diff: int, d_pos: int, capacity: int, width: int, height: int, d_scratch: int,
                  d_wire: int, stream: int = 0) -> None:
    _check(load_library().cvs_wire_encode_device(d_xs, d_diff, d_pos, capacity, width, height, d_scratch, d_wire,
                                                 stream or None))


def decode_device(d_wire: int, d_scratch: int, width: int, height: int, d_frame: int = 0, d_xs: int = 0,
                  d_diff: int = 0, d_pos: int = 0, stream: int = 0) -> None:
    _check(load_library().cvs_wire_decode_device(d_wire, d_scratch, d_frame or None, d_xs or None, d_diff or None,
                                                 d_pos or None, width, height, stream or None))


def decode_status(d_scratch: int, width: int, height: int, stream: int = 0) -> None:
    _check(load_library().cvs_wire_decode_status(d_scratch, width, height, stream or None))
