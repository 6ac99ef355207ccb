"""Opt-in compact wire format CVW1 (SURVEY.md section 8f row 3; include/cvs_b200.h): the GPU encoder and decoder
against the host-side parser, the oracle's payload and the client round trip `reconstructed == reference`.
Default format stays the reference's (threads.cpp:229-231 / client/opencv.cpp:52-66)."""
import ctypes as C
import struct

import numpy as np
import pytest

from util import random_sequence


def _encode_numpy(xs, diff, n):
    """Specification-level encoder (numpy), the twin of cudavideostream_b200.wire.parse."""
    from cudavideostream_b200 import wire
    nt = (n + wire.TILE - 1) // wire.TILE
    pos = int(xs.size)
    counts = np.bincount(xs // wire.TILE, minlength=nt).astype(np.uint8)
    out = np.zeros(wire.HEADER + wire._pad16(nt) + wire._pad16(pos) + pos, dtype=np.uint8)
    out[:16] = np.frombuffer(struct.pack("<4I", wire.MAGIC, pos, nt, wire.TILE), dtype=np.uint8)
    out[16:16 + nt] = counts
    o0 = 16 + wire._pad16(nt)
    out[o0:o0 + pos] = (xs % wire.TILE).astype(np.uint8)
    d0 = o0 + wire._pad16(pos)
    out[d0:d0 + pos] = diff
    return out


def test_parser_round_trip_on_the_oracle_payload(oracle):
    from cudavideostream_b200 import wire
    for w, h, dens in [(7, 5, 0.5), (64, 48, 0.1), (250, 130, 0.01), (64, 48, 1.0), (64, 48, 0.0)]:
        n = 3 * w * h
        base, frames = random_sequence(w, h, 1, dens, seed=w)
        pos, xs, diff, _, _ = oracle.diff_compact(frames[0], base, 20)
        enc = _encode_numpy(xs, diff, n)
        assert wire.size_of(enc) == enc.size == 16 + wire._pad16(wire.ntiles(w, h)) + wire._pad16(pos) + pos
        p2, xs2, diff2 = wire.parse(enc)
        assert p2 == pos and np.array_equal(xs2, xs) and np.array_equal(diff2, diff)
    with pytest.raises(ValueError):
        wire.parse(np.zeros(64, dtype=np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,density", [(7, 5, 0.3), (64, 48, 0.0), (64, 48, 1.0), (250, 130, 0.02), (641, 359, 0.3),
                                         (1920, 1080, 0.1)])
def test_submit_wire_matches_the_oracle_and_round_trips(cvs, oracle, w, h, density):
    import torch
    from cudavideostream_b200 import wire
    n = 3 * w * h
    T = 5 if w < 1000 else 3
    base, frames = random_sequence(w, h, T, density, seed=w + 1)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    fin = cvs.alloc_host(n + 32)
    wout = cvs.alloc_host(wire.bound(w, h) + 64)
    st = torch.cuda.current_stream().cuda_stream
    client = torch.from_numpy(base).cuda()
    client = torch.cat([client, torch.zeros(64, dtype=torch.uint8, device="cuda")])
    d_scr = torch.zeros(wire.scratch_words(w, h), dtype=torch.int32, device="cuda")
    d_xs = torch.zeros(n + 16, dtype=torch.int32, device="cuda")
    d_df = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
    d_pos = torch.zeros(1, dtype=torch.int32, device="cuda")
    for t, f in enumerate(frames):
        fin.array()[:n] = f
        wout.array()[:] = 0xA5
        tk = s.submit_wire_raw(fin.ptr, wout.ptr, None, "")
        s.wait(tk)
        opos, oxs, odiff, _, _ = oc.exec_core(f)
        enc = wout.array()
        size = wire.size_of(enc)
        assert size == 16 + wire._pad16(wire.ntiles(w, h)) + wire._pad16(opos) + opos
        assert bool((enc[wire.bound(w, h):] == 0xA5).all()), "write past cvs_wire_bound"
        pos, xs, diff = wire.parse(enc[:size])
        assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff), f"frame {t}"
        assert np.array_equal(enc[:size], _encode_numpy(oxs, odiff, n)), f"frame {t}: encoded bytes"
        # client side on the GPU: decode into the reference format and apply to the client's frame
        d_wire = torch.from_numpy(enc[:(size + 15) // 16 * 16].copy()).cuda()
        wire.decode_device(d_wire.data_ptr(), d_scr.data_ptr(), w, h, d_frame=client.data_ptr(), d_xs=d_xs.data_ptr(),
                           d_diff=d_df.data_ptr(), d_pos=d_pos.data_ptr(), stream=st)
        wire.decode_status(d_scr.data_ptr(), w, h, st)
        assert int(d_pos[0]) == opos
        assert np.array_equal(d_xs[:opos].cpu().numpy(), oxs) and np.array_equal(d_df[:opos].cpu().numpy(), odiff)
        assert np.array_equal(client[:n].cpu().numpy(), oc.reference()), f"frame {t}: reconstructed != reference"
    assert np.array_equal(s.reference(), oc.reference())
    s.close()


@pytest.mark.gpu
def test_wire_pageable_buffer_and_device_encoder(cvs, oracle):
    import torch
    from cudavideostream_b200 import wire
    w, h = 320, 180
    n = 3 * w * h
    base, frames = random_sequence(w, h, 3, 0.15, seed=8)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    out = np.zeros(wire.bound(w, h), dtype=np.uint8)      # pageable: delivered by a copy in cvs_wait
    for f in frames:
        fr = np.ascontiguousarray(f)
        tk = s.submit_wire_raw(fr.ctypes.data, out.ctypes.data, None, "")
        s.wait(tk)
        opos, oxs, odiff, _, _ = oc.exec_core(f)
        pos, xs, diff = wire.parse(out[:wire.size_of(out)])
        assert pos == opos and np.array_equal(xs, oxs) and np.array_equal(diff, odiff)
    s.close()
    # the stand-alone device encoder on a device-resident payload (what a sequence launch leaves behind)
    st = torch.cuda.current_stream().cuda_stream
    opos, oxs, odiff, _, _ = oracle.diff_compact(frames[0], base, 20)[:5]
    d_xs = torch.zeros(n + 16, dtype=torch.int32, device="cuda")
    d_df = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
    d_xs[:opos] = torch.from_numpy(oxs).cuda()
    d_df[:opos] = torch.from_numpy(odiff).cuda()
    d_pos = torch.tensor([opos], dtype=torch.int32, device="cuda")
    d_scr = torch.zeros(wire.scratch_words(w, h), dtype=torch.int32, device="cuda")
    d_wire = torch.zeros(wire.bound(w, h) + 16, dtype=torch.uint8, device="cuda")
    wire.encode_device(d_xs.data_ptr(), d_df.data_ptr(), d_pos.data_ptr(), n, w, h, d_scr.data_ptr(), d_wire.data_ptr(), st)
    torch.cuda.synchronize()
    enc = d_wire.cpu().numpy()
    assert np.array_equal(enc[:wire.size_of(enc)], _encode_numpy(oxs, odiff, n))
    # a corrupted frame is rejected as a whole
    bad = d_wire.clone()
    bad[16] = (int(bad[16]) + 1) % 193
    frame = torch.zeros(n + 64, dtype=torch.uint8, device="cuda")
    wire.decode_device(bad.data_ptr(), d_scr.data_ptr(), w, h, d_frame=frame.data_ptr(), stream=st)
    with pytest.raises(cvs.CVSError):
        wire.decode_status(d_scr.data_ptr(), w, h, st)
    assert int(frame.sum()) == 0


# ---------------------------------------------------------------------------------------------------------------------
# The CVW1 format at its edges.
#
# _decode_reference is the decoder's specification: a plain walk over the bytes, tile by tile, deliberately separate
# from wire.parse.  For a frame of n bytes (ntiles = ceil(n / 192), every tile 192 bytes long except the last, which
# holds n - 192 * (ntiles - 1)) it accepts a frame exactly when
#   1. the buffer holds at least 16 bytes, the magic is CVW1, tile == 192 and ntiles == ceil(n / 192);
#   2. count[t] <= len(t) for every tile;
#   3. the counts add up to the header's pos (with rule 2: pos <= n);
#   4. inside each tile the count[t] offsets are strictly ascending and below len(t);
#   5. (host buffers only) the buffer holds 16 + pad16(ntiles) + pad16(pos) + pos bytes.
# Pad bytes after the counts and after the offsets may hold anything.  _encode_numpy above is the encoder's.
# ---------------------------------------------------------------------------------------------------------------------
TILE = 192
MAGIC = 0x31575643
THR = 20
G = 16384                      # guard bytes around every device buffer of the decoder tests
REF_DECODE_MAX = 1 << 18       # larger frames are checked against the payload they were encoded from


def _pad16(v):
    return (v + 15) // 16 * 16


def _ntiles(n):
    return (n + TILE - 1) // TILE


def _tile_len(n, t):
    return min(TILE, n - TILE * t)


def _decode_reference(buf, n, host=True):
    """(xs, diff) as lists, or the number of the first rule the frame breaks."""
    b = bytes(buf)
    if len(b) < 16:
        return 1
    magic, pos, nt, tile = struct.unpack_from("<4I", b, 0)
    if magic != MAGIC or tile != TILE or nt != _ntiles(n):
        return 1
    o0 = 16 + _pad16(nt)
    d0 = o0 + _pad16(pos)
    if host and len(b) < d0 + pos:
        return 5
    counts = [b[16 + t] for t in range(nt)]
    for t in range(nt):
        if counts[t] > _tile_len(n, t):
            return 2
    if sum(counts) != pos:
        return 3
    xs, diff = [], []
    i = 0
    for t in range(nt):
        prev = -1
        for _ in range(counts[t]):
            off = b[o0 + i]
            if off >= _tile_len(n, t) or off <= prev:
                return 4
            prev = off
            xs.append(t * TILE + off)
            diff.append(b[d0 + i])
            i += 1
    return xs, diff


def _raw_frame(n, tiles, vals=None, *, magic=MAGIC, pos=None, ntiles=None, tile=TILE, pad=0):
    """The bytes of a CVW1 frame with the per-tile offsets `tiles`, written as given (no checks), so that malformed
    frames can be built.  The layout follows len(tiles) and the total entry count; header fields can be overridden.
    `pad` fills the pad bytes after the counts and after the offsets."""
    counts = [len(o) for o in tiles]
    offs = [o for ts in tiles for o in ts]
    p = len(offs)
    vals = [(37 * i + 11) & 255 for i in range(p)] if vals is None else list(vals)
    o0 = 16 + _pad16(len(tiles))
    d0 = o0 + _pad16(p)
    out = bytearray([pad]) * (d0 + p)
    struct.pack_into("<4I", out, 0, magic, p if pos is None else pos, len(tiles) if ntiles is None else ntiles, tile)
    out[16:16 + len(tiles)] = bytes(counts)
    out[o0:o0 + p] = bytes(offs)
    out[d0:d0 + p] = bytes(vals)
    return np.frombuffer(bytes(out), dtype=np.uint8).copy()


def _valid_tiles(n, rng, density=0.3):
    return [sorted(rng.choice(_tile_len(n, t), size=int(rng.binomial(_tile_len(n, t), density)), replace=False).tolist())
            for t in range(_ntiles(n))]


def _set_header(buf, **kw):
    buf = buf.copy()
    magic, pos, nt, tile = struct.unpack_from("<4I", buf, 0)
    f = dict(magic=magic, pos=pos, ntiles=nt, tile=tile)
    f.update(kw)
    buf[:16] = np.frombuffer(struct.pack("<4I", f["magic"], f["pos"], f["ntiles"], f["tile"]), dtype=np.uint8)
    return buf


MAL_W, MAL_H = 70, 3   # the hand-built frames: n = 630, four tiles, the last one 54 bytes long


def _mutations(count, seed):
    """Seeded structural mutations of valid frames of four small geometries: count and offset bytes changed, the
    header's pos set to the new sum and the buffer extended to the size the new header gives.  Returns a list of
    (w, h, buffer)."""
    rng = np.random.default_rng(seed)
    geoms = [(10, 5), (64, 2), (70, 3), (100, 7)]
    out = []
    for k in range(count):
        w, h = geoms[k % len(geoms)]
        n = 3 * w * h
        nt = _ntiles(n)
        buf = bytearray(_raw_frame(n, _valid_tiles(n, rng, rng.choice([0.05, 0.3, 0.9, 1.0]))).tobytes())
        pos = struct.unpack_from("<I", buf, 4)[0]
        o0 = 16 + _pad16(nt)
        for _ in range(int(rng.integers(1, 3))):
            kind = int(rng.choice(5, p=[0.2, 0.15, 0.2, 0.1, 0.35]))
            t = int(rng.integers(0, nt))
            ln = _tile_len(n, t)
            if kind == 0 or pos == 0:       # a count byte: near its limits or anything
                buf[16 + t] = int(rng.choice([0, ln - 1, ln, ln + 1, 191, 192, 193, 255, rng.integers(0, 256)]) & 255)
            elif kind == 1:                 # a count moves by one: the offsets of every later tile shift
                buf[16 + t] = (buf[16 + t] + int(rng.choice([-1, 1]))) & 255
            elif kind == 2:                 # an offset byte: near the limits, a neighbour's value or anything
                i = int(rng.integers(0, pos))
                nb = buf[o0 + max(i - 1, 0)]
                buf[o0 + i] = int(rng.choice([0, ln - 1, ln, 191, 192, 255, nb, rng.integers(0, 256)]) & 255)
            elif kind == 3:                 # two neighbouring offsets swap
                i = int(rng.integers(0, max(pos - 1, 1)))
                if i + 1 < pos:
                    buf[o0 + i], buf[o0 + i + 1] = buf[o0 + i + 1], buf[o0 + i]
            else:                           # an offset moves to a free value between its neighbours in its tile
                i = int(rng.integers(0, pos))
                ends = np.cumsum(list(buf[16:16 + nt]))
                t = int(np.searchsorted(ends, i, side="right"))
                if t < nt:
                    first = int(ends[t]) - buf[16 + t]
                    lo = buf[o0 + i - 1] + 1 if i > first else 0
                    hi = buf[o0 + i + 1] if i + 1 < ends[t] else _tile_len(n, t)
                    if lo < hi:
                        buf[o0 + i] = int(rng.integers(lo, hi))
        pos = sum(buf[16:16 + nt])
        struct.pack_into("<I", buf, 4, pos)
        need = o0 + _pad16(pos) + pos
        if len(buf) < need:
            buf += bytes(rng.integers(0, 256, size=need - len(buf), dtype=np.uint8))
        out.append((w, h, np.frombuffer(bytes(buf), dtype=np.uint8).copy()))
    return out


def _parse_verdict(buf, w, h):
    from cudavideostream_b200 import wire
    try:
        pos, xs, diff = wire.parse(buf, (w, h))
    except ValueError:
        return None
    assert pos == xs.size == diff.size
    return xs.tolist(), diff.tolist()


def _ref_verdict(buf, n, host=True):
    r = _decode_reference(buf, n, host)
    return None if isinstance(r, int) else r


# ------------------------------------------------------------------ CPU: the two specifications and the host parser
def test_reference_decoder_inverts_the_reference_encoder():
    from cudavideostream_b200 import wire
    rng = np.random.default_rng(1)
    for n in [3, 189, 192, 195, 381, 384, 387, 2880, 3072, 3264, 3 * 255 * 17]:
        for dens in [0.0, 0.01, 0.5, 1.0]:
            xs = np.flatnonzero(rng.random(n) < dens).astype(np.int32)
            diff = rng.integers(0, 256, size=xs.size, dtype=np.uint8)
            enc = _encode_numpy(xs, diff, n)
            assert enc.size == 16 + _pad16(_ntiles(n)) + _pad16(xs.size) + xs.size
            assert _decode_reference(enc, n) == (xs.tolist(), diff.tolist()), (n, dens)
            assert _decode_reference(enc[:-1], n) == 5, (n, dens)
            pos, xs2, diff2 = wire.parse(enc, (n // 3, 1) if n % 2 == 0 else None)
            assert pos == xs.size and np.array_equal(xs2, xs) and np.array_equal(diff2, diff)


# (name, frame, n, expected verdict of the reference decoder: a rule number, or "ok").  In the malformed ones the
# header's pos is the counts' sum, except where the sum is what is wrong, so that the sum check does not catch them.
def _hand_built():
    n = 3 * MAL_W * MAL_H
    last = _tile_len(n, 3)
    good = [[1, 5, 9], [0, 40, 191], [7, 8], [0, last - 1]]
    ok = _raw_frame(n, good)
    full = [list(range(_tile_len(n, t))) for t in range(4)]
    cases = [
        ("valid", ok, n, "ok"),
        ("valid_garbage_pads", _raw_frame(n, good, pad=0xEE), n, "ok"),
        ("header_15_bytes", ok[:15], n, 1),
        ("magic", _set_header(ok, magic=MAGIC + 1), n, 1),
        ("tile_191", _set_header(ok, tile=191), n, 1),
        ("tile_193", _set_header(ok, tile=193), n, 1),
        ("ntiles_3", _set_header(ok, ntiles=3), n, 1),
        ("ntiles_5", _set_header(ok, ntiles=5), n, 1),
        ("count_192_middle", _raw_frame(n, [good[0], list(range(192)), good[2], good[3]]), n, "ok"),
        ("count_193_middle", _raw_frame(n, [good[0], list(range(192)) + [191], good[2], good[3]]), n, 2),
        ("count_255_middle", _raw_frame(n, [good[0], good[1], list(range(192)) + [191] * 63, good[3]]), n, 2),
        ("last_count_len", _raw_frame(n, good[:3] + [list(range(last))]), n, "ok"),
        ("last_count_len_plus_1", _raw_frame(n, good[:3] + [list(range(last)) + [last - 1]]), n, 2),
        ("sum_equals_pos", _set_header(ok, pos=10), n, "ok"),
        ("sum_above_pos", _set_header(ok, pos=9), n, 3),
        ("sum_below_pos", np.append(_set_header(ok, pos=11), np.uint8(0)), n, 3),
        ("pos_n", _raw_frame(n, full), n, "ok"),
        ("pos_n_plus_1", _raw_frame(n, [full[0], full[1] + [191], full[2], full[3]]), n, 2),
        ("offset_191", _raw_frame(n, [good[0], [0, 40, 191], good[2], good[3]]), n, "ok"),
        ("offset_192", _raw_frame(n, [good[0], [0, 40, 192], good[2], good[3]]), n, 4),
        ("offset_255", _raw_frame(n, [good[0], [0, 40, 255], good[2], good[3]]), n, 4),
        ("last_offset_len_minus_1", _raw_frame(n, good[:3] + [[0, last - 1]]), n, "ok"),
        ("last_offset_len", _raw_frame(n, good[:3] + [[0, last]]), n, 4),
        ("last_offset_255", _raw_frame(n, good[:3] + [[0, 255]]), n, 4),
        ("ascending_offsets", _raw_frame(n, [good[0], [0, 40, 41], good[2], good[3]]), n, "ok"),
        ("equal_offsets", _raw_frame(n, [good[0], [0, 40, 40], good[2], good[3]]), n, 4),
        ("descending_offsets", _raw_frame(n, [good[0], [0, 41, 40], good[2], good[3]]), n, 4),
        ("descending_first_pair", _raw_frame(n, [[5, 1, 9], good[1], good[2], good[3]]), n, 4),
    ]
    # k_wire_check compares each entry with the one before it, which a different lane or loop iteration of the warp
    # handles at entries 32 and 64 of a tile: a near-full tile with the fault there, and the valid tile beside them
    near_full = [o for o in range(192) if o not in (100, 150)]         # 190 entries, strictly ascending
    for at in (32, 64):
        eq, desc = list(near_full), list(near_full)
        eq[at] = eq[at - 1]
        desc[at - 1], desc[at] = desc[at], desc[at - 1]
        cases += [(f"near_full_tile_equal_at_{at}", _raw_frame(n, [good[0], eq, good[2], good[3]]), n, 4),
                  (f"near_full_tile_descending_at_{at}", _raw_frame(n, [good[0], desc, good[2], good[3]]), n, 4)]
    cases += [
        ("near_full_tile", _raw_frame(n, [good[0], near_full, good[2], good[3]]), n, "ok"),
        ("buffer_exact", ok, n, "ok"),
        ("buffer_one_short", ok[:-1], n, 5),
        ("empty_frame", _raw_frame(n, [[], [], [], []]), n, "ok"),
        ("one_tile_partial", _raw_frame(150, [[0, 149]]), 150, "ok"),
        ("one_tile_partial_offset_150", _raw_frame(150, [[0, 150]]), 150, 4),
    ]
    return cases


HAND_BUILT = _hand_built()
# what the device decoder must refuse: every malformed hand-built frame of the 70x3 geometry but the short buffer
MALFORMED = {name: buf for name, buf, n, want in HAND_BUILT if want not in ("ok", 5) and n == 3 * MAL_W * MAL_H}


@pytest.mark.parametrize("case", range(len(HAND_BUILT)), ids=[c[0] for c in HAND_BUILT])
def test_reference_decoder_on_hand_built_frames(case):
    name, buf, n, want = HAND_BUILT[case]
    got = _decode_reference(buf, n)
    if want == "ok":
        assert not isinstance(got, int), (name, got)
    else:
        assert got == want, name
    if want != 5:  # the device decoder applies every rule but the buffer length
        assert _decode_reference(buf, n, host=False) == got, name


@pytest.mark.parametrize("case", range(len(HAND_BUILT)), ids=[c[0] for c in HAND_BUILT])
def test_host_parser_on_hand_built_frames(case):
    from cudavideostream_b200 import wire
    name, buf, n, want = HAND_BUILT[case]
    w, h = (MAL_W, MAL_H) if n == 3 * MAL_W * MAL_H else (50, 1)
    assert _parse_verdict(buf, w, h) == _ref_verdict(buf, n), name
    # without a geometry the parser checks ntiles against the header's own and takes every tile as 192 bytes long
    nt = struct.unpack_from("<I", buf, 8)[0] if buf.size >= 16 else 0
    want_loose = _ref_verdict(buf, TILE * nt) if buf.size >= 16 else None
    try:
        pos, xs, diff = wire.parse(buf)
        loose = xs.tolist(), diff.tolist()
    except ValueError:
        loose = None
    assert loose == want_loose, name


def test_reference_decoder_and_host_parser_agree_on_mutated_frames():
    corpus = _mutations(600, 5)
    verdicts = []
    for w, h, buf in corpus:
        n = 3 * w * h
        ref = _ref_verdict(buf, n)
        assert _parse_verdict(buf, w, h) == ref
        if ref is not None:
            assert ref[0] == sorted(set(ref[0])) and all(0 <= x < n for x in ref[0])
        verdicts.append(ref is not None)
    # the corpus holds both kinds in numbers
    assert 100 <= sum(verdicts) <= len(corpus) - 100, sum(verdicts)


def test_host_parser_refuses_a_short_buffer():
    from cudavideostream_b200 import wire
    n = 3 * MAL_W * MAL_H
    ok = _raw_frame(n, [[1, 5, 9], [0], [], [3]])
    for cut in (0, 8, 15, 16, 31, ok.size - 1):
        with pytest.raises(ValueError):
            wire.parse(ok[:cut], (MAL_W, MAL_H))
        with pytest.raises(ValueError):
            wire.parse(ok[:cut])
    assert wire.parse(ok, (MAL_W, MAL_H))[0] == 5


def test_wire_size_is_computed_in_64_bits(cvs):
    lib = cvs.load_library()
    for w, h in [(70, 3), (1920, 1080), (3840, 2160)]:
        n = 3 * w * h
        bound = int(lib.cvs_wire_bound(w, h))
        assert bound == 16 + _pad16(_ntiles(n)) + _pad16(n) + n
        for nt in (_ntiles(n), 0xFFFFFFF0, 0xFFFFFFF1, 0xFFFFFFFF):
            for pos in (0, n, n + 1, 0xFFFFFFF0, 0xFFFFFFF1, 0xFFFFFFFF):
                hdr = C.create_string_buffer(struct.pack("<4I", MAGIC, pos, nt, TILE), 16)
                got = int(lib.cvs_wire_size(C.addressof(hdr)))
                assert got >= 16 + _pad16(nt) + _pad16(pos) + pos, (w, h, nt, pos)
                if pos > n or nt > _ntiles(n):
                    assert got > bound, (w, h, nt, pos)
                if (nt, pos) == (_ntiles(n), n):
                    assert got == bound
        hdr = C.create_string_buffer(struct.pack("<4I", MAGIC + 1, 0, 1, TILE), 16)
        assert int(lib.cvs_wire_size(C.addressof(hdr))) == 0


# ------------------------------------------------------------------ GPU: designed frames through encoder and decoder
class _Rig:
    """One geometry: a random base frame, a stream, pinned and pageable wire buffers with guard bytes after
    cvs_wire_bound, and the device buffers of the decoder with guard bands of G bytes on both sides."""

    def __init__(self, cvs, oracle, w, h, seed):
        import torch
        from cudavideostream_b200 import wire
        self.cvs, self.oracle, self.torch, self.wire = cvs, oracle, torch, wire
        self.w, self.h, self.n = w, h, 3 * w * h
        self.nt = _ntiles(self.n)
        self.last = _tile_len(self.n, self.nt - 1)
        self.bound = wire.bound(w, h)
        self.rng = np.random.default_rng(seed)
        self.base = self.rng.integers(0, 256, size=self.n, dtype=np.uint8)
        self.s = cvs.Stream(w, h, self.base)
        self.pinned = cvs.alloc_host(self.bound + G)
        self.st = torch.cuda.current_stream().cuda_stream
        self.d_scr = torch.zeros(wire.scratch_words(w, h), dtype=torch.int32, device="cuda")
        self.d_base = torch.from_numpy(self.base).cuda()
        self._ranks = None

    def close(self):
        self.s.close()
        self.pinned.free()

    # --- designed frames
    def frame(self, mask, prev=None):
        """Bytes under the mask move by 100..156 (mod 256) from prev (the base frame), every other byte stays: at
        threshold 20 exactly the masked bytes change, and the stream's reference becomes the frame."""
        prev = self.base if prev is None else prev
        d = self.rng.integers(100, 157, size=self.n, dtype=np.int16)
        moved = ((prev.astype(np.int16) + d) & 255).astype(np.uint8)
        return np.where(mask, moved, prev)

    def ranks(self):
        if self._ranks is None:
            keys = self.rng.random((self.nt, TILE))
            keys[-1, self.last:] = 2.0
            order = np.argsort(keys, axis=1)
            self._ranks = np.empty((self.nt, TILE), dtype=np.uint8)
            np.put_along_axis(self._ranks, order, np.arange(TILE, dtype=np.uint8)[None, :], axis=1)
        return self._ranks

    def mask_from_counts(self, counts):
        counts = np.asarray(counts, dtype=np.int64)
        lens = np.full(self.nt, TILE)
        lens[-1] = self.last
        assert (counts >= 0).all() and (counts <= lens).all()
        return (self.ranks() < counts[:, None]).reshape(-1)[:self.n]

    def random_counts(self):
        c = self.rng.integers(0, TILE + 1, size=self.nt)
        c[-1] = min(c[-1], self.last)
        return c

    def pattern(self, name):
        n, nt = self.n, self.nt
        m = np.zeros(nt * TILE, dtype=bool)
        if name == "full":
            m[:] = True
        elif name == "offset_0":
            m[::TILE] = True
        elif name == "offset_191":
            m[TILE - 1::TILE] = True
            m[n - 1] = True
        elif name == "alternate":
            m.reshape(nt, TILE)[::2] = True
        elif name == "random":
            return self.mask_from_counts(self.random_counts())
        elif name == "empty":
            pass
        return m[:n]

    # --- encoder
    def encode(self, mask, tag):
        """The frame through cvs_submit_wire into the pinned buffer and into a pageable one; both must be
        _encode_numpy of the oracle's payload, and the oracle's count the designed one."""
        f = np.ascontiguousarray(self.frame(mask))
        opos, oxs, odiff, _, _ = self.oracle.diff_compact(f, self.base, THR)
        assert opos == int(mask.sum()), f"{tag}: the construction gives {opos} changes, designed {int(mask.sum())}"
        want = _encode_numpy(oxs, odiff, self.n)
        pageable = np.empty(self.bound + G, dtype=np.uint8)
        for kind, buf in (("pinned", self.pinned.array()), ("pageable", pageable)):
            buf[:] = 0xA5
            self.s.reset(self.base)
            self.s.wait(self.s.submit_wire_raw(f.ctypes.data, buf.ctypes.data, None, ""))
            assert bool((buf[self.bound:] == 0xA5).all()), f"{tag} {kind}: write past cvs_wire_bound"
            assert self.wire.size_of(buf) == want.size, f"{tag} {kind}: size"
            bad = np.flatnonzero(buf[:want.size] != want)
            assert bad.size == 0, f"{tag} {kind}: {bad.size} encoded bytes differ, first at {bad[0]}"
        return want, oxs, odiff

    # --- decoder
    def guarded(self, nbytes, fill=None):
        torch = self.torch
        raw = torch.full((nbytes + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
        if fill is not None:
            raw[G:G + nbytes] = fill
        return raw

    def decode(self, buf, outputs=("frame", "xs", "diff", "pos")):
        """Decodes buf on the device into fresh guarded outputs (frame pre-filled with the base frame, the rest with
        0xA5).  Returns (refused, outputs before, outputs after)."""
        torch, n = self.torch, self.n
        wbytes = max(self.bound, buf.size)
        d_wire = torch.full((wbytes + G,), 0xA5, dtype=torch.uint8, device="cuda")
        d_wire[:buf.size] = torch.from_numpy(buf).cuda()
        raw = {"frame": self.guarded(n, self.d_base), "xs": self.guarded(4 * n), "diff": self.guarded(n),
               "pos": self.guarded(4)}
        before = {k: v.clone() for k, v in raw.items()}
        ptr = {k: (raw[k].data_ptr() + G if k in outputs else 0) for k in raw}
        self.wire.decode_device(d_wire.data_ptr(), self.d_scr.data_ptr(), self.w, self.h, d_frame=ptr["frame"],
                                d_xs=ptr["xs"], d_diff=ptr["diff"], d_pos=ptr["pos"], stream=self.st)
        try:
            self.wire.decode_status(self.d_scr.data_ptr(), self.w, self.h, self.st)
            refused = False
        except self.cvs.CVSError as e:
            assert e.status == 1, e
            refused = True
        return refused, before, raw

    def check_decoded(self, buf, xs, diff, tag, combos=(("frame",), ("xs", "diff", "pos"), ("frame", "xs", "diff", "pos"), ())):
        """Each combination of outputs gives the payload (xs ascending, diff) and frame + diff; nothing else moves."""
        torch, n = self.torch, self.n
        d_xs = torch.from_numpy(np.ascontiguousarray(xs, dtype=np.int32)).cuda()
        d_df = torch.from_numpy(np.ascontiguousarray(diff, dtype=np.uint8)).cuda()
        pos = int(d_xs.numel())
        want_frame = self.d_base.clone()
        want_frame[d_xs.long()] += d_df
        for outputs in combos:
            refused, before, raw = self.decode(buf, outputs)
            assert not refused, f"{tag}: a valid frame was refused"
            for k in ("frame", "xs", "diff", "pos"):
                if k not in outputs:
                    assert torch.equal(raw[k], before[k]), f"{tag} {outputs}: {k} was written"
                    continue
                r = raw[k]
                assert torch.equal(r[:G], before[k][:G]) and torch.equal(r[-G:], before[k][-G:]), f"{tag}: {k} guard"
            if "frame" in outputs:
                assert torch.equal(raw["frame"][G:G + n], want_frame), f"{tag}: frame + diff"
            if "pos" in outputs:
                assert int(raw["pos"][G:G + 4].view(torch.int32)[0]) == pos, f"{tag}: pos"
            if "xs" in outputs:
                got = raw["xs"][G:G + 4 * n].view(torch.int32)
                assert torch.equal(got[:pos], d_xs), f"{tag}: xs"
                assert torch.equal(raw["xs"][G + 4 * pos:], before["xs"][G + 4 * pos:]), f"{tag}: xs past pos"
            if "diff" in outputs:
                assert torch.equal(raw["diff"][G:G + pos], d_df), f"{tag}: diff"
                assert torch.equal(raw["diff"][G + pos:], before["diff"][G + pos:]), f"{tag}: diff past pos"

    def check_frame(self, mask, tag):
        enc, xs, diff = self.encode(mask, tag)
        if self.n <= REF_DECODE_MAX:
            assert _decode_reference(enc, self.n) == (xs.tolist(), diff.tolist()), tag
        self.check_decoded(enc, xs, diff, tag)
        # garbage in the pad bytes after the counts and after the offsets changes nothing
        g = enc.copy()
        o0 = 16 + _pad16(self.nt)
        g[16 + self.nt:o0] = self.rng.integers(0, 256, size=o0 - 16 - self.nt, dtype=np.uint8)
        g[o0 + xs.size:o0 + _pad16(xs.size)] = self.rng.integers(0, 256, size=_pad16(xs.size) - xs.size, dtype=np.uint8)
        if self.n <= REF_DECODE_MAX:
            assert _decode_reference(g, self.n) == (xs.tolist(), diff.tolist()), tag
        self.check_decoded(g, xs, diff, f"{tag} (garbage in the pads)", combos=(("frame", "xs", "diff", "pos"),))

    def check_refused(self, buf, tag):
        """The unfixed decoder applied such frames: the test first makes sure its furthest reach -- offset 255 in the
        last tile, as many entries as the counts add up to, the offset and value bytes those entries read -- lies in
        the guard bands.  A refused frame leaves every output and guard byte as it was."""
        n, nt = self.n, self.nt
        s = int(buf[16:16 + nt].astype(np.int64).sum())
        assert (nt - 1) * TILE + 256 <= n + G, tag
        assert 4 * s <= 4 * n + G and s <= n + G, tag
        assert 16 + _pad16(nt) + _pad16(s) + s <= max(self.bound, buf.size) + G, tag
        refused, before, raw = self.decode(buf)
        assert refused, f"{tag}: a malformed frame was accepted"
        for k in raw:
            assert self.torch.equal(raw[k], before[k]), f"{tag}: {k} was written"


@pytest.fixture
def rig(cvs, oracle):
    made = []

    def make(w, h, seed=0):
        r = _Rig(cvs, oracle, w, h, seed)
        made.append(r)
        return r
    yield make
    for r in made:
        r.close()


@pytest.mark.gpu
def test_every_residue_of_the_last_tile(rig):
    """Widths 64..127 at height 1: n = 3w takes every residue mod 192.  Last tile full, empty, and one entry at its
    last byte."""
    assert len({(3 * v) % TILE for v in range(64, 128)}) == 64
    for w in range(64, 128):
        r = rig(w, 1, seed=w)
        c = r.random_counts()
        c[-1] = r.last
        r.check_frame(r.mask_from_counts(c), f"{w}x1 last full")
        c = r.random_counts()
        c[-1] = 0
        r.check_frame(r.mask_from_counts(c), f"{w}x1 last empty")
        m = np.zeros(r.n, dtype=bool)
        m[r.n - 1] = True
        r.check_frame(m, f"{w}x1 one entry at len(last) - 1")
        r.close()


PATTERNS = ("full", "offset_0", "offset_191", "alternate", "random", "empty")


# ntiles 1, 1 (partial), 15, 16, 17; 1023, 1024, 1024 (last tile 189 bytes), 1025; 1080p and 4K
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(64, 1), (10, 5), (60, 16), (64, 16), (68, 16), (1023, 64), (256, 256), (255, 257),
                                 (320, 205), (1920, 1080), (3840, 2160)])
def test_per_tile_patterns(rig, w, h):
    r = rig(w, h, seed=w * h)
    assert r.nt in (1, 15, 16, 17, 1023, 1024, 1025, 32400, 129600)
    for p in PATTERNS:
        m = r.pattern(p)
        r.check_frame(m, f"{w}x{h} {p}")


@pytest.mark.gpu
def test_every_payload_size_mod_16(rig):
    """k_wire_pack writes 16 entries per thread and then the tail: every pos % 16, below and above 16."""
    r = rig(64, 16, seed=3)
    for pos in list(range(16)) + list(range(48, 64)):
        m = np.zeros(r.n, dtype=bool)
        m[r.rng.choice(r.n, size=pos, replace=False)] = True
        r.check_frame(m, f"pos {pos}")


@pytest.mark.gpu
def test_device_payloads_of_a_sequence(rig, cvs, oracle):
    """cvs_run_sequence_device, then cvs_wire_encode_device frame by frame on d_xs + t*cap and d_diff + t*cap.  With a
    capacity below a frame's count the header's pos is the capacity and the body the first cap entries; a capacity
    that is not a multiple of 16 misaligns d_diff from frame 1 on."""
    import torch
    from cudavideostream_b200 import wire
    r = rig(256, 16, seed=9)                   # n = 12288, 64 tiles
    n, T = r.n, 6
    frames, counts = [], []
    for t in range(T):
        m = r.mask_from_counts(r.random_counts()) if t % 3 else r.pattern(("full", "alternate")[t % 2])
        frames.append(r.frame(m, frames[-1] if frames else None))
        counts.append(int(m.sum()))
    oc = oracle.OracleCore(r.w, r.h, r.base)
    pay = []
    for t in range(T):
        opos, oxs, odiff, _, _ = oc.exec_core(frames[t])
        assert opos == counts[t], t
        pay.append((oxs, odiff))
    oc.close()
    st = r.st
    d_frames = torch.from_numpy(np.stack(frames)).cuda().reshape(-1)
    below = sorted(counts)[T // 2] // 16 * 16
    assert any(c > below for c in counts) and any(c <= below for c in counts)
    for cap in (n, below, below + 4):
        s = cvs.Stream(r.w, r.h, r.base)
        d_pos = torch.zeros(T, dtype=torch.int32, device="cuda")
        d_xs = torch.zeros(T * cap, dtype=torch.int32, device="cuda")
        d_df = torch.zeros(T * cap, dtype=torch.uint8, device="cuda")
        s.run_sequence_device(d_frames.data_ptr(), n, T, d_pos.data_ptr(), d_xs.data_ptr(), d_df.data_ptr(), cap,
                              cuda_stream=st)
        torch.cuda.synchronize()
        if cap >= max(counts):
            s.sequence_status()
        else:
            with pytest.raises(cvs.CVSError):
                s.sequence_status()
        s.close()
        assert d_pos.cpu().tolist() == counts
        d_wire = torch.full((wire.bound(r.w, r.h) + G,), 0xA5, dtype=torch.uint8, device="cuda")
        for t in range(T):
            args = (d_xs.data_ptr() + 4 * t * cap, d_df.data_ptr() + t * cap, d_pos.data_ptr() + 4 * t, cap, r.w, r.h,
                    r.d_scr.data_ptr(), d_wire.data_ptr(), st)
            if cap % 16:
                if t == 0:
                    wire.encode_device(*args)
                else:
                    with pytest.raises(cvs.CVSError) as e:
                        wire.encode_device(*args)
                    assert e.value.status == 4, t  # CVS_ERR_ALIGN
                    break
            else:
                d_wire.fill_(0xA5)
                wire.encode_device(*args)
            torch.cuda.synchronize()
            enc = d_wire.cpu().numpy()
            k = min(counts[t], cap)
            want = _encode_numpy(pay[t][0][:k], pay[t][1][:k], n)
            assert struct.unpack_from("<I", enc, 4)[0] == k, (cap, t)
            assert np.array_equal(enc[:want.size], want), (cap, t)
            assert bool((enc[wire.bound(r.w, r.h):] == 0xA5).all()), (cap, t)
            if cap % 16 == 0:
                r.check_decoded(enc[:want.size], pay[t][0][:k], pay[t][1][:k], f"cap {cap} frame {t}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(MALFORMED))
def test_malformed_frame_is_refused_and_writes_nothing(rig, case):
    r = rig(MAL_W, MAL_H, seed=4)
    buf = MALFORMED[case]
    assert isinstance(_decode_reference(buf, r.n), int), case
    r.check_refused(buf, case)


@pytest.mark.gpu
def test_mutated_frames_get_the_reference_verdict_on_the_device(rig):
    rigs = {}
    corpus = _mutations(300, 6)
    accepted = 0
    for i, (w, h, buf) in enumerate(corpus):
        if (w, h) not in rigs:
            rigs[(w, h)] = rig(w, h, seed=w)
        r = rigs[(w, h)]
        ref = _ref_verdict(buf, r.n)
        tag = f"{w}x{h} mutation {i}"
        if ref is None:
            r.check_refused(buf, tag)
        else:
            accepted += 1
            r.check_decoded(buf, np.array(ref[0], dtype=np.int32), np.array(ref[1], dtype=np.uint8), tag)
        assert _parse_verdict(buf, w, h) == ref, tag
    assert 50 <= accepted <= len(corpus) - 50, accepted
