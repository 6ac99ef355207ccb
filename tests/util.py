"""Shared helpers for the parity tests."""
import re
import time

import numpy as np

CHARS_STR = "0123456789BFPSWbkps :/"  # server/include/common.h:13


def glyph_atlas(gw=7, gh=5, seed=3):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, size=(len(CHARS_STR), gh, gw, 3), dtype=np.uint8)


def random_sequence(width, height, nframes, density, seed=0, drift=True):
    """numpy-only frame generator for small shapes: base + frames with `density` of bytes changed by a
    super-threshold delta and (optionally) sub-threshold drift on the rest."""
    rng = np.random.default_rng(seed)
    n = 3 * width * height
    base = rng.integers(0, 256, size=n, dtype=np.uint8)
    frames = np.empty((nframes, n), dtype=np.uint8)
    prev = base.astype(np.int64)
    for t in range(nframes):
        big = rng.random(n) < density
        delta = rng.integers(21, 120, size=n) * rng.choice([-1, 1], size=n)
        small = rng.integers(-3, 4, size=n) if drift else np.zeros(n, dtype=np.int64)
        cur = np.where(big, prev + delta, prev + small)
        cur = np.where((cur < 0) | (cur > 255), prev - (cur - prev), cur)
        cur = np.clip(cur, 0, 255)
        frames[t] = cur.astype(np.uint8)
        prev = cur
    return base, frames


def run_oracle_sequence(oracle, width, height, base, frames, **kw):
    """Runs OracleCore frame by frame.  Returns list of (pos, xs, diff, show) and the final reference."""
    core = oracle.OracleCore(width, height, base, **kw)
    text = kw.pop("text", "") if "text" in kw else ""
    out = []
    for f in frames:
        pos, xs, diff, show, _ = core.exec_core(f, text)
        out.append((pos, xs, diff, show))
    ref = core.reference()
    core.close()
    return out, ref


def strip_dht(jpg: bytes) -> bytes:
    """The JPEG without its DHT segments (MJPG as cameras send it: the standard Huffman tables are implied)."""
    out, i = bytearray(jpg[:2]), 2
    while i < len(jpg):
        m, ln = jpg[i + 1], (jpg[i + 2] << 8) | jpg[i + 3]
        if m == 0xDA:
            out += jpg[i:]
            break
        if m != 0xC4:
            out += jpg[i:i + 2 + ln]
        i += 2 + ln
    return bytes(out)


_ZIGZAG = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
           35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]


def transcode_huffman(jpg: bytes, coef: np.ndarray, hs: int, vs: int, ncomp: int, dc_len: int, ac_len: int,
                      restart_interval: int = 0) -> bytes:
    """Re-encodes the entropy-coded segment of a baseline JPEG (no restart intervals) with Huffman tables in which EVERY
    DC code is dc_len bits and EVERY AC code ac_len bits long (one table pair for all components).  `coef` are the file's
    quantised coefficients [nblocks, 64] in scan order / natural order with absolute DC (oracle.jpeg_coefficients), so the
    result decodes to the same picture.  Long uniform codes give a decoder's look-up tables their worst case: hundreds
    of distinct long prefixes.  With restart_interval > 0 the stream gets a DRI segment and an RSTn marker after every
    restart_interval MCUs (DC prediction restarts from 0 there).  DC differences must stay within category 11
    (|difference| <= 2047), AC values within category 10."""
    dc_syms = list(range(12))
    ac_syms = [0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 11)]
    assert len(dc_syms) <= (1 << dc_len) - 1 and len(ac_syms) <= (1 << ac_len) - 1
    dc_code = {s: (i, dc_len) for i, s in enumerate(dc_syms)}
    ac_code = {s: (i, ac_len) for i, s in enumerate(ac_syms)}

    def dht(tc, syms, length):
        bits = [0] * 16
        bits[length - 1] = len(syms)
        body = bytes([tc << 4]) + bytes(bits) + bytes(syms)
        return b"\xff\xc4" + (len(body) + 2).to_bytes(2, "big") + body

    # header: everything up to SOS except DHT; SOS rewritten to select table 0 / 0 for every component
    out, i = bytearray(jpg[:2]), 2
    while True:
        m, ln = jpg[i + 1], (jpg[i + 2] << 8) | jpg[i + 3]
        if m == 0xDA:
            break
        assert m != 0xDD, "source must not use restart intervals"
        if m != 0xC4:
            out += jpg[i:i + 2 + ln]
        i += 2 + ln
    out += dht(0, dc_syms, dc_len) + dht(1, ac_syms, ac_len)
    if restart_interval:
        out += b"\xff\xdd\x00\x04" + restart_interval.to_bytes(2, "big")
    sos = bytearray(jpg[i:i + 2 + ln])
    for c in range(ncomp):
        sos[4 + 1 + 2 * c + 1] = 0x00
    out += sos

    acc, nacc, data = 0, 0, bytearray()

    def put(v, n):
        nonlocal acc, nacc
        acc = (acc << n) | (v & ((1 << n) - 1))
        nacc += n
        while nacc >= 8:
            b = (acc >> (nacc - 8)) & 0xFF
            data.append(b)
            if b == 0xFF:
                data.append(0)
            nacc -= 8
        acc &= (1 << nacc) - 1

    def amp(v):
        s = int(abs(v)).bit_length()
        return s, (v if v >= 0 else v + (1 << s) - 1)

    bpm = hs * vs + (2 if ncomp == 3 else 0)
    pred = [0, 0, 0]
    for b in range(coef.shape[0]):
        j = b % bpm
        m = b // bpm
        if restart_interval and j == 0 and m and m % restart_interval == 0:
            if nacc:
                put((1 << (8 - nacc)) - 1, 8 - nacc)
            data += bytes([0xFF, 0xD0 + (m // restart_interval - 1) % 8])
            pred = [0, 0, 0]
        c = 0 if (ncomp == 1 or j < hs * vs) else j - hs * vs + 1
        blk = coef[b]
        d = int(blk[0]) - pred[c]
        pred[c] = int(blk[0])
        s, a = amp(d)
        put(*dc_code[s])
        if s:
            put(a, s)
        run = 0
        last = max([k for k in range(1, 64) if blk[_ZIGZAG[k]] != 0], default=0)
        for k in range(1, last + 1):
            v = int(blk[_ZIGZAG[k]])
            if v == 0:
                run += 1
                continue
            while run >= 16:
                put(*ac_code[0xF0])
                run -= 16
            s, a = amp(v)
            put(*ac_code[(run << 4) | s])
            put(a, s)
            run = 0
        if last < 63:
            put(*ac_code[0x00])
    if nacc:
        put((1 << (8 - nacc)) - 1, 8 - nacc)
    return bytes(out) + bytes(data) + b"\xff\xd9"


# which stream / filter kernels a piece of work launched
_KERNEL = re.compile(r"(k_stream_ws_batch|k_stream_ws|k_stream|k_filter)(?:<([^<>]*)>|I((?:L[ib]\d+E)+)E)")


def kernel_id(name):
    """'k_stream_ws<1,0>' for 'void cvs::k_stream_ws<1, false>(cvs::StreamParams)' or its mangled name, None
    for any other kernel."""
    m = _KERNEL.search(name)
    if not m:
        return None
    if m.group(2) is not None:
        args = [re.sub(r"^\(\w+\)", "", a.strip()) for a in m.group(2).split(",")]
        vals = [1 if a == "true" else 0 if a == "false" else int(a) for a in args]
    else:
        vals = [int(v) for v in re.findall(r"L[ib](\d+)E", m.group(3))]
    return f"{m.group(1)}<{','.join(map(str, vals))}>"


def launched(fn):
    """Runs fn() under torch.profiler with CUDA activities (nothing is timed).  Returns fn's result and the set of
    stream / filter kernels that ran, as kernel_id names.  The session is kept open a little before and after the
    work, so that even a single kernel of a few microseconds lies well inside it."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        time.sleep(0.02)
        out = fn()
        torch.cuda.synchronize()
        time.sleep(0.02)
    return out, {k for k in (kernel_id(e.name) for e in prof.events()) if k}
