"""Payload emission of the stream kernels at the sparse / dense boundary of a back warp.

A back warp of k_stream_ws emits the entries of 32 consecutive 96-byte chunks.  With at most kWarpEntries = 512 entries
it compacts them into its shared-memory window and flushes that (the flush is shifted by the warp's global offset mod 4
and mod 16); with more it stores them straight out of the stage (emit_coop), clipped to the capacity when the warp
crosses it.  Random densities put warps far from that boundary, so the frames here give every chunk an exact number of
changed bytes: any 32 consecutive chunks hold one chunk of each residue mod 32, so the per-chunk counts fix every full
warp's total without knowing the launch geometry --
  512    16 per chunk: a full sparse window
  513    16 per chunk, 17 in chunks = r (mod 32): the smallest dense warp
  511    16 per chunk, 15 in chunks = r (mod 32)
  mixed  regions of 96, 16 and 0 per chunk with boundaries at odd chunk offsets: sparse and dense warps in one block
plus 0..15 extra changes in the frame's first chunk, which moves the global offset of every later warp through all
residues mod 16.  Changed bytes move by threshold + 1 or jump across the range (0 <-> 255), every other byte drifts by at
most the threshold.  Every path of the library runs the same frames: k_stream_ws with the reference in registers
(1080p sequences), in bands (3840x2160 sequences) and through L2 (CVS_STREAM_KERNEL=ws, a 3840x2160 single frame),
and k_stream (3840x2160 single frames, CVS_STREAM_KERNEL=v1 sequences)."""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CHUNK = 96
THR = 20
PATTERNS = ("512", "513", "511", "mixed")
SPECIAL = (0, 47, 48, 95)  # always among a chunk's changed bytes (when it has four or more)


def chunk_counts(pattern, nchunks, r, extra):
    c = np.arange(nchunks)
    if pattern == "512":
        cnt = np.full(nchunks, 16)
    elif pattern == "513":
        cnt = 16 + (c % 32 == r)
    elif pattern == "511":
        cnt = 16 - (c % 32 == r)
    else:  # an odd first region, then even ones: every boundary at an odd chunk offset
        cnt = np.empty(nchunks, dtype=np.int64)
        runs = [(2 * r + 1, 16)] + [(38, 96), (52, 16), (30, 0), (46, 96), (20, 0), (64, 16)] * (nchunks // 250 + 1)
        at = 0
        for length, v in runs:
            cnt[at:at + length] = v
            at += length
            if at >= nchunks:
                break
    cnt = cnt.astype(np.int64)
    cnt[0] += extra
    assert cnt.max() <= CHUNK
    return cnt


@functools.lru_cache(maxsize=None)
def _ranks(nchunks, seed):
    """Per chunk, the rank of each byte in a seeded order that starts with SPECIAL."""
    keys = np.random.default_rng(seed).random((nchunks, CHUNK))
    keys[:, SPECIAL] = -1.0
    order = np.argsort(keys, axis=1, kind="stable")
    ranks = np.empty((nchunks, CHUNK), dtype=np.uint8)
    np.put_along_axis(ranks, order, np.arange(CHUNK, dtype=np.uint8)[None, :], axis=1)
    return ranks


def next_frame(ref, cnt, t, seed):
    """A frame with exactly cnt[c] bytes of chunk c further than THR from the reference ref.  Returns (frame, new ref)."""
    n = ref.size
    nchunks = n // CHUNK
    rng = np.random.default_rng((seed, t))
    ranks = np.roll(_ranks(nchunks, seed), 7 * t, axis=0)  # other positions every frame
    changed = (ranks < cnt[:, None].astype(np.uint8)).reshape(-1)
    r = ref.astype(np.int16)
    kind = rng.integers(0, 3, size=n, dtype=np.int8)
    up, down = r + THR + 1, r - THR - 1
    big = np.where(kind == 0, np.where(up <= 255, up, down), np.where(down >= 0, down, up))
    big = np.where(kind == 2, np.where(r < 128, 255, 0), big)
    small = np.clip(r + rng.integers(-THR, THR + 1, size=n, dtype=np.int16), 0, 255)
    cur = np.where(changed, big, small).astype(np.uint8)
    return cur, np.where(changed, cur, ref)


@functools.lru_cache(maxsize=None)
def scenario(width, height, nframes, seed):
    """Base frame, frames and the designed count of every frame.  Frame t: pattern t % 4, extra changes (t // 4) % 16
    in chunk 0, r = (5t + 3) % 32."""
    n = 3 * width * height
    assert n % CHUNK == 0
    base = np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8)
    frames = np.empty((nframes, n), dtype=np.uint8)
    counts = []
    ref = base
    for t in range(nframes):
        cnt = chunk_counts(PATTERNS[t % 4], n // CHUNK, (5 * t + 3) % 32, (t // 4) % 16)
        frames[t], ref = next_frame(ref, cnt, t, seed)
        counts.append(int(cnt.sum()))
    return base, frames, counts


def _check_frame(t, oc, frame, count, pos, xs, diff):
    opos, oxs, odiff, _, _ = oc.exec_core(frame)
    assert opos == count, f"frame {t}: the construction gives {opos} changes, designed {count}"
    assert pos == opos, f"frame {t}: count {pos} != {opos}"
    bad = np.flatnonzero(xs != oxs)
    assert bad.size == 0, f"frame {t}: xs differ at {bad.size} entries, first {bad[0]}"
    bad = np.flatnonzero(diff != odiff)
    assert bad.size == 0, f"frame {t}: diff differs at {bad.size} entries, first {bad[0]} (xs {oxs[bad[0]]})"


def _run_sequence(cvs, oracle, w, h, nframes, seed):
    import torch
    base, frames, counts = scenario(w, h, nframes, seed)
    n = 3 * w * h
    cap = n
    d_frames = torch.from_numpy(frames).cuda().reshape(-1)
    d_pos = torch.zeros(nframes, dtype=torch.int32, device="cuda")
    d_xs = torch.empty(nframes * cap, dtype=torch.int32, device="cuda")
    d_diff = torch.empty(nframes * cap, dtype=torch.uint8, device="cuda")
    s = cvs.Stream(w, h, base)
    s.run_sequence_device(d_frames.data_ptr(), n, nframes, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(), cap,
                          cuda_stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    s.sequence_status()
    pos = d_pos.cpu().numpy()
    oc = oracle.OracleCore(w, h, base)
    for t in range(nframes):
        p = int(pos[t])
        _check_frame(t, oc, frames[t], counts[t], p, d_xs[t * cap:t * cap + p].cpu().numpy(),
                     d_diff[t * cap:t * cap + p].cpu().numpy())
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()


def _run_single_frames(cvs, oracle, w, h, nframes, seed):
    base, frames, counts = scenario(w, h, nframes, seed)
    s = cvs.Stream(w, h, base)
    oc = oracle.OracleCore(w, h, base)
    for t in range(nframes):
        pos, xs, diff, _ = s.exec(frames[t])
        _check_frame(t, oc, frames[t], counts[t], pos, xs, diff)
    assert np.array_equal(s.reference(), oc.reference())
    s.close()
    oc.close()


@pytest.mark.parametrize("kernel", ["default", "v1"])
def test_1080p_sequence(cvs, oracle, monkeypatch, kernel):
    # default: k_stream_ws, reference in registers; v1: k_stream.  64 frames: every pattern with every extra count
    if kernel == "default":
        monkeypatch.delenv("CVS_STREAM_KERNEL", raising=False)
    else:
        monkeypatch.setenv("CVS_STREAM_KERNEL", kernel)
    _run_sequence(cvs, oracle, 1920, 1080, 64, 11)


def test_4k_sequence_in_bands(cvs, oracle, monkeypatch):
    monkeypatch.delenv("CVS_STREAM_KERNEL", raising=False)
    _run_sequence(cvs, oracle, 3840, 2160, 16, 12)


@pytest.mark.parametrize("kernel", ["default", "ws"])
def test_4k_single_frames(cvs, oracle, monkeypatch, kernel):
    # default: k_stream in segments; ws: k_stream_ws with the reference through L2 (REFREG = false)
    if kernel == "default":
        monkeypatch.delenv("CVS_STREAM_KERNEL", raising=False)
    else:
        monkeypatch.setenv("CVS_STREAM_KERNEL", kernel)
    _run_single_frames(cvs, oracle, 3840, 2160, 4, 13)


def test_capacity_at_the_dense_boundary(cvs, oracle, monkeypatch):
    """The 513 pattern (every full warp dense) with the last 128 chunks full (96 each).  A capacity equal to the count
    is no overflow; the next smaller capacity (capacities are multiples of 4), or a cut in the middle of the full
    chunks, reports CVS_ERR_CAPACITY and delivers exactly the first `cap` entries without writing past them."""
    import torch
    monkeypatch.delenv("CVS_STREAM_KERNEL", raising=False)
    w, h, Gd = 1920, 1080, 4096
    n = 3 * w * h
    nchunks = n // CHUNK
    base = np.random.default_rng(14).integers(0, 256, size=n, dtype=np.uint8)
    cnt = chunk_counts("513", nchunks, 7, 0)
    cnt[-128:] = CHUNK
    cnt[0] += -int(cnt.sum()) % 4  # a count that is itself a valid capacity
    f, _ = next_frame(base, cnt, 0, 14)
    count = int(cnt.sum())
    assert count % 4 == 0
    oc = oracle.OracleCore(w, h, base)
    opos, oxs, odiff, _, _ = oc.exec_core(f)
    assert opos == count
    d_frame = torch.from_numpy(f).cuda()
    st = torch.cuda.current_stream().cuda_stream

    def guarded(nbytes, dtype=torch.uint8):
        raw = torch.full((nbytes + 2 * Gd,), 0xA5, dtype=torch.uint8, device="cuda")
        return raw, raw[Gd:Gd + nbytes].view(dtype)

    for cap in (count, count - 4, count - 64 * CHUNK - 8):
        raw_p, d_pos = guarded(4, torch.int32)
        raw_x, d_xs = guarded(4 * cap, torch.int32)
        raw_d, d_diff = guarded(cap)
        s = cvs.Stream(w, h, base)
        s.run_sequence_device(d_frame.data_ptr(), n, 1, d_pos.data_ptr(), d_xs.data_ptr(), d_diff.data_ptr(), cap,
                              cuda_stream=st)
        torch.cuda.synchronize()
        if cap == count:
            s.sequence_status()
        else:
            with pytest.raises(cvs.CVSError) as e:
                s.sequence_status()
            assert e.value.status == 5, cap  # CVS_ERR_CAPACITY
        assert int(d_pos[0]) == count, cap
        assert np.array_equal(d_xs.cpu().numpy(), oxs[:cap]), cap
        assert np.array_equal(d_diff.cpu().numpy(), odiff[:cap]), cap
        for raw in (raw_p, raw_x, raw_d):
            assert bool((raw[:Gd] == 0xA5).all()) and bool((raw[-Gd:] == 0xA5).all()), cap
        assert np.array_equal(s.reference(), oc.reference()), cap
        s.close()
    oc.close()
