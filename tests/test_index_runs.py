"""CPU test of the index lane's runs (clx_lanes.h: RiceCursor::skip_run, IndexLane::run) through the host harness.

The index kernel steps over the Rice codes of every channel but the last in runs of up to IndexLane::RUN groups of
eight codes behind one ring refill.  A run commits group by group and ends early at a group that does not fit the
32-bit window; a partition with fewer groups left than a run is finished by a shorter run.  Whatever the run length,
the lane must record the same residual start bit for every subframe, and the frames must decode as the oracle
decodes them.  The streams below are built to reach every way a run ends."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import claxon_b200 as cb
from claxon_b200 import synth
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "tools", "scratch", "seq_host_runs.so")
SRC = os.path.join(ROOT, "tools", "seq_host.cpp")
HDR = os.path.join(ROOT, "claxon_b200", "csrc", "clx_lanes.h")
RUN = 4  # IndexLane::RUN


@pytest.fixture(scope="module")
def harness():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas",
                               "-I", os.path.join(ROOT, "include"), "-o", SO, SRC])
    L = C.CDLL(SO)
    L.seq_host_index.restype = C.c_int
    L.seq_host_index.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
    L.seq_host_decode.restype = C.c_int
    L.seq_host_decode.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                  C.c_void_p]
    return L


def index_walk(L, data, descs, run_groups):
    """res_bit per (frame, channel slot), status per frame, run statistics (see seq_host_index)."""
    n = len(descs)
    ch = 1
    while ch < int(descs["n_channels"].max()):
        ch *= 2
    padded = np.concatenate([data, np.zeros(256, np.uint8)])
    res_bit = np.zeros(n * ch, np.uint32)
    status = np.zeros(n, np.int32)
    stats = np.zeros(10, np.uint64)
    got = L.seq_host_index(padded.ctypes.data, data.size, descs.ctypes.data, n, run_groups, res_bit.ctypes.data,
                           status.ctypes.data, stats.ctypes.data)
    assert got == ch
    return res_bit.reshape(n, ch), status, stats


def check_frames(L, data, offs, lens):
    """Index walks with runs of 1 .. RUN groups agree; the full lane path agrees with the oracle.  Returns the
    statistics of the walk with runs of RUN groups."""
    data = np.ascontiguousarray(data, np.uint8)
    offs = np.asarray(offs, np.uint64)
    lens = np.asarray(lens, np.uint32)
    descs, out_elems = cb.descs_from_offsets(data, offs, lens)
    descs = np.ascontiguousarray(descs)
    bits1, st1, _ = index_walk(L, data, descs, 1)
    for g in range(2, RUN + 1):
        bits, st, stats = index_walk(L, data, descs, g)
        assert np.array_equal(st, st1), g
        assert np.array_equal(bits, bits1), g
    bad, ost, ref = O.decode_batch(data, offs, lens, descs["out_offset"], max(1, out_elems), n_threads=4,
                                   verify_crc=False)
    padded = np.concatenate([data, np.zeros(256, np.uint8)])
    out = np.full(max(1, out_elems), 0x5A5A5A5A, np.int32)
    res = np.zeros(len(offs), dtype=[("status", "<i4"), ("consumed", "<u4")])
    assert L.seq_host_decode(padded.ctypes.data, data.size, descs.ctypes.data, len(offs), 0, out.ctypes.data,
                             res.ctypes.data, None) == 0
    for i in range(len(offs)):
        if res["status"][i] != 0:
            continue
        assert ost[i] == 0, f"frame {i}: lane accepted a frame the oracle rejects with {ost[i]}"
        o, n = int(descs[i]["out_offset"]), int(descs[i]["n_channels"]) * int(descs[i]["block_size"])
        assert np.array_equal(out[o:o + n], ref[o:o + n]), i
        assert res["consumed"][i] == lens[i]
    return stats, res, ost


def check_stream(L, cfg):
    b = synth.generate(cfg)
    stats, res, ost = check_frames(L, b.data, b.frame_offsets[:-1], b.frame_lengths)
    assert (ost == 0).all() and (res["status"] == 0).all()  # valid streams are neither rejected nor declined
    return stats


def stereo(**kw):
    base = dict(n_frames=24, block_size=4096, n_channels=2, bps=16, stereo_mode=10, type_mask=8, lpc_min_order=8,
                lpc_max_order=8, qlp_precision=12, rice_mode=4, max_porder=0, residual_mean=11.5)
    base.update(kw)
    return synth.SynthConfig(**base)


def test_runs_end_on_long_codes_at_every_group(harness):
    """Codes longer than the window (one huge residual per subframe) end runs at each of their groups."""
    stats = check_stream(harness, stereo(long_unary_per_mille=1000))
    assert stats[0] > 1000
    assert all(stats[2 + j] > 0 for j in range(RUN)), stats


@pytest.mark.parametrize("k", [6, 7])
def test_runs_either_side_of_pair_kmax(harness, k):
    """k = 6 takes two codes per window refill, k = 7 one (PAIR_KMAX = 6); with long codes in both."""
    stats = check_stream(harness, stereo(rice_mode=k, residual_mean=float(2 ** k), long_unary_per_mille=1000))
    assert stats[0] > 100 and sum(stats[2:2 + RUN]) > 0, stats


@pytest.mark.parametrize("block_size,porder", [(4096, 7), (1280, 3), (1152, 2), (576, 2), (2304, 4), (200, 1)])
def test_partitions_shorter_than_or_equal_to_a_run(harness, block_size, porder):
    """Partitions of 32 codes end exactly where a run ends; 40, 72, 144, 288 and 100 codes end with a shorter run;
    the first partition is shorter by the predictor order."""
    stats = check_stream(harness, stereo(block_size=block_size, min_porder=porder, max_porder=porder, rice_mode=-2,
                                         rice_kmin=2, rice_kmax=9, n_frames=16))
    assert stats[0] + stats[1] > 0, stats


def test_mixed_shapes(harness):
    """Every subframe type, Rice2, wasted bits, 1..8 channels, long unary runs."""
    for seed in range(4):
        rng = np.random.default_rng(900 + seed)
        nch = int(rng.integers(2, 9))
        check_stream(harness, synth.SynthConfig(
            seed=int(rng.integers(1, 2**31)), n_frames=30, block_size=int(rng.choice([576, 1152, 4096, 4608])),
            n_channels=nch, bps=int(rng.choice([12, 16, 20, 24])), stereo_mode=-1 if nch == 2 else 0,
            type_mask=15, lpc_min_order=1, lpc_max_order=32, qlp_precision=0, rice_mode=-2, rice_kmin=0,
            rice_kmax=14, max_porder=int(rng.integers(0, 7)), rice2=2, wasted_max=3, long_unary_per_mille=20))


def test_run_at_the_end_of_the_buffer(harness):
    """A frame that is the last thing in the buffer, so that a run's look-ahead reaches past its bytes; with and
    without its footer.  (The host harness reads zeros there; the device ring's zero-fill is covered by the GPU
    parity tests.)"""
    b = synth.generate(stereo(n_frames=6))
    last = len(b.frame_lengths) - 1
    lo, n = int(b.frame_offsets[last]), int(b.frame_lengths[last])
    for cut in (0, 1, 2, 7, 16):
        data = b.data[:lo + n - cut]
        offs = [lo]
        lens = [n - cut]
        stats, res, ost = check_frames(harness, data, offs, lens)
        if cut == 0:
            assert res["status"][0] == 0


def test_truncated_frames(harness):
    """Frames cut anywhere: the index walk agrees across run lengths, and what the lane accepts is what the oracle
    accepts, bit for bit."""
    b = synth.generate(stereo(n_frames=8, long_unary_per_mille=1000))
    rng = np.random.default_rng(11)
    frames = []
    for i in range(120):
        j = int(rng.integers(0, b.n_frames))
        f = b.data[int(b.frame_offsets[j]):int(b.frame_offsets[j + 1])]
        frames.append(f[:int(rng.integers(6, f.size))].copy())
    frames = [f for f in frames if cb.parse_frame_header(f)[0] == 0]
    assert len(frames) > 50
    data = np.concatenate(frames)
    lens = np.array([f.size for f in frames], np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    check_frames(harness, data, offs, lens)
