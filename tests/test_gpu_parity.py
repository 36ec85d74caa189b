"""Parity tests proper (-m gpu): the CUDA path, called through the C ABI, against
  (1) the committed golden fixtures (reference test streams, PCM pinned by STREAMINFO MD5),
  (2) the CPU oracle on seeded synthetic inputs, incl. every error the reference defines,
  (3) size-independent properties at BASELINE.json's full sizes.
Bit-exact everywhere: this path is integer only."""
import hashlib
import json
import os

import numpy as np
import pytest

import claxon_b200 as cb
from claxon_b200 import synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAT = json.load(open(os.path.join(ROOT, "tests", "golden", "kat.json")))


def gpu_decode(ctx, data, offsets, lengths):
    descs, out_elems = cb.descs_from_offsets(data, offsets, lengths)
    out, res = ctx.decode_frames(data, descs, out_elems=out_elems)
    return descs, out, res


def assert_batch_equals_oracle(ctx, b, check_expected=True):
    descs, out, res = gpu_decode(ctx, b.data, b.frame_offsets[:-1], b.frame_lengths)
    bad, st, ref = O.decode_batch(b.data, b.frame_offsets[:-1], b.frame_lengths, descs["out_offset"],
                                  out.size, n_threads=8)
    assert np.array_equal(res["status"], st)
    assert np.array_equal(res["consumed"][st == 0], b.frame_lengths[st == 0])
    for i in range(b.n_frames):
        o, n = int(descs[i]["out_offset"]), int(descs[i]["n_channels"]) * int(descs[i]["block_size"])
        assert np.array_equal(out[o:o + n], ref[o:o + n]), f"frame {i} differs from the oracle"
        if check_expected:
            lo, hi = int(b.pcm_offsets[i]), int(b.pcm_offsets[i + 1])
            assert np.array_equal(out[o:o + n], b.pcm[lo:hi]), f"frame {i} differs from the generator's PCM"


# --------------------------------------------------------------------------- golden fixtures

@pytest.mark.parametrize("name", ["pop", "short", "wasted_bits", "non_subset", "empty_vorbis_comment",
                                  "repeated_vorbis_comment"])
def test_golden_streams_through_flac_reader(ctx, golden, name):
    """C1 of BASELINE.json: decode testsamples/*.flac via FlacReader -> FrameReader (device path)."""
    data = golden[f"{name}__bytes"]
    reader = cb.FlacReader.new(data, ctx)
    rows = golden[f"{name}__frames"]
    exp = golden[f"{name}__pcm"]
    si = reader.streaminfo()
    frames = reader.blocks()
    pos, buffer, inter = 0, None, []
    for r in rows:
        if r[1] != 0:
            break
        block = frames.read_next_or_eof(buffer)
        assert block is not None
        n = int(r[4] * r[5])
        assert block.duration() == r[4] and block.channels() == r[5] and block.time() == r[7]
        assert np.array_equal(block.into_buffer(), exp[pos:pos + n])
        inter.append(block.into_buffer().reshape(int(r[5]), int(r[4])).T.copy())
        pos += n
        buffer = block.into_buffer()  # recycle, as claxon users do
    assert frames.read_next_or_eof(buffer) is None  # Ok(None) at the end
    if name in KAT["fixture_md5"]:
        nb = (si.bits_per_sample + 7) // 8
        raw = np.concatenate(inter).astype("<i4").view(np.uint8).reshape(-1, 4)[:, :nb].tobytes()
        assert hashlib.md5(raw).hexdigest() == KAT["fixture_md5"][name] == si.md5sum.hex()


def test_golden_samples_iterator(ctx, golden):
    # reference doc-test (src/lib.rs:15-64): iterate samples of pop.flac
    r = cb.FlacReader.new(golden["pop__bytes"], ctx)
    got = list(r.samples())
    assert got == golden["pop__pcm"].tolist()  # mono: interleaved == planar


def test_fuzz_corpus_error_parity(golden):
    """Every fuzz regression stream yields the status the oracle derived, with and without CRC checks."""
    for verify in (True, False):
        c = cb.Context(device=0, verify_crc=verify)
        for name in golden["names"]:
            name = str(name)
            meta, rows = golden[f"{name}__meta"], golden[f"{name}__frames"]
            if not name.startswith("fuzz__") or meta[0] != 0:
                continue
            fr = cb.FrameReader(golden[f"{name}__bytes"][int(meta[1]):], c)
            exp = int(rows[0, 1] if verify else rows[0, 2])
            if exp == 0:
                blk = fr.read_next_or_eof()
                assert np.array_equal(blk.into_buffer(), golden[f"{name}__pcm"][: blk.len()])
            else:
                with pytest.raises(cb.Error) as e:
                    fr.read_next_or_eof()
                assert e.value.status == exp, (name, verify, e.value.status, exp)
        c.close()


def test_all_overwritten_13_vs_17(ctx, golden):
    """tests/testsamples.rs:498-540 / fuzz/fuzzers/diff.rs: output must not depend on buffer contents."""
    for name in golden["names"]:
        name = str(name)
        meta = golden[f"{name}__meta"]
        if meta[0] != 0:
            continue
        data = golden[f"{name}__bytes"][int(meta[1]):]
        outs = []
        for fill in (13, 17):
            fr = cb.FrameReader(data, ctx)
            buf = np.full(8 * 65535, fill, dtype=np.int32)
            try:
                blk = fr.read_next_or_eof(buf)
                outs.append(None if blk is None else blk.into_buffer().copy())
            except cb.Error as e:
                outs.append(e.status)
        if isinstance(outs[0], np.ndarray):
            assert np.array_equal(outs[0], outs[1])
        else:
            assert outs[0] == outs[1]


# --------------------------------------------------------------------------- synthetic vs oracle

SYNTH_CASES = {
    "c2-ms": synth.workload_config("c2", 96),
    "c2-indep": synth.workload_config("c2-indep", 64),
    "c3": synth.workload_config("c3", 96),
    "c4-files": synth.workload_config("c4", 132),
    "c5-order32-8ch": synth.workload_config("c5", 6),
    "all-types-wasted-rice2": synth.SynthConfig(n_frames=256, block_size=1152, n_channels=2, bps=16, stereo_mode=-1,
        type_mask=15, lpc_min_order=1, lpc_max_order=32, qlp_precision=0, rice_mode=-2, rice_kmin=0, rice_kmax=14,
        max_porder=6, rice2=2, wasted_max=5, long_unary_per_mille=100),
    "ragged-3ch-24bit": synth.SynthConfig(n_frames=77, block_size=1000, tail_block_size=37, n_channels=3, bps=24,
        stereo_mode=0, type_mask=15, lpc_min_order=1, lpc_max_order=12, qlp_precision=0, rice_mode=-1, max_porder=3,
        wasted_max=3),
    "tiny-blocks-8bit": synth.SynthConfig(n_frames=50, block_size=16, tail_block_size=5, n_channels=2, bps=8,
        stereo_mode=-1, type_mask=15, lpc_min_order=1, lpc_max_order=16, qlp_precision=0, rice_mode=-1, max_porder=2,
        force_bs16=1),
    "mono-20bit-k0": synth.SynthConfig(n_frames=40, block_size=4608, n_channels=1, bps=20, type_mask=12,
        lpc_min_order=1, lpc_max_order=12, qlp_precision=14, rice_mode=0, residual_mean=0.4, max_porder=8),
    "8ch-12bit-fixed": synth.SynthConfig(n_frames=33, block_size=576, n_channels=8, bps=12, type_mask=4,
        rice_mode=-1, max_porder=4),
    "max-blocksize": synth.SynthConfig(n_frames=3, block_size=65535, n_channels=2, bps=16, stereo_mode=10,
        type_mask=8, lpc_min_order=12, lpc_max_order=12, rice_mode=-1, rice_kmax=14),
    "rice2-big-k": synth.SynthConfig(n_frames=20, block_size=2048, n_channels=2, bps=24, stereo_mode=9, type_mask=8,
        lpc_min_order=2, lpc_max_order=20, qlp_precision=15, rice_mode=-2, rice_kmin=15, rice_kmax=22, rice2=1,
        max_porder=3),
    "variable-blocking": synth.SynthConfig(n_frames=30, block_size=1024, n_channels=2, bps=16, stereo_mode=8,
        type_mask=12, lpc_min_order=1, lpc_max_order=8, variable_blocking=1, rice_mode=-1, max_porder=2),
}


@pytest.mark.parametrize("case", sorted(SYNTH_CASES))
def test_synthetic_vs_oracle(ctx, case):
    assert_batch_equals_oracle(ctx, synth.generate(SYNTH_CASES[case]))


@pytest.mark.parametrize("seed", range(6))
def test_random_configs_vs_oracle(ctx, seed):
    rng = np.random.default_rng(1000 + seed)
    nch = int(rng.integers(1, 9))
    cfg = synth.SynthConfig(
        seed=int(rng.integers(1, 2**31)), n_frames=int(rng.integers(1, 200)),
        block_size=int(rng.choice([16, 192, 576, 1000, 1152, 2304, 4096, 4608, int(rng.integers(1, 9000))])),
        n_channels=nch, bps=int(rng.choice([8, 12, 16, 20, 24])), stereo_mode=-1 if nch == 2 else 0,
        type_mask=int(rng.integers(1, 16)), lpc_min_order=1, lpc_max_order=int(rng.integers(1, 33)),
        qlp_precision=0, rice_mode=int(rng.choice([-1, -2])), rice_kmin=0, rice_kmax=14,
        max_porder=int(rng.integers(0, 8)), rice2=int(rng.integers(0, 3)), wasted_max=int(rng.integers(0, 6)),
        long_unary_per_mille=int(rng.choice([0, 50])))
    assert_batch_equals_oracle(ctx, synth.generate(cfg))


def test_corrupted_frames_status_parity(ctx):
    """Bit flips and truncations: status (and PCM / consumed when it still decodes) must match the oracle,
    with CRC checks on and off (the latter is the reference's cfg(fuzzing) build)."""
    base = synth.generate(synth.SynthConfig(n_frames=40, block_size=576, n_channels=2, bps=16, stereo_mode=-1,
                                           type_mask=15, lpc_min_order=1, lpc_max_order=32, qlp_precision=0,
                                           rice_mode=-1, max_porder=4, rice2=2, wasted_max=4))
    rng = np.random.default_rng(42)
    frames = []
    for trial in range(600):
        i = int(rng.integers(0, base.n_frames))
        f = base.data[int(base.frame_offsets[i]):int(base.frame_offsets[i + 1])].copy()
        kind = trial % 3
        if kind == 0:   # flip a few bits early in the subframe area (headers / params / partition headers)
            for _ in range(int(rng.integers(1, 4))):
                p = int(rng.integers(5, min(f.size, 60)))
                f[p] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:  # flip bits anywhere
            for _ in range(int(rng.integers(1, 3))):
                f[int(rng.integers(5, f.size))] ^= 1 << int(rng.integers(0, 8))
        else:           # truncate
            f = f[: int(rng.integers(6, f.size))]
        st, d = cb.parse_frame_header(f)
        if st != 0:
            continue  # header-level damage is host-side (test_host.py)
        frames.append(f)
    data = np.concatenate(frames)
    lengths = np.array([f.size for f in frames], dtype=np.uint32)
    offsets = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.uint64)
    seen = set()
    for verify in (False, True):
        c = cb.Context(device=0, verify_crc=verify)
        descs, out_elems = cb.descs_from_offsets(data, offsets, lengths, flags=0 if verify else 1)
        out, res = c.decode_frames(data, descs, out_elems=out_elems)
        bad, st, ref = O.decode_batch(data, offsets, lengths, descs["out_offset"], out_elems, n_threads=8,
                                      verify_crc=verify)
        assert np.array_equal(res["status"], st), np.nonzero(res["status"] != st)[0][:10]
        for i in np.nonzero(st == 0)[0]:
            o, n = int(descs[i]["out_offset"]), int(descs[i]["n_channels"]) * int(descs[i]["block_size"])
            assert np.array_equal(out[o:o + n], ref[o:o + n])
        seen |= set(st.tolist())
        c.close()
    # the corruption corpus really exercises the error catalogue
    assert {2, 23}.issubset(seen) and len(seen) >= 8, sorted(seen)


def test_wrapping_arithmetic_parity(ctx):
    """Streams whose samples overflow i32 decode to *defined* wrapped values (all wrapping_* in the
    reference); build them by coding huge residuals with Rice2 and compare with the oracle."""
    cfg = synth.SynthConfig(n_frames=24, block_size=512, n_channels=2, bps=24, stereo_mode=-1, type_mask=12,
                            lpc_min_order=1, lpc_max_order=12, qlp_precision=15, rice_mode=-2, rice_kmin=26,
                            rice_kmax=29, rice2=1, residual_mean=3.0e8, max_porder=2)
    b = synth.generate(cfg)
    assert np.abs(b.pcm.astype(np.int64)).max() > 2**30  # really in wrap territory
    assert_batch_equals_oracle(ctx, b)


def test_narrow_accumulator_shortcut_is_verified(ctx):
    """Small coefficients pick the fast path's i32 accumulator; huge (wrapping) samples then violate its
    exactness condition, which the kernel must notice and hand the frame to the exact path."""
    cfg = synth.SynthConfig(n_frames=16, block_size=1024, n_channels=2, bps=16, stereo_mode=0, type_mask=8,
                            lpc_min_order=1, lpc_max_order=8, qlp_precision=5, rice_mode=-2, rice_kmin=26,
                            rice_kmax=29, rice2=1, residual_mean=2.0e8, max_porder=1)
    b = synth.generate(cfg)
    assert np.abs(b.pcm.astype(np.int64)).max() > 2**29
    assert_batch_equals_oracle(ctx, b)


def test_failed_frame_does_not_poison_batch(ctx):
    b = synth.workload("c2", 48)
    data = b.data.copy()
    victims = [5, 17, 40]
    for v in victims:
        st, hd = cb.parse_frame_header(data, int(b.frame_offsets[v]))
        data[int(b.frame_offsets[v]) + hd.header_len] ^= 0x80  # subframe pad bit -> "invalid subframe header"
    descs, out, res = gpu_decode(ctx, data, b.frame_offsets[:-1], b.frame_lengths)
    for i in range(b.n_frames):
        o, n = int(descs[i]["out_offset"]), 8192
        if i in victims:
            assert res["status"][i] == 11
        else:
            assert res["status"][i] == 0
            assert np.array_equal(out[o:o + n], b.pcm[int(b.pcm_offsets[i]):int(b.pcm_offsets[i + 1])])


def test_unaligned_offsets_and_unknown_lengths(ctx):
    """Frames at arbitrary byte offsets; byte_len given as 'rest of the stream' (boundary unknown)."""
    b = synth.workload("c3", 20)
    pad = 3
    data = np.concatenate([np.full(pad, 0xAB, np.uint8), b.data])
    offs = b.frame_offsets[:-1] + np.uint64(pad)
    lens = (np.uint64(data.size) - offs).astype(np.uint32)
    descs, out, res = gpu_decode(ctx, data, offs, lens)
    assert (res["status"] == 0).all()
    assert np.array_equal(res["consumed"], b.frame_lengths)
    for i in range(b.n_frames):
        o = int(descs[i]["out_offset"]); lo, hi = int(b.pcm_offsets[i]), int(b.pcm_offsets[i + 1])
        assert np.array_equal(out[o:o + hi - lo], b.pcm[lo:hi])


def test_frame_reader_batch_extension(ctx):
    b = synth.workload("c4", 33)
    file_bytes = synth.make_file(b, 0, 33, padding=100)
    r = cb.FlacReader.new(file_bytes, ctx)
    si = r.streaminfo()
    assert si.channels == 2 and si.bits_per_sample == 16 and si.samples == b.n_samples // 2
    blocks = r.blocks().read_batch(1000)
    assert len(blocks) == 33
    md5 = hashlib.md5()
    for i, blk in enumerate(blocks):
        lo, hi = int(b.pcm_offsets[i]), int(b.pcm_offsets[i + 1])
        assert np.array_equal(blk.into_buffer(), b.pcm[lo:hi])
        md5.update(synth.interleaved_le_bytes(blk.into_buffer(), 2, 16))
    assert md5.digest() == si.md5sum  # the synthetic corpus is self-verifying
    assert r.blocks().read_batch(10) == []


def test_frame_reader_sequential_equals_batch(ctx):
    b = synth.workload("c3", 9)
    fr = cb.FrameReader(b.data, ctx)
    buf = None
    for i in range(9):
        blk = fr.read_next_or_eof(buf)
        lo, hi = int(b.pcm_offsets[i]), int(b.pcm_offsets[i + 1])
        assert np.array_equal(blk.into_buffer(), b.pcm[lo:hi]) and blk.time() == 4096 * i
        buf = blk.into_buffer()
    assert fr.read_next_or_eof(buf) is None
    # one byte left: still Ok(None) (src/frame.rs:140-143); garbage: sync error
    assert cb.FrameReader(b.data[:1].copy(), ctx).read_next_or_eof() is None
    with pytest.raises(cb.Error) as e:
        cb.FrameReader(np.array([1, 2, 3, 4], np.uint8), ctx).read_next_or_eof()
    assert e.value == cb.Error(3)


# --------------------------------------------------------------------------- full-size properties

def test_c2_full_size_bit_exact_and_resident_batch(ctx):
    """BASELINE configs[1] at full size: every sample equals the generator's by-construction PCM and the
    oracle; the device-resident path (the one bench.py times) gives the same bits as the host path."""
    b = synth.workload("c2")
    descs, out_elems = cb.descs_from_offsets(b.data, b.frame_offsets[:-1], b.frame_lengths)
    out, res = ctx.decode_frames(b.data, descs, out_elems=out_elems)
    assert (res["status"] == 0).all() and np.array_equal(res["consumed"], b.frame_lengths)
    assert out_elems == b.n_samples and np.array_equal(out[:b.n_samples], b.pcm)
    bad, st, ref = O.decode_batch(b.data, b.frame_offsets[:-1], b.frame_lengths, descs["out_offset"], out_elems,
                                  n_threads=8)
    assert bad == 0 and np.array_equal(ref, out[:out_elems])
    dev = ctx.upload(b.data, descs, out_elems)
    for s in range(3):
        dev.decode(s)
    out2, res2 = dev.read()
    assert np.array_equal(out2[:out_elems], out[:out_elems]) and (res2["status"] == 0).all()
    assert dev.kernel_ms() > 0
    dev.close()


def test_c3_and_c5_large_by_checksum(ctx):
    """Larger slices of C3 / C5 checked through a checksum of checksums against the generator."""
    for name, n in (("c3", 1024), ("c5", 48)):
        b = synth.workload(name, n)
        descs, out_elems = cb.descs_from_offsets(b.data, b.frame_offsets[:-1], b.frame_lengths)
        out, res = ctx.decode_frames(b.data, descs, out_elems=out_elems)
        assert (res["status"] == 0).all()
        assert hashlib.sha1(out[:b.n_samples].tobytes()).digest() == hashlib.sha1(b.pcm.tobytes()).digest()


# --------------------------------------------------------------------------- output stage (interleave + narrow)

def _interleaved_expected(b, descs, out_elems, mode):
    """Oracle PCM (planar) re-laid out on the host the way FlacSamples yields it (src/lib.rs:473-519)."""
    bad, st, ref = O.decode_batch(b.data, b.frame_offsets[:-1], b.frame_lengths, descs["out_offset"], out_elems, n_threads=8)
    assert bad == 0
    exp = np.zeros(out_elems, dtype=np.int32)
    for i in range(b.n_frames):
        o, nch, bs = int(descs[i]["out_offset"]), int(descs[i]["n_channels"]), int(descs[i]["block_size"])
        exp[o:o + nch * bs] = ref[o:o + nch * bs].reshape(nch, bs).T.reshape(-1)
    return exp


@pytest.mark.parametrize("case", ["c2-ms", "c4-files", "ragged-3ch-24bit", "tiny-blocks-8bit", "8ch-12bit-fixed", "mono-20bit-k0"])
def test_interleaved_output_modes_vs_oracle(ctx, case):
    """SURVEY.md §8 f2: the device-side interleave + narrow stage against the oracle's PCM, every element size."""
    b = synth.generate(SYNTH_CASES[case])
    descs, out_elems = cb.descs_from_offsets(b.data, b.frame_offsets[:-1], b.frame_lengths)
    bps = int(descs["bits_per_sample"].max())
    exp = _interleaved_expected(b, descs, out_elems, None)
    live = np.zeros(out_elems, dtype=bool)
    for d in descs:
        live[int(d["out_offset"]):int(d["out_offset"]) + int(d["n_channels"]) * int(d["block_size"])] = True
    out32, res = ctx.decode_frames(b.data, descs, out_elems=out_elems, mode=cb.OUT_INTERLEAVED_I32)
    assert (res["status"] == 0).all() and np.array_equal(out32[:out_elems][live], exp[live])
    if bps <= 24:
        out24, res = ctx.decode_frames(b.data, descs, out_elems=out_elems, mode=cb.OUT_INTERLEAVED_I24)
        got = out24[:3 * out_elems].reshape(-1, 3).astype(np.int32)
        val = got[:, 0] | (got[:, 1] << 8) | (got[:, 2] << 16)
        val = (val ^ 0x800000) - 0x800000  # sign-extend 24 bits
        assert (res["status"] == 0).all() and np.array_equal(val[live], exp[live])
    if bps <= 16:
        out16, res = ctx.decode_frames(b.data, descs, out_elems=out_elems, mode=cb.OUT_INTERLEAVED_I16)
        assert out16.dtype == np.int16 and (res["status"] == 0).all()
        # (the c4 generator's forced Rice parameters push some "16-bit" samples out of range: truncated like `as i16`)
        assert np.array_equal(out16[:out_elems][live], exp[live].astype(np.int16))
    else:
        with pytest.raises(cb.Error) as e:  # 20/24-bit samples do not fit 16 bits: refused, not truncated
            ctx.decode_frames(b.data, descs, out_elems=out_elems, mode=cb.OUT_INTERLEAVED_I16)
        assert e.value.status == 90


def test_interleaved_output_md5_of_reference_fixtures(ctx, golden):
    """The STREAMINFO MD5 (libFLAC's encoder-side digest, src/metadata.rs:52-53) is defined over exactly what the
    interleaved little-endian modes deliver: hash the device's bytes as they come."""
    for name in ("pop", "short", "wasted_bits"):
        data = golden[f"{name}__bytes"]
        si, first = cb.open_stream(data)
        descs, nxt, total, stop = cb.demux_frames(data, first)
        assert stop == 1 and si.bits_per_sample == 16
        out, res = ctx.decode_frames(data, descs, out_elems=total, mode=cb.OUT_INTERLEAVED_I16)
        assert (res["status"] == 0).all()
        md5 = hashlib.md5()
        for d in descs:
            o, n = int(d["out_offset"]), int(d["n_channels"]) * int(d["block_size"])
            md5.update(out[o:o + n].astype("<i2").tobytes())
        assert md5.digest() == si.md5sum, name
    # a synthetic stereo file carries the digest of its by-construction PCM
    b = synth.workload("c4", 22)
    file_bytes = np.frombuffer(synth.make_file(b, 0, 22), dtype=np.uint8)
    si, first = cb.open_stream(file_bytes)
    descs, nxt, total, stop = cb.demux_frames(file_bytes, first)
    out, res = ctx.decode_frames(file_bytes, descs, out_elems=total, mode=cb.OUT_INTERLEAVED_I16)
    md5 = hashlib.md5()
    for d in descs:
        o, n = int(d["out_offset"]), int(d["n_channels"]) * int(d["block_size"])
        md5.update(out[o:o + n].astype("<i2").tobytes())
    assert (res["status"] == 0).all() and md5.digest() == si.md5sum


# --------------------------------------------------------------------------- BASELINE.json's configurations at full size

@pytest.mark.parametrize("name,frames", [("c3", 8192), ("c4", 11000), ("c5", 512)])
def test_full_size_configs_vs_oracle(name, frames):
    """configs[2..4] at (per-GPU) full size through the device-resident throughput path, against the ORACLE's PCM
    (and the generator's by-construction PCM): c3 = the whole 8192-frame batch; c4 = 1000 files with forced Rice
    parameters 0..14 (the largest of them code 16-bit audio with residuals beyond 16 bits); c5 = one GPU's eighth
    of the 4096-frame stress batch (8 channels, LPC order 32, block size 16384)."""
    c = cb.Context(device=0, lane_per_frame=True)
    b = synth.workload(name, frames)
    descs, out_elems = cb.descs_from_offsets(b.data, b.frame_offsets[:-1], b.frame_lengths)
    assert out_elems == b.n_samples
    bad, st, ref = O.decode_batch(b.data, b.frame_offsets[:-1], b.frame_lengths, descs["out_offset"], out_elems,
                                  n_threads=min(64, os.cpu_count() or 8))
    assert bad == 0 and hashlib.sha1(ref.tobytes()).digest() == hashlib.sha1(b.pcm.tobytes()).digest()
    dev = c.upload(b.data, descs, out_elems)
    dev.decode(0)
    out, res = dev.read()
    dev.close()
    c.close()
    assert (res["status"] == 0).all() and np.array_equal(res["consumed"], b.frame_lengths)
    if not np.array_equal(out[:out_elems], ref):
        badf = [i for i in range(b.n_frames) if not np.array_equal(
            out[int(descs[i]["out_offset"]):int(descs[i]["out_offset"]) + int(descs[i]["n_channels"]) * int(descs[i]["block_size"])],
            ref[int(descs[i]["out_offset"]):int(descs[i]["out_offset"]) + int(descs[i]["n_channels"]) * int(descs[i]["block_size"])])]
        raise AssertionError(f"{name}: {len(badf)} frames differ from the oracle, first {badf[:5]}")


def test_resident_batch_reports_crc_mismatch():
    """The device-resident path verifies the frame CRC-16 too (src/frame.rs:752-763): a flipped residual bit comes
    back as "frame CRC mismatch", not as CLX_OK with wrong PCM."""
    c = cb.Context(device=0)
    b = synth.workload("c2", 64)
    data = b.data.copy()
    victims = [3, 40]
    for v in victims:
        data[int(b.frame_offsets[v]) + int(b.frame_lengths[v]) // 2] ^= 0x10
    descs, out_elems = cb.descs_from_offsets(data, b.frame_offsets[:-1], b.frame_lengths)
    dev = c.upload(data, descs, out_elems)
    dev.decode(0)
    out, res = dev.read()
    bad, st, ref = O.decode_batch(data, b.frame_offsets[:-1], b.frame_lengths, descs["out_offset"], out_elems, n_threads=4)
    assert np.array_equal(res["status"], st) and set(np.nonzero(st)[0].tolist()) == set(victims)
    dev.close()
    c.close()


@pytest.mark.parametrize("workload,frames,sampled", [("c2", 64, False), ("c5", 256, True)])
def test_bench_dump_outputs_are_the_last_timed_step(tmp_path, workload, frames, sampled):
    """bench.py --dump-outputs: 4 timed steps over 2 units end on unit 1, whose PCM and per-frame results are written
    bit for bit as the generator made them, within 64 MB in all (a c5 unit's 134 MB of samples: a seeded selection
    of whole frames)."""
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--inflight", "2", "--streams", "2",
           "--steps", "4", "--warmup", "1", "--e2e-steps", "1", "--cpu-seconds", "0", "--no-extra",
           "--frames", str(frames), "--dump-outputs", str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 4 and line["timed_steps"] == 4 and line["bit_exact"]
    cfg = synth.workload_config(workload, frames)
    cfg.seed += 1000003  # unit 1 (bench.unit_config)
    b = synth.generate(cfg)
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 * 10**6
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("pcm", "pcm_frames", "status", "consumed")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert (got["status"] == 0).all() and np.array_equal(got["consumed"], b.frame_lengths)
    sel = got["pcm_frames"].astype(np.int64)
    assert 0 < sel.size <= b.n_frames and sampled == (sel.size < b.n_frames)
    exp = np.concatenate([b.pcm[int(b.pcm_offsets[i]):int(b.pcm_offsets[i + 1])] for i in sel])
    assert np.array_equal(got["pcm"].astype(np.int64), exp)


def test_constant_frames_through_read_batch(ctx):
    """Digital silence: 14-byte frames that decode to 8192 samples each (ADVICE r1: the batched reader used to size
    its buffer from the remaining BYTES and failed on such streams)."""
    cfg = synth.SynthConfig(n_frames=40, block_size=4096, n_channels=2, bps=16, stereo_mode=0, type_mask=1)
    b = synth.generate(cfg)
    assert b.data.size < 40 * 64
    fr = cb.FrameReader(b.data, ctx)
    blocks = fr.read_batch(1000)
    assert len(blocks) == 40
    for i, blk in enumerate(blocks):
        lo, hi = int(b.pcm_offsets[i]), int(b.pcm_offsets[i + 1])
        assert np.array_equal(blk.into_buffer(), b.pcm[lo:hi])
    assert fr.read_batch(10) == []


def test_tightly_packed_odd_blocks_many_chunks(ctx):
    """ADVICE r1: >= 256 frames (several chunks on several streams) whose out_offsets are NOT multiples of 4 and
    leave no gap: neighbouring chunks must not touch each other's samples."""
    cfg = synth.SynthConfig(n_frames=700, block_size=333, n_channels=1, bps=16, type_mask=12, lpc_min_order=1,
                            lpc_max_order=8, rice_mode=-1, max_porder=0)
    b = synth.generate(cfg)
    descs, _ = cb.descs_from_offsets(b.data, b.frame_offsets[:-1], b.frame_lengths)
    descs["out_offset"] = np.arange(b.n_frames, dtype=np.uint64) * 333 + 1  # packed, odd
    out = np.full(b.n_frames * 333 + 2, 77, dtype=np.int32)
    out, res = ctx.decode_frames(b.data, descs, out=out)
    assert (res["status"] == 0).all() and out[0] == 77 and out[-1] == 77
    assert np.array_equal(out[1:-1], b.pcm)


def test_batch_from_device_bytes_checks_crc_on_device():
    """clx_batch_create_ex(CLX_BATCH_BYTES_ON_DEVICE): the shard a rank received over NVLink never visits the host; its
    frame CRC-16 is verified by the device kernel — statuses (incl. "frame CRC mismatch") as the oracle's."""
    import torch
    c = cb.Context(device=0)
    b = synth.workload("c3", 200)
    data = b.data.copy()
    victims = [7, 150]
    for v in victims:
        data[int(b.frame_offsets[v]) + int(b.frame_lengths[v]) // 3] ^= 0x04
    descs, out_elems = cb.descs_from_offsets(data, b.frame_offsets[:-1], b.frame_lengths)
    t = torch.from_numpy(data).cuda()
    dev = c.adopt(t.data_ptr(), t.numel(), descs, out_elems)
    dev.decode(0)
    out, res = dev.read()
    bad, st, ref = O.decode_batch(data, b.frame_offsets[:-1], b.frame_lengths, descs["out_offset"], out_elems, n_threads=8)
    assert np.array_equal(res["status"], st) and set(np.nonzero(st)[0].tolist()) == set(victims)
    for i in np.nonzero(st == 0)[0]:
        o, n = int(descs[i]["out_offset"]), int(descs[i]["n_channels"]) * int(descs[i]["block_size"])
        assert np.array_equal(out[o:o + n], ref[o:o + n])
    dev.close()
    c.close()
