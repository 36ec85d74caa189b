"""Generates tests/golden/fixtures.npz from the reference's own test streams.

Run with the test streams of a claxon checkout:

    python tests/golden/make_golden.py <claxon checkout>/testsamples

For every stream in that directory (incl. the fuzz corpus) it stores the raw
bytes, the status the oracle reports at open / first failing frame, and — for streams that
decode — the oracle's planar PCM per frame, which is pinned independently by the STREAMINFO MD5
(libFLAC's encoder-side digest) wherever the file carries one.  The npz is what the `-m gpu`
parity tests compare the CUDA path against.
"""
import glob
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402


def main(ref):
    out = {}
    names = []
    files = sorted(glob.glob(os.path.join(ref, "*.flac"))) + sorted(glob.glob(os.path.join(ref, "fuzz", "*.flac")))
    for path in files:
        rel = os.path.relpath(path, ref)
        key = rel.replace("/", "__").replace(".flac", "")
        data = np.fromfile(path, dtype=np.uint8)
        names.append(key)
        out[f"{key}__bytes"] = data
        st, si, first = O.open_stream(data)
        meta = [st, first, si.channels, si.bits_per_sample, si.samples]
        out[f"{key}__md5"] = np.frombuffer(bytes(si.md5sum), dtype=np.uint8)
        # frames, crc verified (normal build) and unverified (cfg(fuzzing)) statuses
        frame_rows, pcm = [], []
        if st == 0:
            at = first
            while True:
                f = O.decode_frame(data, at)
                fz = O.decode_frame(data, at, verify_crc=False)
                h = f.info.header
                frame_rows.append([at, f.status, fz.status, f.info.consumed, h.block_size, h.n_channels,
                                   h.bits_per_sample, f.info.time])
                if f.status != 0:
                    if fz.status == 0:
                        pcm.append(fz.samples.copy())  # what decodes when CRCs are ignored
                    break
                pcm.append(f.samples.copy())
                at += f.info.consumed
        out[f"{key}__meta"] = np.array(meta, dtype=np.int64)
        out[f"{key}__frames"] = np.array(frame_rows, dtype=np.int64).reshape(-1, 8)
        out[f"{key}__pcm"] = np.concatenate(pcm) if pcm else np.zeros(0, dtype=np.int32)
        # cross-check against the file's own MD5 when it has one
        good = [r for r in frame_rows if r[1] == 0]
        if st == 0 and any(si.md5sum) and len(good) == len(frame_rows) - 1 and frame_rows[-1][1] == 1:
            inter = []
            pos = 0
            for r in good:
                n = r[4] * r[5]
                inter.append(out[f"{key}__pcm"][pos:pos + n].reshape(r[5], r[4]).T)
                pos += n
            nb = (si.bits_per_sample + 7) // 8
            raw = np.concatenate(inter).astype("<i4").view(np.uint8).reshape(-1, 4)[:, :nb].tobytes()
            assert hashlib.md5(raw).digest() == bytes(si.md5sum), f"{rel}: oracle PCM does not match STREAMINFO MD5"
            print(f"{rel}: MD5 ok ({len(good)} frames)")
        else:
            print(f"{rel}: open={st} frames={[(r[1], r[2]) for r in frame_rows]}")
    out["names"] = np.array(names)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "fixtures.npz"), **out)
    print("wrote fixtures.npz with", len(names), "streams")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_golden.py <claxon checkout>/testsamples")
    main(sys.argv[1])
