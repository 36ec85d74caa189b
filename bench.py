#!/usr/bin/env python
"""bench.py — headline benchmark of claxon_b200 (contract: see the task prompt / DESIGN.md §6).

Metric (BASELINE.json): Msamples/s decoded, bit-exact, samples = sum(block_size * channels).
Workload at N=1: BASELINE.json configs[1] ("c2"): batch of 1024 synthetic stereo 16-bit frames,
block size 4096, LPC order 8, Rice parameter 4, mid/side.  One *step* = one pass of the hot path
(`FrameReader::read_next_or_eof` for every frame of the batch) over one such batch ("unit").

  value  — kernel-only throughput, inputs resident in HBM.  The job is a list of units (128 distinct
           batches per GPU: combined footprint 5 GB > L2, so no step finds its inputs or outputs in L2; 64 in
           flight measured 528, 128 in flight 553 Gsamples/s on the same box); the list is
           partitioned over the ranks by `claxon_b200.shard.plan_shards` (contiguous ranges balanced on
           algorithmic bytes, no data-path collective: frames are independent, reference
           src/frame.rs:603-605) and every rank cycles its units over `--streams` CUDA streams, i.e.
           many batches in flight: the steady-state regime of a decode service.  `--scaling weak`
           (default): `--inflight` units per rank; `--scaling strong`: a fixed corpus of `--units`
           units split over the ranks.  A lone 1024-frame batch is latency-bound by the serial LPC
           recurrence (SURVEY.md §7.3-3) and the sequential Rice walk; its figure is reported next to
           it as `single_batch`.  The timed region is `--steps K` steps issued back to back (no drain in
           between; `--scaling strong`: K steps of the whole corpus, each rank running those of its own
           units); ms_per_step = region / K.  A step takes ~15 us, so K of a few thousand is needed for a
           window of tens of milliseconds.  Every batch's CUDA graph is instantiated when the batch is
           created, and `--warmup W` untimed steps precede the region, never fewer than one per unit.
           `--dump-outputs DIR` then writes what the last timed step computed (`dump_outputs`).
  e2e    — same metric through the public host-buffer call (`clx_decode_frames`): per step the
           compressed frames go pinned-host -> device and the full planar i32 PCM comes back.  The call
           is synchronous; `--e2e-callers` host threads (default 2, each with its own context and pinned
           buffers, as the worker threads of a decode service) call it concurrently, so that one call's
           copy-out overlaps the next one's copy-in and kernels; `e2e.one_caller` is the same with a
           single caller.
           `e2e_i16`: the same call in the interleaved 16-bit output mode (what a WAV writer or the
           STREAMINFO MD5 consumes; half the bytes over PCIe) — a different metric row, reported apart.
  roofline — HBM: algorithmic bytes (frame bytes read once + planar i32 written once) / device
           time, against the measured copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline — the CPU oracle (a C restatement of claxon; kind "port") on all host cores.
  workloads — at N=1, short measurements of BASELINE.json's other configurations (c3, c4, c5) and of C2's
           independent-stereo variant by the same method, bit-exactness checked against the generator's PCM.

`--impl reference` times that CPU port alone, same config/metric (the reference itself is Rust and
cannot be built in this image or on the GPU box: no rustc / cargo on either).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.dont_write_bytecode = True  # the tree may be read-only; the benchmark writes nothing into it

METRIC = "Msamples/s decoded (bit-exact)"
DUMP_LIMIT_BYTES = 64 * 10**6

# frames per unit (one device-resident batch) of each workload, and units of the whole corpus (strong scaling)
UNIT_FRAMES = {"c2": 1024, "c2-indep": 1024, "c3": 8192, "c4": 1100, "c5": 256}
CORPUS_UNITS = {"c2": 128, "c2-indep": 128, "c3": 16, "c4": 128, "c5": 16}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons; `stop(t0, t1)` keeps the samples taken inside the
    timed region [t0, t1] (wall clock), falling back to the nearest ones when the region is shorter than
    the sampling period."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t_end = time.time() + 3.0
            while not self.rows and time.time() < t_end:  # wait for the first sample: nvidia-smi starts slowly
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        parsed = []
        for ts, r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                parsed.append((ts, float(f[1]), float(f[2]), [n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [p for p in parsed if t0 is not None and t0 - 0.02 <= p[0] <= t1 + 0.04]
        note = "inside timed region"
        if not inside and parsed:
            mid = ((t0 or 0) + (t1 or 0)) / 2
            inside = sorted(parsed, key=lambda p: abs(p[0] - mid))[:3]
            note = "timed region shorter than the sampling period: nearest samples"
        sm = [p[1] for p in inside]
        reasons = sorted({n for p in inside for n in p[3]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": inside[0][2] if inside else None,
                "reasons": reasons, "samples": len(sm), "note": note}


def measured_peak_gbs():
    p = os.path.join(HERE, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic():
    """dram bytes per launch of the decode kernels from the committed ncu capture, if any."""
    p = os.path.join(HERE, "profiles", "traffic.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


def cpu_model():
    """Model name of the host CPU (for the cpu_baseline record); never raises."""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def _numa_of(local):
    import torch
    p = torch.cuda.get_device_properties(local)
    with open(f"/sys/bus/pci/devices/{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0/numa_node") as f:
        return int(f.read())


def pin_to_gpu_numa_node(local, world):
    """Keeps this rank's host threads (CRC pool, staging copies) on the NUMA node its GPU hangs off, and
    returns (threads this rank may use, note).  Ranks that share a node split its CPUs between them."""
    total = os.cpu_count() or 1
    try:
        node = _numa_of(local)
        if node < 0:
            raise ValueError("no NUMA node recorded")
        cpus = []
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus += list(range(int(lo), int(hi or lo) + 1))
        peers = [r for r in range(world) if _numa_of(r) == node]
        mine = cpus[peers.index(local)::len(peers)] if local in peers else cpus
        os.sched_setaffinity(0, mine)
        return len(mine), f"pinned to NUMA node {node}: {len(mine)} of its {len(cpus)} CPUs"
    except Exception as e:  # no sysfs entry, no permission ...: split the machine evenly instead
        n = max(1, total // max(1, world))
        return n, f"not pinned ({type(e).__name__}); {n} threads per rank"


def cpu_decode_rate(batch, threads, min_seconds):
    from oracle import oracle as O
    offs, lens, poffs = batch.frame_offsets[:-1], batch.frame_lengths, batch.pcm_offsets[:-1]
    out = np.zeros(batch.n_samples, dtype=np.int32)
    O.decode_batch(batch.data, offs, lens, poffs, batch.n_samples, n_threads=threads, out=out)  # warm
    reps, t0 = 0, time.perf_counter()
    while True:
        bad, _, _ = O.decode_batch(batch.data, offs, lens, poffs, batch.n_samples, n_threads=threads, out=out)
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            break
    assert bad == 0 and np.array_equal(out, batch.pcm), "CPU oracle output differs from expected PCM"
    return batch.n_samples * reps / dt / 1e6, reps, dt


def describe(workload, cfg):
    return (f"{workload}: {cfg.n_frames} frames x {cfg.n_channels}ch x bs{cfg.block_size}, {cfg.bps}-bit, "
            f"LPC order {cfg.lpc_min_order}-{cfg.lpc_max_order}, Rice k={cfg.rice_mode}, stereo_mode={cfg.stereo_mode}")


def unit_config(synth, workload, unit_index, frames=None):
    """Unit `unit_index` of a workload: same shape, its own content (frame i of a unit depends on seed + i only)."""
    cfg = synth.workload_config(workload, frames or UNIT_FRAMES[workload])
    cfg.seed = cfg.seed + 1000003 * unit_index
    return cfg


def dump_outputs(dirpath, batch):
    """Writes what a caller of the device-resident path gets back from `batch` (clx_batch_read) as .npy files, so
    that two builds can be compared output for output:
      pcm.npy        decoded samples, each frame planar as claxon's Block, frames back to back (the alignment
                     padding between frames in the output buffer is left out); float32 when every sample fits
                     its 24-bit significand, float64 otherwise
      pcm_frames.npy the frame index of each frame in pcm.npy, in order
      status.npy, consumed.npy  every frame's result
    When all samples would not fit DUMP_LIMIT_BYTES in all, pcm.npy holds a fixed, seeded selection of whole
    frames."""
    out, res = batch.read()
    d = batch.descs
    offs = d["out_offset"].astype(np.int64)
    lens = d["n_channels"].astype(np.int64) * d["block_size"].astype(np.int64)
    peak = max((int(np.abs(out[o:o + n].astype(np.int64)).max(initial=0)) for o, n in zip(offs, lens)), default=0)
    dtype = np.dtype(np.float32 if peak <= 2**24 else np.float64)
    fixed = 3 * 8 * d.size + 4 * 4096  # the per-frame arrays and the .npy headers
    sel = np.arange(d.size)
    if int(lens.sum()) * dtype.itemsize + fixed > DUMP_LIMIT_BYTES:
        order = np.random.default_rng(0).permutation(d.size)
        sel = np.sort(order[np.cumsum(lens[order]) * dtype.itemsize + fixed <= DUMP_LIMIT_BYTES])
    pcm = np.concatenate([out[offs[i]:offs[i] + lens[i]] for i in sel] or [np.zeros(0, np.int32)])
    os.makedirs(dirpath, exist_ok=True)
    for name, a in (("pcm", pcm.astype(dtype)), ("pcm_frames", sel.astype(np.float64)),
                    ("status", res["status"].astype(np.float64)), ("consumed", res["consumed"].astype(np.float64))):
        np.save(os.path.join(dirpath, name + ".npy"), a)


class Job:
    """This rank's share of a list of units, resident on the device."""

    def __init__(self, cb, synth, ctx, workload, unit_ids, frames=None, keep_host=2):
        self.batches, self.host = [], []
        self.unit_alg, self.unit_samples = [], []
        for j, u in enumerate(unit_ids):
            b = synth.generate(unit_config(synth, workload, u, frames))
            descs, out_elems = cb.descs_from_offsets(b.data, b.frame_offsets[:-1], b.frame_lengths)
            self.batches.append(ctx.upload(b.data, descs, out_elems))
            if j < keep_host:
                self.host.append((b, descs, out_elems))
            self.unit_alg.append(int(b.data.size) + 4 * b.n_samples)
            self.unit_samples.append(b.n_samples)
        self.alg_bytes = sum(self.unit_alg)
        self.n_samples = sum(self.unit_samples)

    def exact(self, idx=0):
        """The timed kernels' output of unit `idx` equals the generator's PCM bit for bit (and every status is OK)."""
        bt = self.batches[idx]
        bt.decode(0)
        out, res = bt.read()
        b, d, out_elems = self.host[idx]
        if not bool((res["status"] == 0).all()):
            return False
        if out_elems == b.n_samples:
            return hashlib.sha1(out[:out_elems].tobytes()).digest() == hashlib.sha1(b.pcm.tobytes()).digest()
        for i in range(b.n_frames):
            o = int(d[i]["out_offset"]); lo, hi = int(b.pcm_offsets[i]), int(b.pcm_offsets[i + 1])
            if not np.array_equal(out[o:o + hi - lo], b.pcm[lo:hi]):
                return False
        return True

    def steady(self, ctx, steps, streams, regions, sync=None, warmup=0):
        """`warmup` untimed steps (every batch once, at least), then `regions` timed regions of `steps` steps each
        (round-robin over this rank's units); device ms each."""
        n = len(self.batches)
        ctx.run_steps(self.batches, max(n, 3, warmup), streams)
        out = []
        for _ in range(max(1, regions)):
            if sync:
                sync()
            out.append(ctx.run_steps(self.batches, steps, streams))
        return out

    def per_steps(self, steps):
        """(samples, algorithmic bytes) that `steps` round-robin steps cover."""
        n = len(self.batches)
        full, rem = divmod(steps, n)
        return (full * self.n_samples + sum(self.unit_samples[:rem]), full * self.alg_bytes + sum(self.unit_alg[:rem]))

    def close(self):
        for b in self.batches:
            b.close()
        self.batches = []


def short_line(cb, synth, ctx, workload, n_units, streams, min_ms=40.0):
    """A short steady-state measurement of another BASELINE.json configuration on this GPU."""
    t0 = time.time()
    job = Job(cb, synth, ctx, workload, list(range(n_units)), keep_host=1)
    exact = job.exact(0)
    one = ctx.run_steps(job.batches, n_units, streams) / n_units  # ms per step, rough
    steps = max(n_units * 2, int(min_ms / max(one, 1e-3)))
    ms = float(np.median(job.steady(ctx, steps, streams, 3)))
    samples, alg = job.per_steps(steps)
    peak, _ = measured_peak_gbs()
    cfg = unit_config(synth, workload, 0)
    line = {"config": describe(workload, cfg), "frames_per_step": UNIT_FRAMES[workload], "units_in_flight": n_units,
            "footprint_mb": round(job.alg_bytes / 1e6), "steps": steps, "ms_per_step": ms / steps,
            "value": samples / (ms / 1e3) / 1e6, "unit": "Msamples/s", "bit_exact": bool(exact),
            "bytes_per_sample": alg / samples, "roofline_frac": alg / (ms / 1e3) / 1e9 / peak}
    job.close()
    line["wall_s"] = round(time.time() - t0, 1)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000, help="steps in the timed region")
    ap.add_argument("--warmup", type=int, default=5, help="untimed steps before it (at least one per unit)")
    ap.add_argument("--impl", default="claxon_b200", choices=["claxon_b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(UNIT_FRAMES))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--frames", type=int, default=None, help="override frames per unit")
    ap.add_argument("--inflight", type=int, default=None, help="weak scaling: units per rank (default: the workload's corpus)")
    ap.add_argument("--units", type=int, default=None, help="strong scaling: units of the whole corpus")
    ap.add_argument("--streams", type=int, default=128)
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--e2e-callers", type=int, default=2)
    ap.add_argument("--cpu-seconds", type=float, default=3.0)
    ap.add_argument("--no-extra", action="store_true", help="skip the short c3 / c4 / c5 lines at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step decoded to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "claxon_b200":
        ap.error("--dump-outputs writes the outputs of the device path (--impl claxon_b200)")

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # more hardware work queues than the default 8, so that the batches in flight really overlap
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "64")
    from claxon_b200 import synth

    cfg = unit_config(synth, args.workload, 0, args.frames)
    config = {"workload": describe(args.workload, cfg), "frames_per_step": cfg.n_frames}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        batch = synth.generate(cfg)
        cores = os.cpu_count() or 1
        from oracle import oracle as O
        offs, lens, poffs = batch.frame_offsets[:-1], batch.frame_lengths, batch.pcm_offsets[:-1]
        out = np.zeros(batch.n_samples, dtype=np.int32)
        for _ in range(max(1, args.warmup)):
            O.decode_batch(batch.data, offs, lens, poffs, batch.n_samples, n_threads=cores, out=out)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            bad, _, _ = O.decode_batch(batch.data, offs, lens, poffs, batch.n_samples, n_threads=cores, out=out)
        dt = time.perf_counter() - t0
        ok = bad == 0 and np.array_equal(out, batch.pcm)
        v = batch.n_samples * args.steps / dt / 1e6
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int32/int64",
            "data": "synthetic", "config": config, "bit_exact": bool(ok),
            "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port", "cpu_model": cpu_model(),
                             "sample": f"{args.steps} x full {args.workload} batch ({batch.n_samples} samples)",
                             "note": "C restatement of claxon v0.4.3 (oracle/), frames sharded over threads; "
                                     "claxon itself is Rust and cannot be built here (no rustc / cargo)"},
            "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------ GPU arm
    import claxon_b200 as cb
    from claxon_b200 import shard

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        # NCCL prints its version banner on STDOUT when a communicator comes up (NCCL_DEBUG=VERSION and above, which
        # some launchers set); this script's stdout is one JSON line, so file descriptor 1 points at stderr until the
        # first collective has run.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
            warm = torch.zeros(1, device=f"cuda:{local}")
            dist_mod.all_reduce(warm)
            dist_mod.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
        dist = dist_mod

    def barrier():
        if dist is not None:
            dist.barrier()

    def reduce_ranks(x, op):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce_ranks(x, dist.ReduceOp.MAX) if dist is not None else x

    def sum_over_ranks(x):
        return reduce_ranks(x, dist.ReduceOp.SUM) if dist is not None else x

    host_threads, pin_note = pin_to_gpu_numa_node(local, world)
    host_threads = max(1, min(32, host_threads))
    ctx = cb.Context(device=local, n_streams=max(2, args.streams), host_threads=host_threads)

    # ---- the job: a list of units, partitioned over the ranks by plan_shards (equal shapes: equal shares)
    if args.scaling == "weak":
        n_units = (args.inflight or CORPUS_UNITS[args.workload]) * world
    else:
        n_units = args.units or CORPUS_UNITS[args.workload]
    unit_descs = np.zeros(n_units, dtype=cb.DESC_DTYPE)  # one pseudo-frame per unit: every unit costs the same
    unit_descs["byte_len"] = 1
    unit_descs["n_channels"] = 1
    unit_descs["block_size"] = 1
    lo, hi = shard.plan_shards(unit_descs, world)[rank]
    job = Job(cb, synth, ctx, args.workload, list(range(lo, hi)), args.frames)
    n_mine = hi - lo
    config.update({"parallelism": f"{n_units} units over {world} GPU(s) by plan_shards, no collective on the data path",
                   "units": n_units, "units_this_rank": n_mine, "streams": args.streams, "host": pin_note,
                   "l2": f"steps cycle over {n_mine} distinct batches per GPU, footprint {job.alg_bytes / 1e6:.0f} MB > 126 MB L2"})

    exact = job.exact(0) if n_mine else True

    # ---- single-batch (latency regime): one batch, serialised steps (reported only)
    single_ms = None
    if n_mine:
        for _ in range(3):
            job.batches[0].decode(0); job.batches[0].sync()
        single = []
        for i in range(10):
            bt = job.batches[(i + 1) % n_mine]
            bt.decode(0); bt.sync()
            single.append(bt.kernel_ms())
        single_ms = float(np.median(single))

    # ---- steady state
    if args.scaling == "weak":
        my_steps = args.steps                  # per rank; the job's steps are world x that
        timed_steps = my_steps * world
    else:  # a step = one unit of the corpus; step i decodes unit i % n_units, on the rank that holds it
        full, rem = divmod(args.steps, n_units)
        my_steps = full * n_mine + max(0, min(hi, rem) - lo)
        timed_steps = args.steps
    warm_steps = max(n_mine, 3, args.warmup)
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ctx.launch_count
    t_wall0 = time.time()
    regions = [max_over_ranks(r) for r in (job.steady(ctx, my_steps, args.streams, 1, barrier, warm_steps) if n_mine
                                            else [0.0])]
    t_wall1 = time.time()
    launches_all = ctx.launch_count - launches0
    barrier()
    clocks = sampler.stop(t_wall0, t_wall1)
    ms = float(np.median(regions))
    my_samples, my_alg = job.per_steps(my_steps) if n_mine else (0, 0)
    gpu_launches = int(round(launches_all * my_steps / (my_steps + warm_steps))) if n_mine else 0
    if args.dump_outputs and rank == 0 and my_steps:
        dump_outputs(args.dump_outputs, job.batches[(my_steps - 1) % n_mine])
    tot_samples, tot_alg = sum_over_ranks(my_samples), sum_over_ranks(my_alg)
    value = tot_samples / (ms / 1e3) / 1e6
    peak, peak_src = measured_peak_gbs()
    achieved = tot_alg / world / (ms / 1e3) / 1e9  # per GPU
    traffic = load_traffic()

    # ---- end to end through the host-buffer call, pinned memory
    e2e = {}
    if n_mine:
        e2e_steps = args.e2e_steps or max(20, min(args.steps, 40))
        hb, hd, hout_elems = job.host[0]
        callers = max(1, args.e2e_callers)
        # one context + pinned buffers per caller (a clx_ctx belongs to one host thread)
        slots = []
        for c in range(callers):
            cx = cb.Context(device=local, n_streams=8, host_threads=max(1, host_threads // callers))
            pb = cx.host_alloc(int(hb.data.size) + 64)
            pb[: hb.data.size] = hb.data
            slots.append((cx, pb, cx.host_alloc(4 * hout_elems + 64), np.zeros(hd.size, dtype=cb.RESULT_DTYPE)))

        def run(mode, n_callers):
            def worker(slot, n):
                cx, pb, po, rs = slot
                for _ in range(n):
                    cx.decode_frames_raw(pb.ctypes.data, hb.data.size, hd.ctypes.data, hd.size, po.ctypes.data, hout_elems,
                                         rs.ctypes.data, mode)
            for slot in slots[:n_callers]:
                worker(slot, 3)
            barrier()
            threads = [threading.Thread(target=worker, args=(slot, e2e_steps)) for slot in slots[:n_callers]]
            t0 = time.perf_counter()
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            dt = time.perf_counter() - t0
            barrier()
            return max_over_ranks(dt), n_callers * e2e_steps

        def check(mode):
            ok = True
            for cx, pb, po, rs in slots:
                ok &= bool((rs["status"] == 0).all())
                view = po[: 4 * hout_elems].view(np.int32) if mode == cb.OUT_PLANAR_I32 else po[: 2 * hout_elems].view(np.int16)
                for i in range(0, hb.n_frames, max(1, hb.n_frames // 64)):
                    o = int(hd[i]["out_offset"]); lo_, hi_ = int(hb.pcm_offsets[i]), int(hb.pcm_offsets[i + 1])
                    exp = hb.pcm[lo_:hi_]
                    if mode != cb.OUT_PLANAR_I32:
                        exp = exp.reshape(int(hd[i]["n_channels"]), -1).T.reshape(-1).astype(np.int16)
                    ok &= bool(np.array_equal(view[o:o + hi_ - lo_], exp))
            return ok

        for mode, key in ((cb.OUT_PLANAR_I32, "e2e"), (cb.OUT_INTERLEAVED_I16, "e2e_i16")):
            if mode == cb.OUT_INTERLEAVED_I16 and cfg.bps > 16:
                continue
            # three timed regions each, the median reported (a region is tens of milliseconds: one slow call shows)
            dt1, n1 = sorted(run(mode, 1) for _ in range(3))[1]
            dt, n = sorted(run(mode, callers) for _ in range(3))[1]
            ok = check(mode)
            d2h = (4 if mode == cb.OUT_PLANAR_I32 else 2) * hout_elems
            e2e[key] = {"value": sum_over_ranks(hb.n_samples) * n / dt / 1e6, "unit": "Msamples/s", "steps": n, "callers": callers,
                        "one_caller": sum_over_ranks(hb.n_samples) * n1 / dt1 / 1e6,
                        "h2d_bytes_per_step": int(hb.data.size + hd.nbytes), "d2h_bytes_per_step": int(d2h + slots[0][3].nbytes),
                        "bit_exact": ok, "output": "planar i32 (Block layout)" if mode == cb.OUT_PLANAR_I32
                        else "interleaved little-endian i16 (a different metric row)"}
            exact = exact and ok

    cpu = None
    extra = None
    demux = None
    if rank == 0 and n_mine:
        # the step before the path (SURVEY §8 f1): frame boundaries of a raw byte stream, found on the host by sync
        # scan + CRC-8 + CRC-16 confirmation (clx_demux_frames), one thread and `host_threads` threads
        hb0 = job.host[0][0]
        stream_bytes = np.concatenate([hb0.data] * 8)  # 8 units back to back: ~50 MB
        rates = {}
        for th in (1, host_threads):
            best = None
            for _ in range(3):
                t0 = time.perf_counter()
                dd, _, _, _ = cb.demux_frames(stream_bytes, threads=th)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            assert dd.size == 8 * hb0.n_frames
            rates[th] = stream_bytes.size / best / 1e9
        demux = {"GBps_one_thread": rates[1], "GBps": rates[host_threads], "threads": host_threads,
                 "Msamples_per_s": rates[host_threads] * 1e9 / (hb0.data.size / hb0.n_samples) / 1e6,
                 "note": "clx_demux_frames_mt on the host: sync scan, header parse + CRC-8, CRC-16 of every byte"}
    if rank == 0 and world == 1:
        if args.cpu_seconds > 0 and n_mine:
            cores = os.cpu_count() or 1
            hb = job.host[0][0]
            v, reps, dt = cpu_decode_rate(hb, cores, args.cpu_seconds)
            try:
                one, _, _ = cpu_decode_rate(hb, 1, 1.0)
            except Exception:
                one = None
            cpu = {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port", "cpu_model": cpu_model(), "one_thread": one,
                   "sample": f"{reps} x one full {args.workload} unit ({hb.n_samples} samples) in {dt:.1f}s, frames sharded over "
                             f"{cores} threads (one_thread: the same port on a single thread, >= 1 s)"}
        if not args.no_extra and args.workload == "c2" and args.scaling == "weak":
            job.close()
            extra = {}
            # Mixed shapes keep fewer lanes of a warp busy, so these batches need more of them in flight than c2 to
            # fill the chip (c4, 1100-frame units: 48 in flight 95, 96 -> 126, 128 -> 146 Gsamples/s,
            # profiles/c4_units_in_flight_r02.txt); c5's frames are 128 times longer than their count suggests.
            cx = cb.Context(device=local, n_streams=128, host_threads=host_threads)
            # (c2-indep: SURVEY §8d asks for the independent-stereo variant of C2 next to the mid/side headline)
            for wl, nu in (("c2-indep", 128), ("c3", 16), ("c4", 128), ("c5", 16)):
                try:
                    extra[wl] = short_line(cb, synth, cx, wl, nu, min(128, nu))
                except Exception as e:  # never lose the headline line to an auxiliary measurement
                    extra[wl] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        e2e_main = e2e.get("e2e", {"value": None, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        line = {
            "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm_steps, "ms_per_step": ms / timed_steps, "timed_steps": timed_steps,
            "region_ms": regions, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int32 samples / int64 accumulate", "data": "synthetic", "config": config, "bit_exact": bool(exact),
            "clocks": clocks, "gpu_launches": gpu_launches,
            "single_batch": {"kernel_ms": single_ms, "value": (job.unit_samples[0] / (single_ms / 1e3) / 1e6) if single_ms else None,
                             "unit": "Msamples/s", "note": "one batch, nothing else in flight (latency regime)"},
            "e2e": e2e_main, "e2e_i16": e2e.get("e2e_i16"),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src, "per": "GPU", "algorithmic_bytes_per_step": job.unit_alg[0] if n_mine else None,
                         "kernels": "all kernels of a step's graph (index_frames_kernel + decode_subframes_kernel<0,false> do the work; "
                                    "alone, same regime: 3.7 + 13.5 us of the step, profiles/SUMMARY_r02.md)",
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                         "traffic_source": (traffic or {}).get("source")},
            "cpu_baseline": cpu, "host_demux": demux, "workloads": extra,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
