#!/usr/bin/env python
"""bench.py -- throughput of the FLAC block encode/decode hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg2_l8|cfg3|cfg4|cfg5] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch (BASELINE configs: 10 000 blocks of 4096 samples; cfg4: 125 files
of 100 blocks per GPU). Prints ONE JSON line (rank 0). See DESIGN.md "Measurement" for the definitions:
  value      whole-job Msamples/s (samples = blocks x blocksize x channels), inputs resident in HBM,
             CUDA events on the launching stream, max over ranks.
  e2e        the same through the C ABI with HOST (pinned) buffers: H2D + kernels + D2H inside the timed region.
             16-/24-bit streams go in as packed little-endian PCM (fb200_encode_host_packed: what a WAV reader
             holds); e2e_int32 is the same through the int32 layout of FLAC__stream_encoder_process_interleaved.
  roofline   dominant kernel: algorithmic bytes per launch / mean launch duration (CUDA events recorded between the
             kernels in the timed region) against the measured HBM peak.
  cpu_baseline / --impl reference
             the compiled reference libFLAC (oracle/_ref) on this box's host cores: one encoder per host thread over
             contiguous block ranges (the honest "all cores" arm for a batch of independent blocks / files), best of
             N; the single-encoder set_num_threads(64) figure and the 1-thread figure are reported next to it.
  frames_compared / frames_equal
             every frame of the GPU stream memcmp'ed against the reference's frame for the same block, in this run.
Without --workload the default line is cfg2 and the other BASELINE configs ride along under extra.workloads,
so that one driver invocation measures all of them. Every timed loop runs K steps.
--dump-outputs DIR
             after the timed steps, rank 0 writes what the last device-resident step of each workload computed to
             DIR/<workload>_<array>.npy (float64, or float32 for bytes), so that two builds can be compared output for
             output: the inputs depend only on the arguments. Encode: every frame offset, and the bytes of a fixed,
             seeded sample of frames; decode: every frame status word and the samples of such a sample of frames.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (channels, bps, rate, level, blocks per GPU per step, blocksize, blocks per file (0 = one stream), description)
    "cfg2": (2, 16, 44100, 5, 10000, 4096, 0, "stereo 16-bit 44.1 kHz, -5, 10 000 blocks of 4096 (BASELINE configs[1])"),
    "cfg2_l8": (2, 16, 44100, 8, 10000, 4096, 0, "stereo 16-bit 44.1 kHz, -8, 10 000 blocks of 4096 (the >=100x target config)"),
    "cfg3": (2, 24, 96000, 8, 10000, 4096, 0, "stereo 24-bit 96 kHz, -8, 10 000 blocks of 4096 (BASELINE configs[2])"),
    "cfg4": (8, 24, 192000, 8, 12500, 4096, 100, "8-channel 24-bit 192 kHz, -8, 125 files x 100 blocks per GPU = 1 000 files over 8 GPUs, file index mod world (BASELINE configs[3])"),
    "cfg5": (2, 16, 44100, 8, 100000, 4096, 0, "decode-only: 100 000 pre-encoded -8 stereo 16-bit frames, offsets supplied (BASELINE configs[4])"),
}
DATA_NOTE = "synthetic: music-like base (SURVEY 8d-i generator) of 256 blocks tiled over the batch + independent +-1 LSB dither per sample"

_pcm_cache = {}
DUMP_FRAMES = 64          # frames per workload in the --dump-outputs sample
DUMP_SEED = 20240601
DUMP_LIMIT = 64 << 20     # bytes, all .npy payloads together


def make_pcm(ch, bps, rate, blocks, bs, seed):
    """Music-like base (SURVEY.md 8d-i) of 256 blocks, tiled, plus independent +-1 LSB dither so that
    no two frames are identical. Deterministic in `seed`."""
    key = (ch, bps, rate, blocks, bs, seed)
    if key in _pcm_cache:
        return _pcm_cache[key]
    import signals
    base_blocks = min(256, blocks)
    base = signals.music_like(base_blocks * bs, ch, bps, rate, seed=seed).astype(np.int32)
    reps = (blocks + base_blocks - 1) // base_blocks
    x = np.tile(base, (reps, 1))[: blocks * bs]
    rng = np.random.default_rng(seed + 12345)
    x = x + rng.integers(-1, 2, size=x.shape, dtype=np.int8)
    lim = (1 << (bps - 1)) - 1
    np.clip(x, -lim - 1, lim, out=x)
    x = np.ascontiguousarray(x.astype(np.int32))
    _pcm_cache.clear()  # one batch at a time (cfg4 is 1.6 GB)
    _pcm_cache[key] = x
    return x


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = []
        with open(self.f.name) as fh:
            for line in fh:
                parts = [s.strip() for s in line.split(",")]
                if len(parts) >= 9:
                    rows.append(parts)
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = []
        reasons = set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            hi = [v for v in sm if v >= 0.5 * max(sm)]  # "under load" = samples in the upper half of the observed range
            out["sm_mhz"] = float(np.median(hi))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh)
    return {}


class Ranks:
    """One process per GPU; the path shards by block ranges / files with no data-path collective, so the only
    collectives are the barrier and the MAX/SUM reductions of timings and unit counts."""

    def __init__(self, backend=None, device=None):
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dist = None
        self.device = device
        if self.world > 1:
            import torch
            import torch.distributed as dist
            self.dist = dist
            if backend == "nccl":
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            else:
                dist.init_process_group(backend or "gloo")

    def shard_seed(self, base=1):
        """Every rank encodes its own block range / files: distinct, deterministic input per rank
        (cfg4: rank r owns the files f with f mod world == r)."""
        return base + self.rank

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def _reduce(self, v, op):
        if self.dist is None:
            return float(v)
        import torch
        t = torch.tensor([float(v)], dtype=torch.float64, device=self.device or "cpu")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, v):
        return self._reduce(v, self.dist.ReduceOp.MAX if self.dist else None)

    def sum(self, v):
        return self._reduce(v, self.dist.ReduceOp.SUM if self.dist else None)

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()
            self.dist = None


def host_threads():
    return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------- reference (CPU) arm
def reference_encode_rates(x, bps, rate, level, bs, reps, single_reps=None, one_thread_blocks=400):
    """The reference libFLAC on this box's host cores over the blocks of x:
      per_core : one encoder per host thread, contiguous block ranges (ref_encode_parallel), best of `reps`
      single   : ONE encoder with set_num_threads(min(cores, 64)) -- libFLAC's own multithreading, best of `single_reps`
      one      : one encoder, one thread, on the first `one_thread_blocks` blocks
    Msamples/s, samples of all channels."""
    import reflib
    n, ch = x.shape
    nt = host_threads()
    # worker counts tried: every hardware thread, and one per two (physical cores on SMT hosts) -- the better one counts
    best, best_w = None, nt
    for w in sorted({nt, max(1, nt // 2)}, reverse=True):
        for _ in range(reps + 1):  # first pass is the warm-up
            sec, nfr, _ = reflib.encode_parallel(x, bps, rate, level, bs, w)
            assert nfr == n // bs
            if best is None or sec < best:
                best, best_w = sec, w
    out = {"per_core": n * ch / best / 1e6, "cores": nt, "workers": best_w}
    st = min(nt, 64)  # FLAC__STREAM_ENCODER_MAX_THREADS
    tb = None
    for _ in range((single_reps if single_reps is not None else max(2, reps // 2)) + 1):
        t = time.perf_counter()
        reflib.encode(x, bps, rate=rate, level=level, blocksize=bs, threads=st, md5=False, want_bytes=False)
        dt = time.perf_counter() - t
        tb = dt if tb is None else min(tb, dt)
    out["single_encoder"] = n * ch / tb / 1e6
    out["single_encoder_threads"] = st
    nb1 = min(one_thread_blocks, n // bs)
    t1 = None
    for _ in range(2):
        t = time.perf_counter()
        reflib.encode(x[: nb1 * bs], bps, rate=rate, level=level, blocksize=bs, threads=1, md5=False, want_bytes=False)
        dt = time.perf_counter() - t
        t1 = dt if t1 is None else min(t1, dt)
    out["one_thread"] = nb1 * bs * ch / t1 / 1e6
    return out


def reference_frames(x, bps, rate, level, bs, file_blocks, variant="default"):
    """The reference's frames for every block of x, as one byte string per file (headers stripped) + frame sizes.
    variant: "default" = the shipped build flags, "strict" = the same sources without the four fast-math flags."""
    import reflib
    nt = min(host_threads(), 64)
    nblocks = x.shape[0] // bs
    per = file_blocks if file_blocks else nblocks
    streams, sizes = [], []
    for f0 in range(0, nblocks, per):
        s, hdr, frames = reflib.encode(x[f0 * bs:(f0 + per) * bs], bps, rate=rate, level=level, blocksize=bs, threads=nt, md5=False, variant=variant)
        streams.append(s[hdr:])
        sizes.extend(len(f) for f in frames)
    return b"".join(streams), np.asarray(sizes, dtype=np.uint64)


def compare_frames(gpu_stream, gpu_offsets, ref_bytes, ref_sizes):
    """memcmp of every frame: returns (frames_compared, frames_equal)."""
    n = len(ref_sizes)
    g_sizes = np.diff(gpu_offsets[: n + 1].astype(np.uint64))
    ref = np.frombuffer(ref_bytes, dtype=np.uint8)
    if np.array_equal(g_sizes, ref_sizes) and ref.size == int(gpu_offsets[n]) and np.array_equal(ref, gpu_stream[: ref.size]):
        return n, n
    r_off = np.concatenate([[0], np.cumsum(ref_sizes)]).astype(np.int64)
    equal = 0
    for i in range(n):
        a = gpu_stream[int(gpu_offsets[i]):int(gpu_offsets[i + 1])]
        b = ref[r_off[i]:r_off[i + 1]]
        equal += int(a.size == b.size and np.array_equal(a, b))
    return n, equal


def config_of(name, world):
    ch, bps, rate, level, blocks, bs, fblocks, desc = WORKLOADS[name]
    cfg = {"workload": f"{name}: {desc}", "channels": ch, "bits_per_sample": bps, "sample_rate": rate,
           "compression_level": level, "blocks_per_gpu_per_step": blocks, "blocksize": bs,
           "sharding": f"{world} rank(s) x independent " + ("files (file index mod world)" if fblocks else "block ranges") + ", no data-path collective",
           "l2_policy": "inputs (%.0f MB int32/step/GPU) exceed the 126 MB L2" % (blocks * bs * ch * 4 / 1e6)}
    if fblocks:
        cfg["blocks_per_file"] = fblocks
        cfg["files_per_gpu"] = blocks // fblocks
    return cfg


def run_reference_arm(args, name):
    ch, bps, rate, level, blocks, bs, fblocks, desc = WORKLOADS[name]
    if args.blocks:
        blocks = args.blocks
    config = config_of(name, args.gpus)
    config["blocks_per_gpu_per_step"] = blocks
    nthreads = host_threads()
    steps = args.steps
    if name == "cfg5":
        # the reference decoder is single-threaded per stream; every host core decodes its own stream
        # (ctypes releases the GIL), as a many-file batch would
        import reflib
        from concurrent.futures import ThreadPoolExecutor
        sample_blocks = 500
        x = make_pcm(ch, bps, rate, sample_blocks, bs, seed=1)
        ref_stream, _, _ = reflib.encode(x, bps, rate=rate, level=level)
        times = []
        with ThreadPoolExecutor(nthreads) as pool:
            for i in range(args.warmup + steps):
                t0 = time.perf_counter()
                list(pool.map(lambda _: reflib.decode(ref_stream, sample_blocks * bs, ch)[0].shape, range(nthreads)))
                if i >= args.warmup:
                    times.append(time.perf_counter() - t0)
        best = min(times)
        val = nthreads * sample_blocks * bs * ch / best / 1e6
        cpu = {"value": round(val, 3), "unit": "Msamples/s", "cores": nthreads, "kind": "reference",
               "sample": f"{nthreads} streams x {sample_blocks} frames per step, one reference libFLAC 1.5.0 stream decoder per host thread, MD5 off, in-memory callbacks, best of {steps}"}
        metric, ms = "decode_msamples_per_s", 1e3 * best
    else:
        x = make_pcm(ch, bps, rate, blocks, bs, seed=1)
        r = reference_encode_rates(x, bps, rate, level, bs, reps=steps)
        val = r["per_core"]
        ms = blocks * bs * ch / val / 1e3
        cpu = {"value": round(val, 3), "unit": "Msamples/s", "cores": r["cores"], "workers": r["workers"], "kind": "reference",
               "value_single_encoder": round(r["single_encoder"], 3), "single_encoder_threads": r["single_encoder_threads"],
               "value_1_thread": round(r["one_thread"], 3),
               "sample": f"all {blocks} blocks of the workload per step, reference libFLAC 1.5.0 (oracle/_ref, shipped flags), one encoder per host thread "
                         f"over contiguous block ranges, MD5 off, in-memory callbacks, best of {steps}; value_single_encoder = one encoder with set_num_threads"}
        metric = "encode_msamples_per_s"
    return {"impl": "reference", "metric": metric, "value": round(val, 3), "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": DATA_NOTE, "config": config, "cpu_baseline": cpu,
            "e2e": {"value": round(val, 3), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def dump_sample(blocks):
    """The frames whose contents --dump-outputs writes: a fixed, seeded choice, the same for the same arguments."""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(blocks, min(DUMP_FRAMES, blocks), replace=False))


def write_dump(path, arrays):
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT}"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- B200 arm: decode
def bench_decode(args, ranks, name, steps, warmup, with_cpu, dump=None):
    import ctypes as C
    import torch
    import flac_b200
    rank, local_rank, world = ranks.rank, ranks.local_rank, ranks.world
    ch, bps, rate, level, blocks, bs, fblocks, desc = WORKLOADS[name]
    if args.blocks:
        blocks = args.blocks
    config = config_of(name, world)
    x = make_pcm(ch, bps, rate, blocks, bs, seed=ranks.shard_seed())
    enc = flac_b200.Encoder(flac_b200.preset(ch, bps, rate, level, bs), device=local_rank, max_blocks_per_launch=4096)
    stream_np, offs_np = enc.encode(x)
    enc.close()
    total_bytes = int(offs_np[blocks])
    h_stream = torch.empty(total_bytes + 64, dtype=torch.uint8, pin_memory=True)
    h_stream.numpy()[:total_bytes] = stream_np
    h_stream.numpy()[total_bytes:] = 0
    h_offs = torch.empty(blocks + 1, dtype=torch.int64, pin_memory=True)
    h_offs.numpy()[:] = offs_np.view(np.int64)
    d_stream = h_stream.to("cuda")
    d_offs = h_offs.to("cuda")
    d_pcm = torch.empty((blocks * bs, ch), dtype=torch.int32, device="cuda")
    d_status = torch.empty(blocks, dtype=torch.int32, device="cuda")
    h_pcm = torch.empty((blocks * bs, ch), dtype=torch.int32, pin_memory=True)
    dec = flac_b200.Decoder(ch, bps, rate, bs, device=local_rank, max_frames_per_launch=131072)
    stream = torch.cuda.current_stream()

    def step_device():
        dec.decode_device(d_stream.data_ptr(), d_offs.data_ptr(), blocks, d_pcm.data_ptr(), blocks * bs, d_status.data_ptr(), stream.cuda_stream)

    nbytes_out = 2 if bps <= 16 else 3
    h_packed = torch.empty(blocks * bs * ch * nbytes_out, dtype=torch.uint8, pin_memory=True)

    def step_host():
        # the call a client makes: frames in pinned host memory -> packed 16-/24-bit PCM in pinned host memory
        ns, bad = C.c_uint64(0), C.c_uint32(0)
        rc = flac_b200.lib().fb200_decode_host_packed(dec._h, h_stream.data_ptr(), h_offs.data_ptr(), blocks, h_packed.data_ptr(), nbytes_out, blocks * bs,
                                                      C.byref(ns), C.byref(bad))
        assert rc == 0 and bad.value == 0

    def step_host_int32():
        ns, bad = C.c_uint64(0), C.c_uint32(0)
        rc = flac_b200.lib().fb200_decode_host(dec._h, h_stream.data_ptr(), h_offs.data_ptr(), blocks, h_pcm.data_ptr(), blocks * bs, C.byref(ns), C.byref(bad))
        assert rc == 0 and bad.value == 0

    for _ in range(warmup):
        step_device()
    torch.cuda.synchronize()
    assert int((d_status & 0xff).sum().item()) == 0, "decode errors"
    assert torch.equal(d_pcm.cpu(), torch.from_numpy(x)), "decoded PCM differs from the input"

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dec.set_profiling(True)
    dec.profile(reset=True)
    launches0 = dec.launches
    ranks.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        step_device()
    ev1.record(stream)
    torch.cuda.synchronize()
    ranks.barrier()
    dev_ms = ranks.max(ev0.elapsed_time(ev1))
    launches = dec.launches - launches0
    if dump is not None and rank == 0:  # what the last timed step decoded: status per frame, samples of the sampled frames
        pick = torch.from_numpy(dump_sample(blocks)).to("cuda")
        dump[f"{name}_status"] = d_status.cpu().numpy().astype(np.float64)
        dump[f"{name}_pcm_sample"] = d_pcm.view(blocks, bs, ch)[pick].cpu().numpy().astype(np.float64)
        dump[f"{name}_sample_frames"] = pick.cpu().numpy().astype(np.float64)
    prof = dec.profile(reset=True)
    dec.set_profiling(False)

    for _ in range(2):
        step_host()
    ranks.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host()
    e2e_s = ranks.max(time.perf_counter() - t0)
    ranks.barrier()
    step_host_int32()
    ranks.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host_int32()
    e2e32_s = ranks.max(time.perf_counter() - t0) / steps
    ranks.barrier()
    clocks = sampler.stop() if rank == 0 else None
    assert np.array_equal(h_pcm.numpy(), x), "e2e decoded PCM (int32) differs from the input"
    assert np.array_equal(h_packed.numpy(), flac_b200.pack_pcm(x, nbytes_out)), "e2e decoded PCM (packed) differs from the input"

    samples_per_step = blocks * bs * ch
    total_samples = ranks.sum(float(samples_per_step))
    value = total_samples * steps / (dev_ms / 1e3) / 1e6
    e2e_value = total_samples * steps / e2e_s / 1e6
    dec.close()
    if rank != 0:
        return None
    peak, peak_src = peaks()
    frame_bytes = total_bytes / blocks
    # k_dec_walk measures subframes 0..ch-2 (reads that share of the frame), k_dec_frames reads the frame and writes the PCM
    per_frame = {"k_dec_walk": frame_bytes * (ch - 1) / ch, "k_dec_crc": frame_bytes, "k_dec_frames": frame_bytes + 4 * bs * ch}
    total_kernel_ms = sum(v[0] for v in prof.values()) or 1.0
    kernels = {}
    for kname, (ms, n) in prof.items():
        if n == 0:
            continue
        alg = per_frame.get(kname, 0) * blocks * steps / n
        avg_ms = ms / n
        kernels[kname] = {"ms_per_launch": round(avg_ms, 4), "launches": n, "share": round(ms / total_kernel_ms, 4),
                          "alg_bytes_per_launch": int(alg), "achieved_gbs": round(alg / (avg_ms * 1e-3) / 1e9, 2),
                          "frac": round(alg / (avg_ms * 1e-3) / 1e9 / peak, 4)}
    dominant = max(kernels, key=lambda k: kernels[k]["share"])
    dk = kernels[dominant]
    traffic = ncu_traffic().get(name, {})
    roofline = {"kernel": dominant, "bound": "hbm", "achieved": dk["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dk["frac"],
                "traffic": traffic.get(dominant), "peak_source": peak_src, "share_of_step": dk["share"],
                "pipeline": {"alg_bytes_per_step": int((frame_bytes + 4 * bs * ch) * blocks),
                             "achieved_gbs": round((frame_bytes + 4 * bs * ch) * blocks * steps / (dev_ms * 1e-3) / 1e9, 2)},
                "kernels": kernels}
    cpu = None
    if with_cpu:
        try:
            import reflib
            if reflib.available("default"):
                sb = 2000
                xs = x[: sb * bs]
                ref_stream, _, _ = reflib.encode(xs, bps, rate=rate, level=level)
                t = []
                for i in range(3):
                    t0 = time.perf_counter()
                    y, info = reflib.decode(ref_stream, sb * bs, ch)
                    t.append(time.perf_counter() - t0)
                v1 = sb * bs * ch / min(t[1:]) / 1e6
                cpu = {"value": round(v1, 3), "unit": "Msamples/s", "cores": 1, "kind": "reference",
                       "sample": f"{sb} frames of this workload, reference libFLAC 1.5.0 stream decoder (single-threaded by design), MD5 off, in-memory callbacks"}
        except Exception as ex:
            cpu = {"value": None, "unit": "Msamples/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}
    return {
        "metric": "decode_msamples_per_s", "value": round(value, 3), "unit": "Msamples/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(dev_ms / steps, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": DATA_NOTE, "config": config,
        "e2e": {"value": round(e2e_value, 3), "unit": "Msamples/s", "h2d_bytes_per_step": int(total_bytes + 8 * (blocks + 1)),
                "d2h_bytes_per_step": int(samples_per_step * nbytes_out + 4 * blocks), "ms_per_step": round(1e3 * e2e_s / steps, 4), "bytes_are": "per GPU (rank 0)",
                "output": f"packed {8 * nbytes_out}-bit little-endian PCM in pinned host memory (fb200_decode_host_packed)"},
        "e2e_int32": {"value": round(total_samples / e2e32_s / 1e6, 3), "unit": "Msamples/s", "d2h_bytes_per_step": int(samples_per_step * 4 + 4 * blocks),
                      "ms_per_step": round(1e3 * e2e32_s, 4), "output": "int32 samples (fb200_decode_host)"},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        "bit_exact": "decoded PCM == input asserted in this run (device and e2e paths)",
    }


# ---------------------------------------------------------------------------------------------- B200 arm: encode
def bench_encode(args, ranks, name, steps, warmup, with_cpu, dump=None):
    import torch
    import flac_b200
    rank, local_rank, world = ranks.rank, ranks.local_rank, ranks.world
    ch, bps, rate, level, blocks, bs, fblocks, desc = WORKLOADS[name]
    if args.blocks:
        blocks = args.blocks if not fblocks else max(fblocks, args.blocks // fblocks * fblocks)
    config = config_of(name, world)
    config["blocks_per_gpu_per_step"] = blocks
    samples_per_step = blocks * bs * ch

    # every rank owns its own block range / files (different seed -> different "files")
    x = make_pcm(ch, bps, rate, blocks, bs, seed=ranks.shard_seed())
    nsamp = x.shape[0]
    h_pcm = torch.empty(x.shape, dtype=torch.int32, pin_memory=True)
    h_pcm.numpy()[:] = x
    d_pcm = h_pcm.to("cuda", non_blocking=False)
    nbytes = 2 if bps <= 16 else 3
    packed_np = flac_b200.pack_pcm(x, nbytes)
    h_packed = torch.empty(packed_np.size, dtype=torch.uint8, pin_memory=True)
    h_packed.numpy()[:] = packed_np
    del packed_np

    enc = flac_b200.Encoder(flac_b200.preset(ch, bps, rate, level, bs), device=local_rank,
                            max_blocks_per_launch=int(os.environ.get("FB200_BENCH_MAXBLOCKS", str(blocks))))
    if fblocks:
        enc.set_file_blocks(fblocks)
    out_cap = blocks * enc.max_frame_bytes + 64
    d_out = torch.empty(out_cap, dtype=torch.uint8, device="cuda")
    d_offs = torch.empty(blocks + 1, dtype=torch.int64, device="cuda")
    h_out = torch.empty(out_cap, dtype=torch.uint8, pin_memory=True)
    h_offs = torch.empty(blocks + 1, dtype=torch.int64, pin_memory=True)
    stream = torch.cuda.current_stream()

    def step_device():
        enc.encode_device(d_pcm.data_ptr(), nsamp, d_out.data_ptr(), out_cap, d_offs.data_ptr(), 0, stream.cuda_stream, sync=False)

    def step_host_int32():
        return enc.encode(h_pcm.numpy(), 0, out=h_out.numpy(), offsets=h_offs.numpy().view(np.uint64))

    def step_host_packed():
        return enc.encode_packed(h_packed.numpy(), nbytes, nsamp, 0, out=h_out.numpy(), offsets=h_offs.numpy().view(np.uint64))

    # ---- warm-up
    for _ in range(warmup):
        step_device()
    torch.cuda.synchronize()
    total_bytes = int(d_offs[blocks].item())

    # ---- timed region 1: device-resident (value): K steps between two CUDA events on the launching stream
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = enc.launches
    ranks.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        step_device()
    ev1.record(stream)
    torch.cuda.synchronize()
    ranks.barrier()
    dev_ms = ranks.max(ev0.elapsed_time(ev1))
    launches = enc.launches - launches0
    if dump is not None and rank == 0:  # what the last timed step encoded: every frame offset, the bytes of the sampled frames
        offs = d_offs.cpu().numpy()
        pick = dump_sample(blocks)
        dump[f"{name}_offsets"] = offs.astype(np.float64)
        dump[f"{name}_stream_sample"] = torch.cat([d_out[int(offs[i]):int(offs[i + 1])] for i in pick]).cpu().numpy().astype(np.float32)
        dump[f"{name}_sample_frames"] = pick.astype(np.float64)
    # ---- the same K steps again with CUDA events recorded BETWEEN the kernels (per-kernel durations for the roofline; the
    # events serialise the two kernels the engine otherwise overlaps, so this pass is a little slower than the timed one)
    enc.set_profiling(True)
    enc.profile(reset=True)
    torch.cuda.synchronize()
    evp0, evp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evp0.record(stream)
    for _ in range(steps):
        step_device()
    evp1.record(stream)
    torch.cuda.synchronize()
    prof_ms_per_step = evp0.elapsed_time(evp1) / steps
    prof = enc.profile(reset=True)
    enc.set_profiling(False)

    if args.kernels_only:
        if rank == 0:
            sampler.stop()
        enc.close()
        return {"kernels_only": True, "workload": name, "ms_per_step": dev_ms / steps, "ms_per_step_profiled": prof_ms_per_step, "profile": prof}

    # ---- timed region 2: end to end through the host-buffer C ABI (packed PCM in, frames + offsets out)
    def time_host(fn):
        for _ in range(2):
            fn()
        ranks.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = fn()
        torch.cuda.synchronize()
        dt = ranks.max(time.perf_counter() - t0)
        ranks.barrier()
        return dt, res

    e2e_s, (s_host, o_host) = time_host(step_host_packed)
    gpu_stream = s_host.copy()
    gpu_offsets = o_host.copy()
    e2e32_s, (s32, o32) = time_host(step_host_int32)
    clocks = sampler.stop() if rank == 0 else None
    assert int(o_host[blocks]) == total_bytes and int(o32[blocks]) == total_bytes, "device / packed / int32 paths disagree on the stream size"
    assert np.array_equal(s32, gpu_stream), "packed and int32 host paths produced different streams"

    total_samples = ranks.sum(float(samples_per_step))  # per step, all ranks
    value = total_samples * steps / (dev_ms / 1e3) / 1e6
    e2e_value = total_samples * steps / e2e_s / 1e6
    e2e32_value = total_samples * steps / e2e32_s / 1e6
    enc_nsig = enc.nsig
    enc.close()
    del d_pcm, d_out, d_offs
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    # ---- in-run frame parity: every frame of the GPU stream vs the reference's frame for the same block.
    # Two builds of the SAME reference sources are compared (DESIGN.md (c), SURVEY 0.3): "strict" (no fast-math flags: the
    # floating-point order the source states, which the engine follows by construction -> must be 100 %) and the shipped
    # flags (-fassociative-math ...: GCC re-associates the autocorrelation / Levinson sums; the two builds differ from EACH
    # OTHER on near-singular frames, so this count may fall short and is reported, not asserted).
    frames_compared = frames_equal = frames_equal_shipped = 0
    parity_note = "reference library not present on this box"
    try:
        import reflib
        if reflib.available("strict"):
            ref_bytes, ref_sizes = reference_frames(x, bps, rate, level, bs, fblocks, "strict")
            frames_compared, frames_equal = compare_frames(gpu_stream, gpu_offsets, ref_bytes, ref_sizes)
            del ref_bytes
            ref_bytes, ref_sizes = reference_frames(x, bps, rate, level, bs, fblocks, "default")
            _, frames_equal_shipped = compare_frames(gpu_stream, gpu_offsets, ref_bytes, ref_sizes)
            del ref_bytes
            parity_note = ("memcmp of every frame of the e2e stream against reference libFLAC 1.5.0 (oracle/_ref) in this run: frames_equal vs the build "
                           "without fast-math flags (source-order FP), frames_equal_shipped_flags vs the shipped-flags build (compiler-reassociated FP; "
                           "the two reference builds differ from each other on the frames missing there)")
    except Exception as ex:
        parity_note = f"reference run failed: {ex}"
    if frames_compared != frames_equal:
        raise AssertionError(f"{name}: {frames_compared - frames_equal} of {frames_compared} frames differ from the reference")

    # ---- roofline (rank 0's kernels)
    peak, peak_src = peaks()
    nsig = enc_nsig
    frame_bytes = total_bytes / blocks
    emit_direct = prof.get("k_gather", (0, 0))[1] == 0  # k_emit3 reads the caller's PCM and writes the frame in place
    # raw-PCM pipeline (k_autoc4 / k_search5 / k_emit3, ch <= 2): every kernel reads the caller's interleaved block once;
    # general path: k_prep writes planar signals that the others read
    sig_read = 4 * bs * ch if emit_direct else 4 * bs * nsig
    per_block_bytes = {
        "k_prep": 4 * bs * ch + (0 if emit_direct else 4 * bs * nsig),
        "k_autoc": sig_read,
        "k_lpc": 0,
        "k_search": sig_read,
        "k_emit": 4 * bs * ch + frame_bytes,
        "k_scan": 12,
        "k_gather": 2 * frame_bytes,
    }
    kernel_names = ({"k_prep": "k_meta (only when the wasted-bits OR is not fused into k_autoc4)", "k_autoc": "k_autoc4", "k_lpc": "k_lpc", "k_search": "k_search5",
                     "k_emit": "k_emit3"} if emit_direct else
                    {"k_prep": "k_prep", "k_autoc": "k_autoc3 / k_autoc", "k_lpc": "k_lpc", "k_search": "k_search5 / k_search", "k_emit": "k_emit", "k_scan": "k_scan",
                     "k_gather": "k_gather"})
    traffic_per_block = ncu_traffic().get(name, {})
    traffic = {}
    total_kernel_ms = sum(v[0] for v in prof.values()) or 1.0
    kernels = {}
    for kname, (ms, n) in prof.items():
        if n == 0 or ms / n < 0.004:  # an empty profiling slot (no kernel between its two events)
            continue
        blocks_per_launch = blocks * steps / n
        if isinstance(traffic_per_block.get(kname), (int, float)):
            traffic[kname] = int(traffic_per_block[kname] * blocks_per_launch)
        alg = per_block_bytes[kname] * blocks_per_launch
        avg_ms = ms / n
        kernels[kname] = {"ms_per_launch": round(avg_ms, 4), "launches": n, "share": round(ms / total_kernel_ms, 4),
                          "alg_bytes_per_launch": int(alg), "achieved_gbs": round(alg / (avg_ms * 1e-3) / 1e9, 2),
                          "frac": round(alg / (avg_ms * 1e-3) / 1e9 / peak, 4)}
    dominant = max(kernels, key=lambda k: kernels[k]["share"])
    dk = kernels[dominant]
    roofline = {"kernel": dominant, "bound": "hbm", "achieved": dk["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dk["frac"],
                "traffic": traffic.get(dominant), "peak_source": peak_src, "share_of_step": dk["share"],
                "residual_rice_kernel": {"kernel": "k_emit3" if emit_direct else "k_emit", **kernels.get("k_emit", {})},
                "pipeline": {"alg_bytes_per_step": int((4 * bs * ch + frame_bytes) * blocks),
                             "achieved_gbs": round((4 * bs * ch + frame_bytes) * blocks * steps / (dev_ms * 1e-3) / 1e9, 2)},
                "profiled_ms_per_step": round(prof_ms_per_step, 4),
                "kernel_names": kernel_names, "kernels": kernels}

    # ---- CPU baseline: compiled reference on the host cores, the same procedure as --impl reference
    cpu = None
    if with_cpu:
        try:
            import reflib
            if reflib.available("default"):
                r = reference_encode_rates(x, bps, rate, level, bs, reps=5 if args.full_cpu else 3)
                cpu = {"value": round(r["per_core"], 3), "unit": "Msamples/s", "cores": r["cores"], "workers": r["workers"], "kind": "reference",
                       "value_single_encoder": round(r["single_encoder"], 3), "single_encoder_threads": r["single_encoder_threads"],
                       "value_1_thread": round(r["one_thread"], 3),
                       "sample": f"all {blocks} blocks of this workload, reference libFLAC 1.5.0 built from /root/reference (oracle/_ref, shipped flags), one encoder per "
                                 f"host thread over contiguous block ranges, MD5 off, in-memory callbacks, best of 3-5 (the --impl reference procedure)"}
        except Exception as ex:  # the baseline is reported, never required for the GPU number
            cpu = {"value": None, "unit": "Msamples/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}

    return {
        "metric": "encode_msamples_per_s", "value": round(value, 3), "unit": "Msamples/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(dev_ms / steps, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": DATA_NOTE, "config": config,
        "e2e": {"value": round(e2e_value, 3), "unit": "Msamples/s", "h2d_bytes_per_step": int(nsamp * ch * nbytes),
                "d2h_bytes_per_step": int(total_bytes + 8 * (blocks + 1)), "ms_per_step": round(1e3 * e2e_s / steps, 4), "bytes_are": "per GPU (rank 0)",
                "input": f"packed {8 * nbytes}-bit little-endian PCM in pinned host memory (fb200_encode_host_packed)"},
        "e2e_int32": {"value": round(e2e32_value, 3), "unit": "Msamples/s", "h2d_bytes_per_step": int(nsamp * ch * 4),
                      "d2h_bytes_per_step": int(total_bytes + 8 * (blocks + 1)), "ms_per_step": round(1e3 * e2e32_s / steps, 4),
                      "input": "int32 interleaved (the layout of FLAC__stream_encoder_process_interleaved) in pinned host memory (fb200_encode_host)"},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        "frames_compared": int(frames_compared), "frames_equal": int(frames_equal), "frames_equal_shipped_flags": int(frames_equal_shipped),
        "bit_exact": parity_note,
        "compressed_bytes_per_step": total_bytes,
    }


def summarize(line):
    """What an extra workload contributes to the default line."""
    if line is None:
        return None
    keep = {k: line[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "gpu_launches") if k in line}
    keep["e2e"] = line.get("e2e")
    if "e2e_int32" in line:
        keep["e2e_int32"] = line["e2e_int32"]
    r = line.get("roofline") or {}
    keep["roofline"] = {"kernel": r.get("kernel"), "frac": r.get("frac"), "achieved": r.get("achieved"), "share_of_step": r.get("share_of_step"),
                        "kernels": {k: {"ms_per_launch": v["ms_per_launch"], "frac": v["frac"], "share": v["share"]} for k, v in (r.get("kernels") or {}).items()}}
    for k in ("frames_compared", "frames_equal", "frames_equal_shipped_flags", "bit_exact", "cpu_baseline", "compressed_bytes_per_step"):
        if k in line:
            keep[k] = line[k]
    keep["config"] = line.get("config")
    return keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--blocks", type=int, default=0, help="override the number of blocks (debug)")
    ap.add_argument("--kernels-only", action="store_true", help="profiling aid: device-resident steps only (no e2e, no CPU baseline)")
    ap.add_argument("--no-extras", action="store_true", help="default invocation: only the cfg2 line, no extra.workloads")
    ap.add_argument("--full-cpu", action="store_true", help="cpu_baseline with best of 5 instead of 3")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each workload computed to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    primary = args.workload or "cfg2"
    rank = int(os.environ.get("RANK", "0"))

    # ------------------------------------------------------------------ reference arm (rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        print(json.dumps(run_reference_arm(args, primary)))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: flac_b200 has no CPU fallback"}))
        return 2
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    ranks = Ranks(backend="nccl", device="cuda")

    dump = {} if args.dump_outputs else None

    def run(name, steps, warmup, with_cpu):
        fn = bench_decode if name == "cfg5" else bench_encode
        return fn(args, ranks, name, steps, warmup, with_cpu, dump)

    line = run(primary, args.steps, args.warmup, True)
    if args.workload is None and not args.no_extras and not args.kernels_only:
        extras = {}
        for name in ("cfg2_l8", "cfg3", "cfg4", "cfg5"):
            try:
                extras[name] = summarize(run(name, args.steps, 3, True))
            except AssertionError:
                raise
            except Exception as ex:  # an extra must never take the headline line down
                extras[name] = {"error": f"{type(ex).__name__}: {ex}"}
        if ranks.rank == 0:
            line["extra"] = {"workloads": extras,
                             "note": "the other BASELINE configs, same procedure; parity counted per workload"}
    if ranks.rank == 0:
        if dump is not None:
            write_dump(args.dump_outputs, dump)
        print(json.dumps(line))
    ranks.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
