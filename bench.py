#!/usr/bin/env python
"""bench.py -- SEA hot-path throughput on B200 (BASELINE.json metric: decode & encode Msamples/s, fraction of roofline).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   our arm (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference [--gpus N --steps K --warmup W] the reference's own CPU decoder on the host cores

A "step" is one pass of the hot path over one batch of synthetic streams.  Headline (`value`) = batch decode of BASELINE
config 4 (4096 independent stereo 60 s 44.1 kHz CBR-3 streams PER GPU, weak scaling: every rank owns its own 4096 streams,
nothing is exchanged on the data path), .sea bytes resident in HBM.  The same JSON line carries

  strong        the split the configs themselves state: config 4 = 4096 streams in TOTAL, config 5 = 1024 streams in TOTAL,
                sharded /N over the ranks (dist.shard_streams), max over ranks
  sweep         BASELINE config 5: CBR 1..8 and VBR 1.5..7.3 batch encode of the (sharded) 1024 streams, each row with its INT32
                roofline fraction, its VBR tie count and the decode of what it produced (HBM roofline fraction)
  e2e           the headline through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region), all
                streams of the config per step, next to a plain-copy control of the same bytes (frac_of_copy_ceiling)
  e2e_encode    sea_b200_encode_batch with host buffers, config-5 shape
  roofline      HBM roofline of the decode kernel; cpu_baseline: the reference's C decoder on this box's host cores

Inputs: every stream is unique (tone + noise, generated on the device by the library's synth kernel, bit-identical to
sea_codec_b200/synth.py); the encode streams are selected so that the VBR-3 row has no error ties across a bucket boundary
(where the reference's sort_unstable order -- encoder_vbr.rs:102-103 -- would make "bit-exact" undefined; SURVEY 8d / T13).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)

RATE, CHANNELS, SECONDS = 44100, 2, 60
ALG_OPS_PER_CAND_SAMPLE = 49  # SURVEY.md 8d op count of encoder_base.rs:64-89 + lms.rs
CBR_ROWS = [1, 2, 3, 4, 5, 6, 7, 8]
VBR_ROWS = [1.5, 2.0, 2.5, 3.0, 3.5, 4.0, 5.0, 6.0, 7.0, 7.3]
DUMP_STREAMS, DUMP_WINDOW = 4096, 2048  # --dump-outputs: at most 4096 x 2048 samples, 32 MB as float32


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def host_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"nproc": os.cpu_count(), "usable_cores": host_cores(), "cpu_model": model}


def bind_to_gpu_numa_node(index: int) -> None:
    """Pins this rank's host threads (and so its first-touch pinned buffers) to the CPUs NVML reports as local to the GPU: the
    host-buffer (e2e) path moves ~6.5 GB per step over PCIe, and with several ranks per box remote-node buffers share one
    inter-socket link."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
    except Exception:
        pass


def ncu_traffic(streams: int, seconds: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the decode kernel per launch, from the committed `ncu --set full` capture
    (profiles/r0X_decode_traffic.json: bytes per stream of the 60 s config-4 shape); None when the shape differs."""
    for name in ("r02_decode_traffic.json", "r01_decode_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        try:
            t = json.load(open(p))
            if seconds != t["seconds"]:
                return None
            return float(t["dram_bytes_per_launch"]) / t["streams"] * streams
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None  # the timed region (perf_counter): only samples that arrived inside it are reported

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        inside = [ln for t, ln in self.lines if self.t0 is None or (self.t0 <= t <= (self.t1 or t) + 0.06)]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference arm

def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_decode_baseline(threads: int, reps: int, seconds: int = SECONDS, prefer_ref: bool = True):
    """Times the reference's CPU decode of one config-4 stream per core.  kind 'reference' = the reference's own C decoder
    (c/sea.h compiled into oracle/_ref, forked workers); 'port' = the oracle restatement (pthreads)."""
    from oracle import sea_oracle as O
    from sea_codec_b200 import synth

    pcm = synth.gen_stream(0, seconds * RATE, CHANNELS, RATE)
    st = O.make_settings(3.0)
    t0 = time.perf_counter()
    sea = O.sea_encode(pcm, RATE, CHANNELS, st)
    enc_single_s = time.perf_counter() - t0
    if prefer_ref and os.path.exists(O.REF_BENCH_PATH):
        with tempfile.NamedTemporaryFile(suffix=".sea", delete=False) as f:
            f.write(sea)
            path = f.name
        try:
            secs, samples = O.ref_c_bench(path, threads, reps)
        finally:
            os.unlink(path)
        kind = "reference"
    else:
        secs, samples = O.bench("decode", threads, reps, pcm, RATE, CHANNELS, st, sea)
        kind = "port"
    return dict(kind=kind, secs=secs, samples=samples, value=samples / secs / 1e6, pcm=pcm, sea=sea, settings=st,
                enc_single_msamples=pcm.size / enc_single_s / 1e6)


def reference_arm(args, info):
    if info.rank != 0:
        return
    cores = host_cores()
    # a bounded sample: every core decodes one 60 s stereo stream `reps` times per step
    reps = 4
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_decode_baseline(cores, reps) if i == 0 else r_again(r, cores, reps)
        if i >= args.warmup:
            vals.append(r["value"])
    value = float(np.mean(vals))
    ms = 1e3 * (cores * reps * SECONDS * RATE * CHANNELS) / (value * 1e6)
    sample = f"{cores} host cores x {reps} decodes of one 60 s 44.1 kHz stereo CBR-3 stream per step (config-4 stream shape)"
    print(json.dumps({
        "impl": "reference", "metric": "decode_msamples_per_s", "value": value, "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": r["kind"], "sample": sample},
        "host": host_info(),
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def r_again(prev, cores, reps):
    from oracle import sea_oracle as O

    if prev["kind"] == "reference":
        with tempfile.NamedTemporaryFile(suffix=".sea", delete=False) as f:
            f.write(prev["sea"])
            path = f.name
        try:
            secs, samples = O.ref_c_bench(path, cores, reps)
        finally:
            os.unlink(path)
    else:
        secs, samples = O.bench("decode", cores, reps, prev["pcm"], RATE, CHANNELS, prev["settings"], prev["sea"])
    out = dict(prev)
    out.update(secs=secs, samples=samples, value=samples / secs / 1e6)
    return out


def workload_config(args):
    return {"workload": f"config4: batch decode of {args.streams} independent stereo {args.seconds} s 44.1 kHz CBR-3 .sea streams "
                        f"per GPU (chunk 5120, sf bits 4, sf frames 20); weak scaling, streams sharded by rank, no collectives",
            "streams_per_gpu": args.streams, "seconds": args.seconds, "sample_rate": RATE, "channels": CHANNELS,
            "unique_streams": args.streams, "l2": "inputs larger than L2 (no flush needed)"}


# ------------------------------------------------------------------------------------------------ our arm

class Batch:
    """A batch of equally long streams resident on the device: PCM [n][spp] and, once encoded, .sea [n][stride]."""

    def __init__(self, torch, dev, n, frames, channels):
        self.n, self.frames, self.channels, self.spp = n, frames, channels, frames * channels
        self.pcm = torch.empty(n * self.spp, dtype=torch.int16, device=dev)
        self.pcm_off = np.arange(n, dtype=np.uint64) * self.spp
        self.nframes = np.full(n, frames, dtype=np.uint32)


def encode_device(ctx, torch, dev, b: Batch, n, settings, rate, out=None):
    """Device-resident batch encode of the first n streams of b; returns (sea tensor, stride, lens, kernel ms)."""
    bound = ctx.encode_bound(b.frames, b.channels, settings)
    stride = (bound + 15) // 16 * 16
    if out is None or out.numel() < n * stride:
        out = torch.zeros(n * stride, dtype=torch.uint8, device=dev)
    lens = ctx.encode_batch_device(b.pcm.data_ptr(), b.pcm_off[:n], b.nframes[:n], rate, b.channels, settings, out.data_ptr(),
                                   np.arange(n, dtype=np.uint64) * stride)
    return out, stride, lens, ctx.last_kernel_ms


def decode_device(ctx, sea, stride, lens, headers, pcm_out, spp, n):
    got = ctx.decode_batch_device(sea.data_ptr(), np.arange(n, dtype=np.uint64) * stride, lens[:n], headers[:n], pcm_out.data_ptr(),
                                  np.arange(n, dtype=np.uint64) * spp)
    return got, ctx.last_kernel_ms


def dump_outputs(out_dir, torch, pcm_out, got, n, spp):
    """Writes what the timed decode returned in its last step, as float32 / float64 .npy files: the samples decoded per stream
    and, for every stream (a seeded choice of DUMP_STREAMS when there are more), one seeded window of its decoded PCM.  The
    windows depend only on the stream count and length, so two builds run with the same arguments compare file for file."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    streams = np.arange(n, dtype=np.int64) if n <= DUMP_STREAMS else np.sort(rng.choice(n, DUMP_STREAMS, replace=False))
    width = min(spp, DUMP_WINDOW)
    starts = rng.integers(0, spp - width + 1, size=streams.size, dtype=np.int64)
    idx = streams[:, None] * spp + starts[:, None] + np.arange(width, dtype=np.int64)
    windows = pcm_out[torch.from_numpy(idx).to(pcm_out.device)].float().cpu().numpy()
    np.save(os.path.join(out_dir, "samples_per_stream.npy"), np.asarray(got, dtype=np.float64))
    np.save(os.path.join(out_dir, "pcm_windows.npy"), windows)
    np.save(os.path.join(out_dir, "pcm_window_stream_and_start.npy"), np.stack([streams, starts], axis=1).astype(np.float64))


def positive_int(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=40,  # ~0.6 s timed region: enough nvidia-smi clock samples
                    help="timed steps of the headline decode (value, ms_per_step); the secondary sections time their own "
                         "bounded repeat counts (1 to 10)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="decode streams per GPU (config 4, weak) and in total (strong)")
    ap.add_argument("--enc-streams", type=int, default=1024, help="encode streams per GPU (config 5, weak) and in total (strong)")
    ap.add_argument("--e2e-streams", type=int, default=512, help="streams per host-buffer call (a step loops over all streams)")
    ap.add_argument("--seconds", type=int, default=SECONDS)
    ap.add_argument("--skip-encode", action="store_true", help="skip the encode / sweep / secondary decode sections")
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of what the last timed decode step returned "
                                                          "(rank 0) to DIR/*.npy")
    args = ap.parse_args()

    from sea_codec_b200 import dist

    info = dist.init("gloo" if args.impl == "reference" else None)
    if args.impl == "reference":
        reference_arm(args, info)
        dist.shutdown()
        return

    import torch

    import sea_codec_b200 as S

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libsea_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(info.local_rank)
    bind_to_gpu_numa_node(info.local_rank)
    dev = torch.device("cuda", info.local_rank)
    ctx = S.Context(info.local_rank)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    W = info.world
    cbr3 = S.EncoderSettings()  # CBR 3, chunk 5120, sf bits 4, sf frames 20
    vbr3 = S.EncoderSettings(residual_bits=3.0, vbr=True)
    frames = args.seconds * RATE
    n, ns = args.streams, min(args.enc_streams, args.streams)
    peaks, peak_src = measured_peaks()
    hbm = peaks["hbm_gbs"]

    # ---- inputs: n unique streams per rank, generated on the device.  Stream ids are globally unique (rank * 2^20 + i); the
    # first ns (the encode batch) are re-drawn until the VBR-3 encode of them has no boundary tie.
    b = Batch(torch, dev, n, frames, CHANNELS)
    spp = b.spp
    ids = (info.rank << 20) + np.arange(n, dtype=np.uint32)
    torch.cuda.synchronize()
    ctx.synth_pcm_device(b.pcm.data_ptr(), spp, ids, frames, CHANNELS, RATE)
    tie_rounds, redrawn, fresh = 0, 0, (info.rank << 20) + (1 << 19)
    sea_v = None
    if not args.skip_encode:
        for tie_rounds in range(1, 13):
            sea_v, stride_v, lens_v, _ = encode_device(ctx, torch, dev, b, ns, vbr3, RATE, sea_v)
            per = ctx.last_vbr_ties_per_stream(ns)
            bad = np.nonzero(per)[0]
            if bad.size == 0:
                break
            for i in bad:
                ids[i] = fresh
                fresh += 1
            redrawn += int(bad.size)
            ctx.synth_pcm_device(b.pcm.data_ptr(), spp, ids[:ns], frames, CHANNELS, RATE)
        assert ctx.last_vbr_ties == 0, "could not draw a tie-free VBR-3 encode batch"

    # ---- config 4 inputs: every stream encoded by this library (CBR 3); 8 of them are checked against the oracle below
    sea, stride, lens, enc_all_ms = encode_device(ctx, torch, dev, b, n, cbr3, RATE)
    bound = int(lens[0])
    assert np.all(lens == bound)
    headers = sea.view(n, stride)[:, :22].cpu().numpy()
    pcm_out = torch.empty(n * spp, dtype=torch.int16, device=dev)
    samples_per_step = n * spp
    alg_bytes = float(n * bound + 2 * samples_per_step)

    kernel_ms = []

    def decode_step(m=n):
        got, ms = decode_device(ctx, sea, stride, lens, headers, pcm_out, spp, m)
        kernel_ms.append(ms)
        return got

    sampler = ClockSampler(info.local_rank)
    sampler.start()  # nvidia-smi needs a few hundred ms to deliver its first line: started before the warm-up, filtered to the timed region
    for _ in range(args.warmup):
        decode_step()
    kernel_ms.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    launches0 = ctx.launch_count
    sampler.begin()
    e0.record()
    for _ in range(args.steps):
        got = decode_step()
    e1.record()
    torch.cuda.synchronize()
    sampler.end()
    clocks = sampler.stop()
    dist.barrier()
    launches = ctx.launch_count - launches0
    ms_total = dist.max_over_ranks(e0.elapsed_time(e1))
    ms_per_step = ms_total / args.steps
    value = W * samples_per_step / (ms_per_step * 1e-3) / 1e6
    assert np.all(got == spp)
    if args.dump_outputs and info.rank == 0:
        dump_outputs(args.dump_outputs, torch, pcm_out, got, n, spp)
    k_ms = float(np.mean(kernel_ms))
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "decode_unrolled_kernel<2,3,pair-repl,S=4> (+ decode_staged_kernel<2,0> for the partial last chunks, "
                                          "side stream)",
                "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": ncu_traffic(n, args.seconds),
                "peak_source": peak_src, "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_msamples_per_s": samples_per_step / (k_ms * 1e-3) / 1e6}
    # the honest ALU view (SURVEY 8d): the recurrence is 23 algorithmic integer ops per sample (predict 8, unpack 2, dequant 1, add 1,
    # clamp 2, update 9) against the measured two-pipe INT32 issue peak; the kernel executes 16.0 warp instructions per sample
    # (profiles/r02_s2_final_dec_unrolled_4096_ncu_summary.txt: IMAD fuses multiply and add) -- it is issue-bound, not HBM-bound
    int_peak = max(ctx.int32_peak(m)[0] for m in (0, 1, 2))
    sps_k = samples_per_step / (k_ms * 1e-3)
    roofline["alu_view"] = {"algorithmic_ops_per_sample": 23, "achieved_tops": sps_k * 23 / 1e12, "int32_peak_tops": int_peak / 1e12,
                            "frac": sps_k * 23 / int_peak, "executed_instr_per_sample": 16.0, "executed_frac": sps_k * 16.0 / int_peak}

    # ---- parity on the benchmarked buffers, rank 0 at every N: 8 streams spread over the batch, GPU encode == oracle encode and
    # GPU decode == oracle decode (and == the reference's c/sea.h when oracle/_ref is there), bit for bit
    parity = None
    view = pcm_out.view(n, spp)
    dec0 = view[0].cpu().numpy()  # kept for the host-buffer comparison below (pcm_out is reused by the other sections)
    if info.rank == 0 and not args.skip_cpu:
        from oracle import sea_oracle as O
        from sea_codec_b200 import synth

        probe = sorted(set(int(x) for x in np.linspace(0, n - 1, 8)))
        host_pcm = {i: b.pcm.view(n, spp)[i].cpu().numpy() for i in probe}
        host_sea = {i: sea.view(n, stride)[i, :bound].cpu().numpy().tobytes() for i in probe}
        host_dec = {i: view[i].cpu().numpy() for i in probe}
        assert np.array_equal(host_pcm[probe[0]], synth.gen_stream(int(ids[probe[0]]), frames, CHANNELS, RATE)), "device synth != host recipe"
        have_ref = O.have_ref() and frames % 20 == 0

        def check(i):
            assert O.sea_encode(host_pcm[i], RATE, CHANNELS, O.make_settings(3.0)) == host_sea[i], f"stream {i}: GPU encode != oracle encode"
            assert np.array_equal(O.sea_decode(host_sea[i]).samples, host_dec[i]), f"stream {i}: GPU decode != oracle decode"
            return i

        with ThreadPoolExecutor(8) as ex:
            list(ex.map(check, probe))
        if have_ref:  # c/sea.h keeps static state: one stream, in this thread
            assert np.array_equal(O.ref_c_decode(host_sea[probe[-1]]).samples, host_dec[probe[-1]]), "GPU decode != c/sea.h decode"
        parity = {"streams_checked": probe, "encode_vs_oracle": "bit-exact", "decode_vs_oracle": "bit-exact",
                  "decode_vs_reference_c": "bit-exact (1 stream)" if have_ref else "not run"}
        if sea_v is not None:
            vprobe = sorted(set(int(x) for x in np.linspace(0, ns - 1, 4)))
            vsea = {i: sea_v.view(-1)[i * stride_v: i * stride_v + int(lens_v[i])].cpu().numpy().tobytes() for i in vprobe}
            vpcm = {i: b.pcm.view(n, spp)[i].cpu().numpy() for i in vprobe}

            def vcheck(i):
                ref, ties = O.sea_encode(vpcm[i], RATE, CHANNELS, O.make_settings(3.0, vbr=True), return_ties=True)
                assert ties == 0 and ref == vsea[i], f"stream {i}: GPU VBR-3 encode != oracle encode"

            with ThreadPoolExecutor(4) as ex:
                list(ex.map(vcheck, vprobe))
            parity["vbr3_encode_vs_oracle"] = {"streams_checked": vprobe, "result": "bit-exact", "ties": 0}
        del host_pcm, host_sea, host_dec

    # ---- strong scaling of config 4: 4096 streams in TOTAL, this rank decodes its shard
    strong = {}
    lo, hi = dist.shard_streams(n, info.rank, W)
    m4 = hi - lo
    ks = []
    for _ in range(2 + max(3, min(args.steps, 10))):
        _, ms = decode_device(ctx, sea, stride, lens, headers, pcm_out, spp, m4)
        ks.append(ms)
    ms4 = dist.max_over_ranks(float(np.mean(ks[2:])))
    strong["decode_config4"] = {"streams_total": n, "streams_per_gpu": m4, "value": n * spp / (ms4 * 1e-3) / 1e6, "unit": "Msamples/s",
                                "ms_per_step": ms4, "hbm_frac_per_gpu": (m4 * bound + 2.0 * m4 * spp) / (ms4 * 1e-3) / 1e9 / hbm}

    def hbm_row(n_streams, total_bytes, ms, kernel):
        gbs = total_bytes / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": kernel, "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm}

    def time_decode(sea_t, stride_t, lens_t, m, spp_t, reps=None):
        hd = sea_t.view(-1)[: m * stride_t].view(m, stride_t)[:, :22].cpu().numpy()
        ks = []
        for _ in range(2 + (reps or max(3, min(args.steps, 10)))):
            g, ms = decode_device(ctx, sea_t, stride_t, lens_t, hd, pcm_out, spp_t, m)
            ks.append(ms)
        assert np.all(g == spp_t)
        return float(np.mean(ks[2:]))

    # ---- the VBR twin of the headline (decode_vbr_kernel): the tie-free VBR-3 batch, ns streams per GPU
    vbr_dec = mc_dec = encode = sweep = None
    if not args.skip_encode:
        ms_v = dist.max_over_ranks(time_decode(sea_v, stride_v, lens_v, ns, spp))
        bytes_v = float(lens_v.sum() + 2 * ns * spp)
        vbr_dec = {"value": W * ns * spp / (ms_v * 1e-3) / 1e6, "unit": "Msamples/s", "streams_per_gpu": ns, "ms_per_step": ms_v,
                   "roofline": hbm_row(ns, bytes_v, ms_v, "decode_vbr_kernel<2,KF=3> (fixed-window form)")}

        # ---- BASELINE config 3 shape (8 channels, 48 kHz, CBR 4): 256 unique 60 s streams through decode_mc_kernel
        ch8, rate8, fr8, n8 = 8, 48000, args.seconds * 48000, 256
        b8 = Batch(torch, dev, n8, fr8, ch8)
        ctx.synth_pcm_device(b8.pcm.data_ptr(), b8.spp, (info.rank << 20) + (1 << 18) + np.arange(n8, dtype=np.uint32), fr8, ch8, rate8)
        sea8, stride8, lens8, _ = encode_device(ctx, torch, dev, b8, n8, S.EncoderSettings(residual_bits=4.0), rate8)
        ms8 = dist.max_over_ranks(time_decode(sea8, stride8, lens8, n8, b8.spp))
        mc_dec = {"value": W * n8 * b8.spp / (ms8 * 1e-3) / 1e6, "unit": "Msamples/s", "streams_per_gpu": n8, "channels": ch8,
                  "seconds": args.seconds, "ms_per_step": ms8,
                  "roofline": hbm_row(n8, float(lens8.sum() + 2 * n8 * b8.spp), ms8, "decode_mc_kernel<8,4>")}
        del b8, sea8
        torch.cuda.empty_cache()

        # ---- encode, config-5 shape.  INT32 roofline: measured two-pipe issue peak (sea_b200_int32_peak)
        peaks_int = {m: ctx.int32_peak(m)[0] for m in (0, 1, 2)}
        ops_peak = max(peaks_int.values())
        scratch = torch.zeros(ns * ((ctx.encode_bound(frames, CHANNELS, S.EncoderSettings(residual_bits=8.0)) + 15) // 16 * 16),
                              dtype=torch.uint8, device=dev)

        def time_encode(st_e, m, reps):
            out, stride_e, lens_e, _ = encode_device(ctx, torch, dev, b, m, st_e, RATE, scratch)  # warm-up
            ks = []
            for _ in range(reps):
                out, stride_e, lens_e, ms = encode_device(ctx, torch, dev, b, m, st_e, RATE, scratch)
                ks.append(ms)
            return float(np.mean(ks)), out, stride_e, lens_e

        def int_row(sps_per_gpu, passes):
            ops = ALG_OPS_PER_CAND_SAMPLE * 16 * passes  # 49 * 2^sf_bits * passes (SURVEY 8d)
            return {"bound": "int32", "achieved": sps_per_gpu * ops / 1e12, "peak": ops_peak / 1e12, "unit": "Tops/s",
                    "frac": sps_per_gpu * ops / ops_peak, "ops_per_sample": ops}

        encode = {"streams_per_gpu": ns, "int32_peak_lane_ops_per_s": {"imad": peaks_int[0], "lop3": peaks_int[1], "mixed": peaks_int[2]},
                  "tie_free_selection": {"rounds": tie_rounds, "streams_redrawn": redrawn, "of": ns}}
        reps_e = max(1, min(args.steps, 3))
        for name, st_e, passes in (("cbr3", cbr3, 1), ("vbr3", vbr3, 2)):  # weak: ns streams on every GPU
            dist.barrier()
            ms_e, _, _, lens_e = time_encode(st_e, ns, reps_e)
            ties_e = ctx.last_vbr_ties
            ms_e = dist.max_over_ranks(ms_e)
            encode[name] = {"value": W * ns * spp / (ms_e * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms_e,
                            "bytes_per_stream": int(lens_e[0]), "vbr_ties": int(dist.sum_over_ranks(ties_e)),
                            "roofline": int_row(ns * spp / (ms_e * 1e-3), passes)}
        # the machine full: every stream of the decode batch (n per GPU, 60 s) through the same kernel -- timed while building config 4
        encode["cbr3_all_streams"] = {"value": W * n * spp / (dist.max_over_ranks(enc_all_ms) * 1e-3) / 1e6, "unit": "Msamples/s",
                                      "ms_per_step": enc_all_ms, "streams_per_gpu": n, "seconds": args.seconds,
                                      "roofline": int_row(n * spp / (enc_all_ms * 1e-3), 1)}

        # ---- BASELINE config 5 as stated: ns streams in TOTAL sharded /N, every CBR and VBR bitrate; each row also decodes what it made
        lo5, hi5 = dist.shard_streams(ns, info.rank, W)
        m5 = hi5 - lo5  # this rank's shard = the first m5 of its own (tie-free) streams
        if not args.skip_sweep and m5 > 0:
            sweep = {"streams_total": ns, "streams_per_gpu": m5, "seconds": args.seconds, "rows": []}
            rows = [("cbr", float(r), S.EncoderSettings(residual_bits=float(r)), 1) for r in CBR_ROWS] + \
                   [("vbr", r, S.EncoderSettings(residual_bits=r, vbr=True), 2) for r in VBR_ROWS]
            for mode, bits, st_e, passes in rows:
                ms_e, out, stride_e, lens_e = time_encode(st_e, m5, 2)
                ties_e = ctx.last_vbr_ties if mode == "vbr" else 0
                ms_d = time_decode(out, stride_e, lens_e, m5, spp, reps=3)
                ms_e, ms_d = dist.max_over_ranks(ms_e), dist.max_over_ranks(ms_d)
                tot_bytes = dist.sum_over_ranks(float(lens_e.sum()))
                row = {"mode": mode, "residual_bits": bits, "bits_per_sample": 8.0 * tot_bytes / (ns * spp),
                       "encode_msamples_per_s": ns * spp / (ms_e * 1e-3) / 1e6, "encode_ms": ms_e,
                       "encode_int32_frac_per_gpu": m5 * spp / (ms_e * 1e-3) * ALG_OPS_PER_CAND_SAMPLE * 16 * passes / ops_peak,
                       "decode_msamples_per_s": ns * spp / (ms_d * 1e-3) / 1e6, "decode_ms": ms_d,
                       "decode_hbm_frac_per_gpu": (float(lens_e.sum()) + 2.0 * m5 * spp) / (ms_d * 1e-3) / 1e9 / hbm,
                       "vbr_ties": int(dist.sum_over_ranks(ties_e))}
                sweep["rows"].append(row)
                if mode == "cbr" and bits == 3.0:
                    strong["encode_config5_cbr3"] = {"streams_total": ns, "streams_per_gpu": m5, "value": row["encode_msamples_per_s"],
                                                     "unit": "Msamples/s", "ms_per_step": ms_e, "int32_frac_per_gpu": row["encode_int32_frac_per_gpu"]}
                if mode == "vbr" and bits == 3.0:
                    strong["encode_config5_vbr3"] = {"streams_total": ns, "streams_per_gpu": m5, "value": row["encode_msamples_per_s"],
                                                     "unit": "Msamples/s", "ms_per_step": ms_e, "int32_frac_per_gpu": row["encode_int32_frac_per_gpu"],
                                                     "vbr_ties": row["vbr_ties"]}
            sweep["note"] = ("VBR rows other than 3.0 report the ties their own rank order produces on these inputs: on those chunks the "
                             "reference's sort_unstable order (encoder_vbr.rs:102-103) is unspecified and parity vs the Rust crate undefined")
        del scratch
        torch.cuda.empty_cache()

    # ---- e2e: the headline through the host-buffer C-ABI call.  A step = ALL n streams, as n / ne calls over the same pinned
    # buffers (bounded pinned-host footprint), H2D + D2H inside the timed region.  Control: plain copies of the same bytes.
    e2e = {"value": None, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    e2e_encode = None
    if not args.skip_e2e:
        ne = min(args.e2e_streams, n)
        while n % ne:
            ne -= 1
        while True:  # pinned host memory is a shared resource on a multi-GPU box: shrink the call size rather than fail
            try:
                h_sea = torch.empty(ne * stride, dtype=torch.uint8).pin_memory()
                h_pcm = torch.empty(ne * spp, dtype=torch.int16).pin_memory()
                break
            except RuntimeError:
                if ne <= 16:
                    raise
                ne //= 2
                while n % ne:
                    ne -= 1
        calls = n // ne
        h_sea.copy_(sea[: ne * stride])
        torch.cuda.synchronize()
        sea_off_e, sea_len_e, pcm_off_e = np.arange(ne, dtype=np.uint64) * stride, lens[:ne], np.arange(ne, dtype=np.uint64) * spp

        def e2e_step():
            for _ in range(calls):
                ctx.decode_batch_host(h_sea.data_ptr(), sea_off_e, sea_len_e, h_pcm.data_ptr(), pcm_off_e)

        ctx.decode_batch_host(h_sea.data_ptr(), sea_off_e, sea_len_e, h_pcm.data_ptr(), pcm_off_e)  # warm-up: buffers, both lanes
        dist.barrier()
        e2e_steps = max(2, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = dist.max_over_ranks(time.perf_counter() - t0) / e2e_steps
        assert np.array_equal(h_pcm[:spp].numpy(), dec0), "host-buffer decode differs from the device-resident decode"
        # control: the same byte counts as plain cudaMemcpyAsync, H2D and D2H on two streams at once, all ranks at the same time
        s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
        d_in, d_out = sea[: ne * stride], pcm_out[: ne * spp]

        def copy_step():
            for _ in range(calls):
                with torch.cuda.stream(s_up):
                    d_in.copy_(h_sea, non_blocking=True)
                with torch.cuda.stream(s_dn):
                    h_pcm.copy_(d_out, non_blocking=True)

        copy_step()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            copy_step()
        torch.cuda.synchronize()
        copy_s = dist.max_over_ranks(time.perf_counter() - t0) / e2e_steps
        e2e = {"value": W * n * spp / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(n * bound),
               "d2h_bytes_per_step": int(n * spp * 2), "ms_per_step": e2e_s * 1e3,
               "calls_per_step": calls, "streams_per_call": ne,
               "copy_ceiling_ms": copy_s * 1e3, "copy_ceiling_gbs_per_gpu": (n * bound + n * spp * 2) / copy_s / 1e9,
               "frac_of_copy_ceiling": copy_s / e2e_s,
               "control": "plain cudaMemcpyAsync of the same bytes, one H2D and one D2H stream per rank, all ranks at once: a reference "
                          "pattern, not a strict bound (with several ranks on one host fabric the pipelined call can beat it)",
               "sample": f"all {n} streams per step as {calls} calls of {ne} streams over the same pinned buffers; PCIe-bound"}
        # ---- e2e encode: sea_b200_encode_batch, host PCM in (2 B/sample), .sea out; a step = ns streams as ns / ne_e calls
        if not args.skip_encode:
            # all ns streams in one call when the host has the memory for their pinned PCM (the kernel wants every stream in
            # flight; the library pipelines slices of time, capi.cu encode_batch_sliced), else calls of ne streams
            ne_e = min(ne, ns)
            try:
                import psutil

                if ns * spp * 2 * 2 * W < psutil.virtual_memory().available // 2:
                    ne_e = ns
            except Exception:
                pass
            while ns % ne_e:
                ne_e -= 1
            if ne_e > ne:
                try:
                    del h_pcm
                    h_pcm = torch.empty(ne_e * spp, dtype=torch.int16).pin_memory()
                    h_sea = torch.empty(ne_e * stride, dtype=torch.uint8).pin_memory()
                except RuntimeError:
                    ne_e = ne
                    h_pcm = torch.empty(ne_e * spp, dtype=torch.int16).pin_memory()
            calls_e = ns // ne_e
            h_pcm[: ne_e * spp].copy_(b.pcm[: ne_e * spp])
            torch.cuda.synchronize()
            out_off_e = np.arange(ne_e, dtype=np.uint64) * stride
            pcm_off_e = np.arange(ne_e, dtype=np.uint64) * spp

            def enc_e2e_step():
                for _ in range(calls_e):
                    got_l = ctx.encode_batch_host(h_pcm.data_ptr(), pcm_off_e[:ne_e], b.nframes[:ne_e], RATE, CHANNELS, cbr3, h_sea.data_ptr(),
                                                  out_off_e)
                return got_l

            enc_e2e_step()
            dist.barrier()
            t0 = time.perf_counter()
            for _ in range(2):
                got_l = enc_e2e_step()
            enc_s = dist.max_over_ranks(time.perf_counter() - t0) / 2
            assert np.all(got_l == bound)
            assert torch.equal(h_sea[:bound], sea[:bound].cpu()), "host-buffer encode differs from the device-resident encode"
            e2e_encode = {"value": W * ns * spp / enc_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(ns * spp * 2),
                          "d2h_bytes_per_step": int(ns * bound), "ms_per_step": enc_s * 1e3, "calls_per_step": calls_e,
                          "streams_per_call": ne_e, "workload": "config-5 shape, CBR 3"}
        del h_sea, h_pcm
    del pcm_out, view
    torch.cuda.empty_cache()

    # ---- the other shapes of the reference's own tests (3 channels, scale_factor_bits 3 and 5 -- tests/test.rs:35-64) and what is
    # still left to the staged kernel (3-channel VBR), so that every cliff is on record.  1024 unique 20 s streams each, rank 0's GPU.
    other = None
    if not args.skip_encode and info.rank == 0:
        other = []
        po = torch.empty(1024 * 20 * RATE * 5, dtype=torch.int16, device=dev)
        for chs, kw, kern in ((3, dict(residual_bits=3.0), "decode_mc_kernel<3,3>"),
                              (5, dict(residual_bits=3.0), "decode_mc_kernel<5,3>"),
                              (2, dict(residual_bits=3.0, scale_factor_bits=3), "decode_unrolled_kernel<2,3,pair-repl,S=3>"),
                              (2, dict(residual_bits=3.0, scale_factor_bits=5), "decode_unrolled_kernel<2,3,plain,S=5>"),
                              (2, dict(residual_bits=3.0, scale_factor_bits=5, vbr=True), "decode_vbr_kernel<2,KF=3>"),
                              (3, dict(residual_bits=3.0, vbr=True), "decode_staged_kernel<3,0>")):
            fr_o, n_o = 20 * RATE, 1024
            bo = Batch(torch, dev, n_o, fr_o, chs)
            ctx.synth_pcm_device(bo.pcm.data_ptr(), bo.spp, (1 << 17) + np.arange(n_o, dtype=np.uint32), fr_o, chs, RATE)
            st_o = S.EncoderSettings(**kw)
            so, stride_o, lens_o, _ = encode_device(ctx, torch, dev, bo, n_o, st_o, RATE)
            _, _, _, ms_eo = encode_device(ctx, torch, dev, bo, n_o, st_o, RATE, so)
            hd = so.view(n_o, stride_o)[:, :22].cpu().numpy()
            ks = []
            for _ in range(4):
                g, ms = decode_device(ctx, so, stride_o, lens_o, hd, po, bo.spp, n_o)
                ks.append(ms)
            ms_do = float(np.mean(ks[1:]))
            other.append({"channels": chs, "settings": kw, "streams": n_o, "seconds": 20, "decode_kernel": kern,
                          "encode_msamples_per_s": n_o * bo.spp / (ms_eo * 1e-3) / 1e6,
                          "decode_msamples_per_s": n_o * bo.spp / (ms_do * 1e-3) / 1e6,
                          "decode_hbm_frac": (float(lens_o.sum()) + 2.0 * n_o * bo.spp) / (ms_do * 1e-3) / 1e9 / hbm})
            del bo, so
        del po
        torch.cuda.empty_cache()

    # ---- one-chunk streaming seam: microseconds per make_chunk / decode_chunk call, next to the CPU's per-chunk time
    latency = None
    if info.rank == 0 and W == 1 and not args.skip_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import latency_probe as LP

        latency = []
        for vbr_l in (False, True):
            row = LP.measure(ctx, CHANNELS, 40, vbr_l)
            row["cpu"] = LP.cpu_reference(CHANNELS, vbr_l)
            latency.append(row)

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only): bounded sample of the same stream shape
    cpu = None
    if info.rank == 0 and W == 1 and not args.skip_cpu:
        from oracle import sea_oracle as O

        cores = host_cores()
        reps = 4
        r = cpu_decode_baseline(cores, reps, args.seconds)
        e_secs, e_samples = O.bench("encode", cores, 1, r["pcm"], RATE, CHANNELS, r["settings"])
        cpu = {"value": r["value"], "unit": "Msamples/s", "cores": cores, "kind": r["kind"],
               "sample": f"{cores} cores x {reps} decodes of one {args.seconds} s stereo CBR-3 stream (config-4 stream shape)",
               "encode_cbr3_msamples_per_s": e_samples / e_secs / 1e6, "encode_kind": "port",
               "encode_sample": f"{cores} cores x 1 encode of the same stream (oracle restatement; no Rust toolchain)"}

    if info.rank == 0:
        print(json.dumps({
            "metric": "decode_msamples_per_s", "value": value, "unit": "Msamples/s", "n_gpus": W, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i32", "data": "synthetic", "config": workload_config(args), "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "host": host_info(), "parity": parity,
            "strong": strong, "decode_vbr3": vbr_dec, "decode_8ch_cbr4": mc_dec, "encode": encode, "e2e_encode": e2e_encode,
            "sweep": sweep, "other_shapes": other, "streaming_latency": latency,
        }))
    ctx.close()
    dist.shutdown()


def _main_with_clean_stdout():
    """stdout carries the one JSON line and nothing else: libraries that chat on fd 1 (NCCL prints its version banner there at
    the first collective) are sent to stderr for the duration of the run."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    out = sys.stdout
    sys.stdout = os.fdopen(real, "w", buffering=1)
    try:
        main()
    finally:
        sys.stdout.flush()
        sys.stdout = out


if __name__ == "__main__":
    _main_with_clean_stdout()
