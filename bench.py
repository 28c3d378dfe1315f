#!/usr/bin/env python
"""
bench.py — hours-of-audio/sec, Fbank-80 @ 16 kHz (25 ms / 10 ms, N = 512), batches of 10 s cuts.

    python bench.py --gpus N --steps K --warmup W            # the B200 path (this repository)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU extractor on the host cores

One "step" = `launches_per_step` passes of the hot path, each one fused kernel launch over a device-resident ragged batch
of `--batch` cuts; consecutive launches read DISTINCT input buffers (each far larger than L2) and the launch count is
calibrated so that a step lasts >= ~120 ms (the timed region of the default run is seconds long: clocks, power and
throttle reasons are sampled under sustained load).
  value    : whole-job hours-of-audio/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e      : the same metric through the public API (`B200Fbank.extract_batch` on numpy arrays in pinned host memory ->
             numpy features; H2D + kernel + D2H inside the timed region), >= 1 s timed
  roofline : algorithmic bytes of one launch / its mean duration (CUDA events) vs the measured HBM peak
  extra    : secondary figures with their own CUDA-event timings (MFCC 13/23, N = 400, int16 staging e2e, the reference's
             torch op chain on the same GPU, the CutSet-level sharded store of BASELINE configs[4] at bench size)
  cpu_baseline / clocks / gpu_launches : see DESIGN.md "Measurement"
Multi-GPU: one process per GPU under torchrun, cuts sharded per rank, weak scaling, no data-path collective (table broadcast
at start + a MAX-reduce of the elapsed time only).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 16000
METRIC = "hours-of-audio/sec Fbank-80@16kHz, 10s cuts"
UNIT = "h_audio/s"
BYTES_PER_FRAME = 160 * 4 + 80 * 4  # SURVEY.md §8(d): 640 B read + 320 B written per frame


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own extractor (`lhotse.features.kaldi.extractors.Fbank.extract`, extractors.py:92-115) from the
# reference tree / the oracle/_ref archive (kind "reference"); when neither exists, the oracle port of the same torch op
# chain (kind "port").  One single-threaded worker process per core, per-cut extract — the reference's fastest CPU mode
# (BASELINE.md §3).
# ------------------------------------------------------------------------------------------------
def reference_kind():
    try:
        from oracle import refimport

        return "reference" if refimport.reference_available() else "port"
    except Exception:
        return "port"


def _cpu_worker(args):
    seed, ncuts, nsamp, kind = args
    import numpy as np
    import torch

    torch.set_num_threads(1)
    rs = np.random.RandomState(seed)
    xs = [(0.1 * rs.randn(nsamp)).astype(np.float32) for _ in range(min(ncuts, 4))]
    if kind == "reference":
        from oracle import refimport

        refimport.import_reference()
        from lhotse.features.kaldi.extractors import Fbank, FbankConfig

        ext = Fbank(FbankConfig(num_mel_bins=80))
        run = lambda x: ext.extract(x, SR)  # noqa: E731
    else:
        from oracle import kaldi_oracle as O

        cfg = O.OracleConfig()
        run = lambda x: O.extract(x, cfg)  # noqa: E731
    run(xs[0])  # warm
    t0 = time.perf_counter()
    for i in range(ncuts):
        run(xs[i % len(xs)])
    return time.perf_counter() - t0


def cpu_pass(pool, procs, cuts_per_worker, nsamp, kind):
    t0 = time.perf_counter()
    times = pool.map(_cpu_worker, [(1000 + i, cuts_per_worker, nsamp, kind) for i in range(procs)])
    wall = time.perf_counter() - t0
    slowest = max(times)
    hours = procs * cuts_per_worker * nsamp / SR / 3600.0
    return hours / slowest, slowest, wall


def cpu_pool(procs):
    import multiprocessing as mp

    return mp.get_context("fork").Pool(procs)


def host_cores():
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:  # a cgroup CPU quota caps what the box can really use
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def best_cpu_procs(nsamp, kind, probe_cuts=6):
    """Picks the worker count that gives the reference its best throughput on this box: all usable cores,
    or fewer when memory bandwidth / SMT make oversubscription slower (probed on a small sample)."""
    n = host_cores()
    cands = sorted({n, max(1, n // 2), max(1, n // 4), max(1, n // 8)}, reverse=True)
    best, best_v, best_cut_s = cands[0], -1.0, 0.01
    for c in cands:
        pool = cpu_pool(c)
        try:
            cpu_pass(pool, c, 2, nsamp, kind)
            v, slowest, _ = cpu_pass(pool, c, probe_cuts, nsamp, kind)
        finally:
            pool.close()
        if v > best_v:
            best, best_v, best_cut_s = c, v, slowest / probe_cuts
    return best, best_cut_s


def bounded_cuts_per_worker(requested, cut_seconds_cpu, target_s=1.5):
    """Keeps one CPU step near `target_s` of wall time so K steps finish within minutes on any box."""
    return int(max(4, min(requested, target_s / max(cut_seconds_cpu, 1e-4))))


def cpu_what(kind):
    if kind == "reference":
        return "lhotse.features.kaldi.extractors.Fbank.extract of the UNMODIFIED reference (oracle/_ref archive or /root/reference)"
    return "oracle/kaldi_oracle.py: the reference's torch-CPU op chain (the reference package is not on this box)"


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax = float(r[2]); power.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return  # the CPU arm runs once per box
    nsamp = int(args.cut_seconds * SR)
    kind = reference_kind()
    procs, cut_s = best_cpu_procs(nsamp, kind)
    per = bounded_cuts_per_worker(args.cpu_cuts_per_worker, cut_s)
    pool = cpu_pool(procs)
    try:
        for _ in range(args.warmup):
            cpu_pass(pool, procs, max(1, per // 8), nsamp, kind)
        vals, slow = [], []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            v, s, _ = cpu_pass(pool, procs, per, nsamp, kind)
            vals.append(v); slow.append(s)
        total = time.perf_counter() - t0
    finally:
        pool.close()
    hours = args.steps * procs * per * nsamp / SR / 3600.0
    value = hours / sum(slow)
    sample = (f"{procs} procs (best of n, n/2, n/4, n/8; host has {host_cores()}) x {per} cuts x {args.cut_seconds:g}s per step, "
              f"torch 1 thread/proc, per-cut extract; {cpu_what(kind)}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * sum(slow) / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"Fbank-80 16kHz 25ms/10ms N=512, {args.cut_seconds:g}s cuts (BASELINE configs[1]) — bounded CPU sample",
                   "cuts_per_step": procs * per, "parallelism": f"{procs} cpu procs"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": total,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def _device_leg(torch, eng, xs, lens, offs, launches, steps, warm=3):
    """`steps` timed steps of `launches` launches each over the distinct input buffers `xs` (CUDA events on the current
    stream).  Returns (total ms, per-step ms list, rows per launch)."""
    meta, tot = eng.plan_batch(lens, offs)
    meta_dev = torch.from_numpy(meta).to(xs[0].device)
    outs = [torch.empty((tot.total_rows, eng.feature_dim), dtype=torch.float32, device=xs[0].device) for _ in xs]

    def step():
        for j in range(launches):
            k = j % len(xs)
            eng.extract_device(xs[k], lens, offs, out=outs[k], meta_dev=meta_dev, totals=tot)

    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[-1]), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], int(tot.total_rows), outs


def _calibrate(torch, eng, x, lens, offs, target_ms):
    """Launches per step so that a step lasts >= target_ms."""
    meta, tot = eng.plan_batch(lens, offs)
    meta_dev = torch.from_numpy(meta).to(x.device)
    out = torch.empty((tot.total_rows, eng.feature_dim), dtype=torch.float32, device=x.device)
    for _ in range(3):
        eng.extract_device(x, lens, offs, out=out, meta_dev=meta_dev, totals=tot)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(8):
        eng.extract_device(x, lens, offs, out=out, meta_dev=meta_dev, totals=tot)
    e1.record()
    torch.cuda.synchronize()
    per = e0.elapsed_time(e1) / 8
    return max(1, int(target_ms / max(per, 1e-3) + 0.999))


DUMP_BYTES_PER_ARRAY = 30_000_000  # two arrays: --dump-outputs writes at most 60 MB


def dump_outputs(dirname, arrays, seed=0):
    """Writes `name -> (cuts, T, dim)` feature arrays as DIR/<name>.npy (float32).  Where an array exceeds
    DUMP_BYTES_PER_ARRAY, a fixed seeded sample of whole cuts (ascending cut order) is written instead, so that the same
    arguments always select the same cuts."""
    import numpy as np
    import torch

    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        n = a.shape[0]
        keep = max(1, min(n, DUMP_BYTES_PER_ARRAY // (a[0].numel() * 4 if torch.is_tensor(a) else a[0].nbytes)))
        idx = np.sort(np.random.RandomState(seed).choice(n, keep, replace=False)) if keep < n else np.arange(n)
        if torch.is_tensor(a):
            a = a[torch.from_numpy(idx).to(a.device)].cpu().numpy()
        else:
            a = a[idx]
        np.save(os.path.join(dirname, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))


def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", 1))
    nsamp = int(args.cut_seconds * SR)

    # CPU baseline first (forks workers: must precede CUDA initialisation), rank 0 at N=1 only
    cpu_baseline = None
    if world == 1 and not args.skip_cpu_baseline:
        kind = reference_kind()
        procs, cut_s = best_cpu_procs(nsamp, kind)
        per = bounded_cuts_per_worker(args.cpu_cuts_per_worker, cut_s, target_s=3.0)
        pool = cpu_pool(procs)
        try:
            cpu_pass(pool, procs, max(1, per // 8), nsamp, kind)
            v, slowest, _ = cpu_pass(pool, procs, per, nsamp, kind)
        finally:
            pool.close()
        cpu_baseline = {"value": v, "unit": UNIT, "cores": procs, "kind": kind, "host_cores": host_cores(),
                        "sample": f"{procs} procs (best of n, n/2, n/4, n/8) x {per} cuts x {args.cut_seconds:g}s, {slowest:.2f}s slowest worker "
                                  f"(1 thread/proc, per-cut extract; {cpu_what(kind)})"}

    import numpy as np
    import torch

    import lhotse_b200 as lb
    from lhotse_b200 import dist as lbd
    from lhotse_b200.engine import Engine

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
    rank, world, local = lbd.init_distributed()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: keep this rank's threads and its pinned staging buffers on the GPU's own NUMA node
    numa_node = lbd.bind_host_to_gpu_numa(local)

    cfg = lb.B200FbankConfig(device=f"cuda:{local}", kernel=args.kernel)
    plan = lb.build_plan("fbank", cfg)
    lbd.broadcast_plan_tables(plan)  # NCCL broadcast of the constant tables (rank 0's bits everywhere)
    eng = Engine(plan, device=dev, kernel=args.kernel)

    B = args.batch
    torch.manual_seed(1234 + rank)
    xs = []
    for _ in range(args.buffers):  # synthetic 0.1*N(0,1) audio, generated on device; every buffer is distinct and >> L2
        x = torch.empty(B * nsamp, dtype=torch.float32, device=dev)
        for i in range(0, B, 256):
            j = min(B, i + 256)
            x[i * nsamp: j * nsamp] = 0.1 * torch.randn((j - i) * nsamp, device=dev)
        xs.append(x)
    lens = [nsamp] * B
    offs = [i * nsamp for i in range(B)]
    hours_per_launch = B * nsamp / SR / 3600.0
    NL = args.launches_per_step or _calibrate(torch, eng, xs[0], lens, offs, args.step_ms)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = eng.stats()["kernel_launches"]
    lbd.barrier()
    torch.cuda.synchronize()
    elapsed_ms, per_step_ms, frames, outs = _device_leg(torch, eng, xs, lens, offs, NL, args.steps, warm=max(args.warmup, 3))
    lbd.barrier()
    launches = eng.stats()["kernel_launches"] - launches0 - max(args.warmup, 3) * NL
    elapsed_max_ms = lbd.all_reduce_stats([elapsed_ms], "max")[0]
    value = world * hours_per_launch * NL * args.steps / (elapsed_max_ms / 1000.0)
    assert all(bool(torch.isfinite(o[:: max(1, frames // 4096)]).all()) for o in outs)  # what was timed is real output

    # ---- e2e: the public API call a lhotse user makes — FeatureExtractor.extract_batch(numpy (B, n) float32) ->
    # numpy (B, T, 80) — with the samples in pinned host memory: H2D + kernel + D2H inside the timed region
    # (the call lands in the C ABI's b200feat_extract_host, which pipelines the three over 3 streams).  One e2e step =
    # `e2e_calls` such calls over two distinct host buffers.
    Be = min(B, args.e2e_batch)
    ext = lb.B200Fbank(cfg).use_engine(eng)  # same handle / same (broadcast) tables as the device-resident leg
    hxs = []
    for k in range(2):
        t = torch.empty((Be, nsamp), dtype=torch.float32, pin_memory=True)
        t.copy_(xs[k % len(xs)][: Be * nsamp].view(Be, nsamp))
        hxs.append(t.numpy())
    for k in range(3):
        feats = ext.extract_batch(hxs[k % 2], SR)
    assert isinstance(feats, np.ndarray) and feats.shape == (Be, frames // B, eng.feature_dim)
    lbd.barrier()
    t0 = time.perf_counter()
    checksum = 0.0
    for _ in range(args.e2e_steps):
        for k in range(args.e2e_calls):
            feats = ext.extract_batch(hxs[k % 2], SR)
            checksum += float(feats[0, 0, 0])  # the result is host-resident and readable here
    e2e_s = time.perf_counter() - t0
    lbd.barrier()
    e2e_max = lbd.all_reduce_stats([e2e_s], "max")[0]
    e2e_value = world * (Be * nsamp / SR / 3600.0) * args.e2e_calls * args.e2e_steps / e2e_max
    d2h_bytes = int(feats.size) * 4 * args.e2e_calls
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # every step's first launch reads buffer 0, so outs[0] holds what the last step computed for it whatever the
        # calibrated launch count; `feats` is the last public-API call's result
        dump_outputs(args.dump_outputs, {"fbank_device": outs[0].view(B, frames // B, eng.feature_dim), "fbank_e2e": feats})

    extra = {}
    if not args.no_extra:
        extra = run_extras(args, torch, np, lb, lbd, Engine, dev, local, rank, world, xs, nsamp)

    if rank == 0:
        peak, peak_src = measured_peak()
        kern_ms = statistics.mean(per_step_ms) / NL
        achieved = frames * BYTES_PER_FRAME / (kern_ms / 1000.0) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                if tj.get("kernel") == eng.kernel and tj.get("frames"):
                    traffic = tj["dram_bytes"] * frames / tj["frames"]
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed_max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"Fbank-80 16kHz 25ms/10ms N=512 (L=400,S=160), {NL} launches x {B} x {args.cut_seconds:g}s cuts per GPU per step (BASELINE configs[1])",
                       "cuts_per_gpu_per_launch": B, "launches_per_step": NL, "frames_per_gpu_per_launch": frames, "kernel": eng.kernel,
                       "parallelism": f"dp{world} (cuts sharded per rank, no data-path collective)",
                       "l2_policy": f"{len(xs)} distinct input buffers of {B * nsamp * 4 / 2**20:.0f} MiB (+ {frames * 320 / 2**20:.0f} MiB of output each) visited round-robin: every launch's input >> 126 MiB L2",
                       "host_numa_node": numa_node},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": Be * nsamp * 4 * args.e2e_calls,
                    "d2h_bytes_per_step": d2h_bytes, "cuts_per_step": Be * args.e2e_calls, "steps": args.e2e_steps, "timed_s": e2e_max,
                    "api": "B200Fbank.extract_batch(numpy (B, n) float32 in pinned memory) -> numpy (B, T, 80); C ABI b200feat_extract_host underneath"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel_ms": kern_ms,
                         "algorithmic_bytes_per_launch": frames * BYTES_PER_FRAME,
                         "read_only_frac": frames * 640 / (kern_ms / 1000.0) / 1e9 / peak},
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


def run_extras(args, torch, np, lb, lbd, Engine, dev, local, rank, world, xs, nsamp):
    """Secondary figures, each with its own timing; never part of `value`.  Every rank runs the same legs (weak scaling),
    rank 0 reports whole-job numbers."""
    extra = {}
    B = min(args.batch, 1024)
    lens, offs = [nsamp] * B, [i * nsamp for i in range(B)]
    hours = B * nsamp / SR / 3600.0
    x2 = [x[: B * nsamp] for x in xs]

    def dev_rate(kind, cfg, key, note, sr=SR):
        try:
            hours = B * nsamp / sr / 3600.0
            plan = lb.build_plan(kind, cfg)
            e = Engine(plan, device=dev, kernel=getattr(cfg, "kernel", "auto"))
            NL = _calibrate(torch, e, x2[0], lens, offs, 60.0)
            ms, _, rows, _ = _device_leg(torch, e, x2, lens, offs, NL, 5, warm=2)
            ms = lbd.all_reduce_stats([ms], "max")[0]
            extra[key] = {"value": world * hours * NL * 5 / (ms / 1000.0), "unit": UNIT, "kernel": e.kernel, "timed_ms": ms,
                          "cuts_per_launch": B, "note": note}
            e.close()
        except Exception as ex:  # a secondary figure must never break the headline line
            extra[key] = {"error": repr(ex)}

    # int16 PCM staging through the public API (half the H2D bytes)
    try:
        ext = lb.B200Fbank(lb.B200FbankConfig(device=f"cuda:{local}"))
        Be = min(B, args.e2e_batch)
        h16 = torch.empty((Be, nsamp), dtype=torch.int16, pin_memory=True)
        h16.copy_((xs[0][: Be * nsamp].view(Be, nsamp) * 32767.0).clamp_(-32768, 32767).to(torch.int16))
        a16 = h16.numpy()
        f = None
        for _ in range(3):  # keep the previous result alive while the next call runs, as the timed loop does: both pinned
            f = ext.extract_batch(a16, SR)  # result blocks exist before the clock starts (a fresh 327 MB cudaHostAlloc costs ~150 ms)
        lbd.barrier()
        t0 = time.perf_counter()
        n = 0
        while n < 6:
            f = ext.extract_batch(a16, SR)
            n += 1
        s = lbd.all_reduce_stats([time.perf_counter() - t0], "max")[0]
        extra["int16_e2e"] = {"value": world * (Be * nsamp / SR / 3600.0) * n / s, "unit": UNIT, "timed_s": s,
                              "h2d_bytes_per_call": Be * nsamp * 2, "d2h_bytes_per_call": int(f.size) * 4,
                              "note": "B200Fbank.extract_batch(numpy int16 (B, n) in pinned memory): PCM widened inside the kernel"}
    except Exception as ex:
        extra["int16_e2e"] = {"error": repr(ex)}

    dev_rate("mfcc", lb.B200MfccConfig(num_ceps=13, num_mel_bins=23, device=f"cuda:{local}"), "mfcc_13_23",
             "BASELINE configs[2]: Mfcc(num_ceps=13, num_mel_bins=23), device-resident, CUDA events")
    dev_rate("fbank", lb.B200FbankConfig(round_to_power_of_two=False, device=f"cuda:{local}"), "n400",
             "Fbank-80 with round_to_power_of_two=False (N = L = 400), device-resident, CUDA events")
    dev_rate("fbank", lb.B200FbankConfig(sampling_rate=24000, frame_length=0.05, device=f"cuda:{local}"), "n2048_24k_50ms",
             "Fbank-80 at 24 kHz with 50 ms frames (L = 1200, N = 2048: the fast2048 kernel; the same sample buffer read as 24 kHz "
             "audio), device-resident, CUDA events", sr=24000)
    for k in ("fast", "tc"):
        if k != args.kernel:
            dev_rate("fbank", lb.B200FbankConfig(device=f"cuda:{local}", kernel=k), f"fbank80_kernel_{k}",
                     f"the headline plan on kernel={k} (what AUTO did not pick), device-resident, CUDA events")

    if rank == 0:  # the reference's own op chain on CUDA tensors of the same GPU: the 'GPU baseline to beat' (BASELINE.md §3)
        try:
            from oracle import refimport

            nb = 64
            cut_list = [xs[0][i * nsamp: (i + 1) * nsamp] for i in range(nb)]
            if refimport.reference_available():
                refimport.import_reference()
                from lhotse.features.kaldi.extractors import Fbank, FbankConfig

                ref = Fbank(FbankConfig(num_mel_bins=80, device=f"cuda:{local}"))
                run = lambda: ref.extract_batch(cut_list, SR)  # noqa: E731
                what = "lhotse Fbank(device='cuda').extract_batch(list of cuda tensors) — the unmodified reference"
            else:
                from oracle import kaldi_oracle as O

                ocfg = O.OracleConfig()
                run = lambda: [O.extract(c, ocfg) for c in cut_list]  # noqa: E731
                what = "oracle port of the reference's torch op chain on cuda tensors"
            run(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                run()
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            extra["torch_cuda_chain"] = {"value": nb * nsamp / SR / 3600.0 * 3 / (ms / 1000.0), "unit": UNIT, "timed_ms": ms, "cuts": nb,
                                         "n_gpus": 1, "note": what}
        except Exception as ex:
            extra["torch_cuda_chain"] = {"error": repr(ex)}

    if not args.no_cutset:
        try:
            from scripts.bench_config5 import run_cutset_job

            extra["config4_cutset_store"] = run_cutset_job(rank, world, local, seconds_of_audio=args.cutset_hours * 3600.0)
        except Exception as ex:
            extra["config4_cutset_store"] = {"error": repr(ex)}
        if rank == 0:
            try:
                from scripts.bench_config5 import run_onthefly_job

                extra["config3_onthefly_dataset"] = run_onthefly_job(local)
            except Exception as ex:
                extra["config3_onthefly_dataset"] = {"error": repr(ex)}
        lbd.barrier()
    return extra


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=2048, help="cuts per GPU per launch")
    ap.add_argument("--buffers", type=int, default=4, help="distinct device input buffers visited round-robin")
    ap.add_argument("--launches-per-step", type=int, default=0, help="0 = calibrate so that a step lasts --step-ms")
    ap.add_argument("--step-ms", type=float, default=120.0)
    ap.add_argument("--cut-seconds", type=float, default=10.0)
    ap.add_argument("--kernel", default="auto", choices=["auto", "fast", "tc", "generic"])
    ap.add_argument("--e2e-batch", type=int, default=1024)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-calls", type=int, default=8, help="extract_batch calls per e2e step")
    ap.add_argument("--cpu-cuts-per-worker", type=int, default=200)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cutset", action="store_true")
    ap.add_argument("--cutset-hours", type=float, default=4.0, help="hours of audio per rank in the CutSet-level job of `extra`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's features of the last step as DIR/fbank_device.npy (device-resident "
                         "leg, input buffer 0) and DIR/fbank_e2e.npy (last extract_batch call), float32 (cuts, frames, 80); a fixed "
                         "seeded sample of cuts where an array exceeds 30 MB")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
