#!/usr/bin/env python
"""bench.py — candidate-sites/sec of the Clair3 network forward on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workloads pileup,fa,fa_dwell,cascade]
                    [--dump-outputs DIR]

ONE command measures the whole metric and prints ONE JSON line.  The top-level ``value`` / ``e2e`` / ``roofline`` are the
pileup network on BASELINE.json configs[1] (the configuration the metric is quoted on); ``workloads`` carries one
sub-record per configuration:

    pileup    configs[1]  Clair3_P,  1024x33x18 int32 per step                      weak-scaled over ranks
    fa        configs[2]  Clair3_F,  256x89x33x8  int8 per step                     weak
    fa_dwell  configs[4]  Clair3_F(input_channels=9), 256x89x33x9 int8 per step     weak
    cascade   configs[3]  >= 1 M pileup sites then >= 100 k full-alignment sites (the ~10:1 ratio of
              run_clair3.py:303-313), fed from pinned HOST memory, split into N contiguous site ranges
              (clair3/CallVariantsFromCffiGPU.py:141-156)                            STRONG-scaled over ranks
    pileup_counts  SURVEY.md 8f row N4: the pileup feature counter (calculate_clair3_pileup, src/clair3_pileup.c:142-476) on
              decoded alignment records, aligned bases/s (its own metric; HBM-bound integer work)          weak

A *step* is one forward of the hot path over one synthetic candidate-site batch (for ``cascade``: one pass over all its
sites).  Every timed region is exactly K steps (``timed_region_s``; ``ms_per_step`` = region / K); W warm-up steps precede
it.  A small K times pipeline fill and drain as much as the steady state: pass a K whose region lasts seconds for a rate.
Steps go round-robin over a few CUDA streams of ONE model (each stream owns an activation workspace); device-resident
inputs are rotated over > 126 MB of distinct batches so no step re-reads its input from L2; regions are bracketed by
barrier + synchronize, timed with CUDA events, max over ranks; ``nvidia-smi`` clocks are sampled every 100 ms DURING each
region.  ``e2e`` is the same metric through the module API with pinned HOST input and HOST output (H2D and D2H inside the
timed region): pipelined (``forward_async`` over the streams), through the ``predict_stream`` helper, and synchronous per
step (the reference's ``_torch_predict`` shape).

N > 1: one process per GPU (torchrun), one NCCL broadcast of the packed weight images from rank 0 before timing
(``c3b_bcast_weights``), no data-path collective.

``--impl reference`` times the reference's own CPU implementation of the same steps (torch CPU ops, all host threads)
through ``oracle/torch_port.py`` (the Python reference cannot travel to the GPU box; see DESIGN.md).

``--dump-outputs DIR`` writes, after the timed regions, what the last timed step of each workload returned to its caller as
``DIR/<workload>[_<array>].npy`` (float32 probabilities; integer counts as float64, exact), so that two builds run with the
same arguments - hence the same seeded inputs - can be compared output for output.  Outputs larger than a few MB are a fixed,
seeded sample of rows (``*_rows.npy`` holds the row indices); the whole dump stays under 64 MB.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the tree may be read-only: neither this process nor its CPU-baseline workers write bytecode caches into it
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

from clair3_b200 import synth  # noqa: E402

DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE_ROWS = 65536

# algorithmic FLOPs per site (SURVEY.md 8d) and per tensor-core kernel (2*M*N*K of the layer shapes, clair3/model.py:96-110, 317-344)
WORKLOADS = {
    "pileup": dict(kind="pileup", batch=1024, channels=18, depth=0, add_indel=False, flop=47_785_984, scaling="weak",
                   cfg="Pileup net forward, synthetic batch 1024x33x18 int32 per step (BASELINE configs[1])"),
    "fa": dict(kind="fa", batch=256, channels=8, depth=89, add_indel=True, flop=451_538_432, scaling="weak",
               cfg="Full-alignment net forward, synthetic batch 256x89x33x8 int8 per step (BASELINE configs[2])"),
    "fa_dwell": dict(kind="fa", batch=256, channels=9, depth=89, add_indel=True, flop=452_419_712, scaling="weak",
                     cfg="Dwell-time full-alignment net (--enable_dwell_time, input_channels=9), synthetic batch 256x89x33x9 int8 per "
                         "step (BASELINE configs[4])"),
}
CASCADE_PILEUP_SITES = 1024 * 1024
CASCADE_FA_SITES = 410 * 256          # 104,960: the ~10:1 ratio implied by var_pct_full / ref_pct_full (run_clair3.py:303-313)
CASCADE_CFG = ("Pileup+FA cascade, %d pileup sites then %d full-alignment sites from pinned host memory, contiguous site ranges "
               "per rank (BASELINE configs[3])" % (CASCADE_PILEUP_SITES, CASCADE_FA_SITES))


def kernel_flops(w):
    if w["kind"] == "pileup":
        return {"lstm1": 33 * 2 * 2 * 512 * (18 + 128), "proj2": 33 * 2 * 2 * 640 * 256, "lstm2": 33 * 2 * 2 * 640 * 160,
                "l4": 2 * 10560 * 128, "tail": 2 * 10560 * 128 + 2 * 128 * 128 * 2 + 2 * 128 * 24}
    c = w["channels"]
    return {"conv0": 2 * 45 * 17 * 64 * 9 * c, "conv1": 2 * 45 * 17 * 64 * 576, "conv2": 2 * 45 * 17 * 64 * 576,
            "conv3": 2 * 23 * 9 * 128 * 576, "conv4": 2 * 23 * 9 * 128 * 1152, "conv5": 2 * 23 * 9 * 128 * 1152,
            "conv6": 2 * 12 * 5 * 256 * 1152, "conv7": 2 * 12 * 5 * 256 * 2304, "conv8": 2 * 12 * 5 * 256 * 2304,
            "l4": 2 * 3584 * 256, "tail": 2 * 3584 * 256 + 2 * 256 * 128 * 4 + 2 * 128 * 90}


ALL_KERNEL_NAMES = ["ingest", "lstm1", "proj2", "lstm2", "l4", "heads", "tail", "spp"] + ["conv%d" % i for i in range(9)]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm": d["hbm_gbs"], "which": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "which": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING a timed region (100 ms period)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.lock = threading.Lock()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()                       # the first sample takes a few hundred ms: wait for it so that the
            while not self.lines and time.time() - t0 < 3.0:      # region below is sampled from its first 100 ms on
                time.sleep(0.02)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            with self.lock:
                self.lines.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def window(self, t0, t1):
        """Summary of the samples taken in [t0, t1] (host clock)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        with self.lock:
            lines = [l for (t, l) in self.lines if t0 <= t <= t1 + 0.05]
        sm, mx, pw, reasons = [], [], [], set()
        for l in lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_mhz_min": min(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()


def state_dict_for(w, seed=0):
    if w["kind"] == "pileup":
        return synth.pileup_state_dict(w["add_indel"], seed=seed)
    return synth.fa_state_dict(w["add_indel"], channels=w["channels"], seed=seed)


def make_model(w, device, load_real_weights):
    from clair3_b200.model import Clair3_F, Clair3_P
    sd = state_dict_for(w)
    cls = Clair3_P if w["kind"] == "pileup" else Clair3_F
    m = cls(add_indel_length=w["add_indel"], predict=True, input_channels=w["channels"])
    if not load_real_weights:      # non-root ranks start from zeros and receive the packed images by broadcast
        sd = {k: np.zeros_like(v) for k, v in sd.items()}
    m.to(device)
    m.eval()
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    return m


def make_inputs(w, n_batches, seed, batch=None):
    b = batch or w["batch"]
    if w["kind"] == "pileup":
        return [synth.pileup_inputs(b, seed=seed + i) for i in range(n_batches)]
    base = [synth.fa_inputs(b, depth=w["depth"], channels=w["channels"], seed=seed + i) for i in range(min(n_batches, 4))]
    return [np.roll(base[i % len(base)], i // len(base) + 1, axis=0) for i in range(n_batches)]   # cheap distinct batches


def site_bytes(w):
    return 33 * 18 * 4 if w["kind"] == "pileup" else w["depth"] * 33 * w["channels"]


# ------------------------------------------------------------------------------------------------------- CPU reference legs
def cpu_port(w, sd):
    from oracle import torch_port          # cpu_baseline / reference arm only
    if w["kind"] == "pileup":
        return torch_port.PileupPort(sd, w["add_indel"])
    return torch_port.FullAlignmentPort(sd, w["add_indel"])


def best_cpu_threads(port, x, ncores):
    """The reference lets torch pick its thread count (CallVariantsFromCffi.py:56-63 sets it from --threads); oneDNN's
    LSTM/conv primitives do not scale to every core of a large host, so probe a few counts and keep the fastest."""
    best, best_t = ncores, None
    for n in sorted({c for c in (8, 16, 32, 64, ncores) if c <= ncores}):
        torch.set_num_threads(n)
        port(x)
        t0 = time.perf_counter()
        port(x)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def time_cpu(w, budget_s, threads, min_iters=2):
    port = cpu_port(w, state_dict_for(w))
    xs = make_inputs(w, 2, seed=900)
    threads = best_cpu_threads(port, xs[0], threads)
    port(xs[0])                            # warm-up
    t0 = time.perf_counter()
    iters = 0
    while iters < min_iters or (time.perf_counter() - t0 < budget_s and iters < 64):
        port(xs[iters % 2])
        iters += 1
    dt = time.perf_counter() - t0
    return w["batch"] * iters / dt, iters, dt, threads


def cpu_deployment_shape(wname, ncores, seconds=6.0, steps=0):
    """The reference's own CPU deployment: many single-threaded worker processes (`--threads N` -> N*3/4 callers with
    torch.set_num_threads(1), scripts/clair3_c_impl.sh + CallVariantsFromCffi.py:56-63).  Runs min(3/4 cores, 64) processes of
    the oracle port concurrently - for `seconds` each, or (steps > 0) exactly `steps` calls sized to take about `seconds` - and
    sums their rates."""
    nproc = max(1, min(ncores * 3 // 4, 64))
    sites = 64 if wname == "pileup" else 8
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
    cmd = [sys.executable, "-m", "oracle.torch_port", wname, str(seconds), str(sites)] + ([str(steps)] if steps > 0 else [])
    procs = [subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
             for _ in range(nproc)]
    total, ok, per_call, secs = 0.0, 0, 0, 0.0
    for p in procs:
        try:
            out, _ = p.communicate(timeout=seconds * 10 + 180)
            r = json.loads(out.strip().splitlines()[-1])
            total += r["sites"] / r["seconds"]
            per_call = r["sites_per_call"]
            secs = max(secs, r["seconds"])
            ok += 1
        except Exception:
            p.kill()
    return {"value": total, "unit": "sites/s", "processes": ok, "threads_each": 1, "seconds": secs,
            "sample": "%d single-thread processes, %s of ~%d-site calls each, rates summed"
                      % (ok, ("%d calls" % steps) if steps > 0 else ("%.0f s" % seconds), per_call)}


def cpu_baseline_for(wname, budget_s, dep_seconds):
    """Bounded sample of the workload on the host cores: the stronger of one multi-threaded process and the reference's
    many-single-thread-workers deployment."""
    w = WORKLOADS[wname]
    ncores = len(os.sched_getaffinity(0))
    v, iters, dt, threads = time_cpu(w, budget_s, ncores)
    cpu = {"value": v, "unit": "sites/s", "cores": threads, "kind": "port",
           "sample": "%d steps of %d sites in %.1f s; torch CPU ops of the reference forward (oracle/torch_port.py), fastest of "
                     "{8,16,32,64,all=%d} threads" % (iters, w["batch"], dt, ncores),
           "single_process": {"value": v, "cores": threads}}
    if dep_seconds > 0:
        dep = cpu_deployment_shape(wname, ncores, seconds=dep_seconds)
        cpu["deployment_shape"] = dep
        if dep["value"] > v:
            cpu["value"], cpu["cores"] = dep["value"], dep["processes"]
            cpu["sample"] = dep["sample"] + " (the reference's --threads deployment; beats one multi-threaded process)"
    return cpu


def config_of(wname):
    """Workload-defining keys only: identical in the b200 and the reference arm."""
    cfg = CASCADE_CFG if wname == "cascade" else WORKLOADS[wname]["cfg"]
    return {"workload": cfg, "batch_per_step": 1024 if wname == "cascade" else WORKLOADS[wname]["batch"],
            "weights": "seeded synthetic checkpoint (clair3_b200.synth), random-init of the reference architecture",
            "parallelism": "site-sharded, one process per GPU"}


def run_reference_arm(args, rank, world):
    """The reference's CPU path on this box's host cores (rank 0 only under torchrun)."""
    if rank != 0:
        return
    ncores = len(os.sched_getaffinity(0))
    subs = {}
    for wname in [n for n in args.workloads if n in ("pileup", "fa")]:
        w = WORKLOADS[wname]
        port = cpu_port(w, state_dict_for(w))
        xs = make_inputs(w, 2, seed=900)
        threads = best_cpu_threads(port, xs[0], ncores)
        for i in range(args.warmup):
            port(xs[i % 2])
        # a "step" is a bounded sample of the workload's batch: the K-step run of each workload ends within ~1 minute
        t0 = time.perf_counter()
        port(xs[0])
        t1 = time.perf_counter() - t0
        n_sites = w["batch"]
        budget = 60.0
        if args.steps * t1 > budget:
            n_sites = max(16, int(w["batch"] * budget / (args.steps * t1)) // 16 * 16)
            xs = [x[:n_sites] for x in xs]
            port(xs[0])
        t0 = time.perf_counter()
        for i in range(args.steps):
            port(xs[i % 2])
        dt = time.perf_counter() - t0
        val = n_sites * args.steps / dt
        single = {"value": val, "cores": threads, "sample": "%d steps of %d sites in one process" % (args.steps, n_sites)}
        dep = cpu_deployment_shape(wname, ncores, seconds=15.0, steps=args.steps)
        cores, ms_step = threads, dt / args.steps * 1e3
        sample = "%d steps of %d sites, torch CPU ops of the reference forward (oracle/torch_port.py)" % (args.steps, n_sites)
        if dep["value"] > val:            # all the host threads the reference can use: its many-single-thread-workers deployment
            val, cores = dep["value"], dep["processes"]
            sample = dep["sample"] + ", torch CPU ops of the reference forward (oracle/torch_port.py)"
            ms_step = dep["seconds"] / args.steps * 1e3
        subs[wname] = {"value": val, "unit": "sites/s", "ms_per_step": ms_step, "config": config_of(wname),
                       "cpu_baseline": {"value": val, "unit": "sites/s", "cores": cores, "kind": "port", "sample": sample,
                                        "single_process": single, "deployment_shape": dep}}
    if "pileup" in subs and "fa" in subs:
        t = CASCADE_PILEUP_SITES / subs["pileup"]["value"] + CASCADE_FA_SITES / subs["fa"]["value"]
        subs["cascade"] = {"value": (CASCADE_PILEUP_SITES + CASCADE_FA_SITES) / t, "unit": "sites/s", "config": config_of("cascade"),
                           "derived": "sites / (pileup sites / pileup rate + full-alignment sites / full-alignment rate) from the two "
                                      "measured CPU rates above (running 1.15 M sites through the CPU path would take minutes)"}
    head = subs.get("pileup") or next(iter(subs.values()))
    head_name = "pileup" if "pileup" in subs else next(iter(subs))
    line = {
        "impl": "reference", "metric": "candidate-sites/sec", "value": head["value"], "unit": "sites/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(head_name),
        "cpu_baseline": head["cpu_baseline"],
        "e2e": {"value": head["value"], "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "workloads": subs,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------- B200 arm
class Ctx:
    def __init__(self, args, rank, world, device, sampler):
        self.args, self.rank, self.world, self.device, self.sampler = args, rank, world, device, sampler
        self.streams = [torch.cuda.Stream(device) for _ in range(max(1, args.streams))]
        self.main = torch.cuda.current_stream(device)
        self.dump = {} if args.dump_outputs and rank == 0 else None     # name -> the last timed step's output (host array)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(self.device)

    def max_over_ranks(self, vals):
        if self.world == 1:
            return list(vals)
        import torch.distributed as dist
        t = torch.tensor(list(vals), device=self.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def timed(self, issue, total_calls):
        """barrier+sync, CUDA-event bracket around `issue(total_calls)` fanned over the streams, barrier+sync; returns
        (elapsed ms max over ranks, clocks summary of the region)."""
        self.barrier()
        t0 = self.sampler.mark() if self.sampler else 0
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(self.main)
        for st in self.streams:
            st.wait_event(start)
        issue(total_calls)
        for st in self.streams:
            ev = torch.cuda.Event()
            ev.record(st)
            self.main.wait_event(ev)
        end.record(self.main)
        torch.cuda.synchronize(self.device)
        t1 = self.sampler.mark() if self.sampler else 0
        ms = start.elapsed_time(end)
        clocks = self.sampler.window(t0, t1) if self.sampler else None
        ms = self.max_over_ranks([ms])[0]
        self.barrier()
        return ms, clocks


def sample_rows(n, seed=0):
    """Indices of a fixed, seeded, sorted sample of DUMP_SAMPLE_ROWS of n rows (all rows when n is not larger)."""
    if n <= DUMP_SAMPLE_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, DUMP_SAMPLE_ROWS, replace=False))


def dump_outputs(dirname, arrays):
    """Write name -> array as DIR/<name>.npy: floating outputs as float32, integer ones as float64 (exact below 2**53)."""
    out = {k: np.ascontiguousarray(a, dtype=np.float32 if a.dtype.kind == "f" else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(dirname, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(dirname, k + ".npy"), a)


def parity_spot_check(model, w, x):
    from oracle import clair3_oracle as orc                           # checker only
    sd = state_dict_for(w)
    chk = x[:8]
    ref = orc.pileup_forward(sd, chk, w["add_indel"]) if w["kind"] == "pileup" else orc.fa_forward(sd, chk, w["add_indel"])
    got = model(torch.from_numpy(chk).to(model._device)).cpu().numpy()
    parity = float(np.abs(got - ref).max())
    if not (parity < 2e-2):
        raise SystemExit("parity check failed before timing: max |dp| = %g" % parity)
    return parity


def profile_kernels(ctx, model, w, xs_dev, value, clocks):
    """Per-kernel device time (single stream, CUDA events around every launch inside the library) -> kernels, roofline."""
    from clair3_b200._ffi import check, ffi, lib
    pk = peaks()
    b = w["batch"]
    kflops = kernel_flops(w)
    model.set_option("profile", 1)
    for i in range(40):
        model(xs_dev[i % len(xs_dev)])
    torch.cuda.synchronize(ctx.device)
    kernels, tot, tot_sm = {}, 0.0, 0.0
    n_sm = torch.cuda.get_device_properties(ctx.device).multi_processor_count
    for nme in ALL_KERNEL_NAMES:
        pms, pn, pc = ffi.new("double *"), ffi.new("int64_t *"), ffi.new("double *")
        check(lib().c3b_get_profile(model._handle, nme.encode(), pms, pn))
        if pn[0]:
            check(lib().c3b_get_profile_ctas(model._handle, nme.encode(), pc))
            kernels[nme] = {"ms_per_launch": pms[0] / pn[0], "launches": int(pn[0]), "ctas": pc[0]}
            tot += pms[0] / pn[0]
    model.set_option("profile", 0)
    for nme, k in kernels.items():
        k["share"] = k["ms_per_launch"] / tot
        # SM-time: what the launch costs when several batches share the GPU (tensor-core kernels hold one SM per CTA; the small
        # CUDA-core kernels - ingest, spp - co-reside with them, their grid is capped at the SM count here)
        k["sm_time_ms"] = k["ms_per_launch"] * min(k["ctas"], n_sm)
        tot_sm += k["sm_time_ms"]
        fl = kflops.get(nme)
        if fl:
            k["tflops"] = fl * b / (k["ms_per_launch"] * 1e-3) / 1e12
            k["frac_of_bf16_burst"] = k["tflops"] / pk["bf16_burst"]
            k["frac_of_occupied_sms"] = k["tflops"] / (pk["bf16_burst"] * min(k["ctas"], n_sm) / n_sm)
    for k in kernels.values():
        k["sm_time_share"] = k["sm_time_ms"] / tot_sm
    # dominant = the tensor-core kernel with the largest SM-time (a 2-CTA launch with a long latency does not bound throughput)
    dom = max((n for n in kernels if n in kflops), key=lambda n: kernels[n]["sm_time_ms"])
    # DRAM bytes per launch from the committed ncu capture (profiles/traffic.json, written by tools/ncu_summary.py from
    # `ncu --set full`: dram__bytes_read.sum + dram__bytes_write.sum), if it was taken at this workload's batch size
    traffic, traffic_all = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        tw = tj.get("fa" if w["kind"] == "fa" else "pileup", {})
        ent = tw.get(dom)
        if ent and ent.get("batch") == b:
            traffic = ent["dram_bytes_per_launch"]
        if all(tw.get(n, {}).get("batch") == b for n in kernels if n in tw):
            traffic_all = sum(tw[n]["dram_bytes_per_launch"] for n in kernels if n in tw) or None
    except (OSError, ValueError):
        pass
    whole = w["flop"] * value / ctx.world / 1e12
    roofline = {"bound": "tensor", "kernel": dom, "achieved": kernels[dom]["tflops"], "peak": pk["bf16_burst"],
                "unit": "TFLOP/s", "frac": kernels[dom]["tflops"] / pk["bf16_burst"], "traffic": traffic,
                "peak_source": pk["which"] + ", burst figure (kernel timed alone between CUDA events)",
                "flop_per_launch": kflops[dom] * b, "ctas": kernels[dom]["ctas"], "frac_of_occupied_sms": kernels[dom]["frac_of_occupied_sms"],
                "dominant_by": "SM-time (CTAs x duration; share %.2f of the step's SM-time)" % kernels[dom]["sm_time_share"],
                "sm_time_ms_per_step": tot_sm,
                "whole_step": {"achieved": whole, "frac_of_sustained": whole / pk["bf16_sustained"], "frac_of_burst": whole / pk["bf16_burst"],
                               "dram_bytes_per_step_all_kernels": traffic_all,
                               "compulsory_bytes_per_step": b * (site_bytes(w) + model.out_dim * 4)}}
    if dom in ("lstm1", "lstm2"):
        # The recurrent kernels are not tensor-bound: their epilogue needs 5 tanh evaluations per (site, step, direction, unit)
        # and the SFU pipe delivers 16 per clock and SM (tanh.approx.f32: 16 lanes/clk; the packed f16x2 form: two results per
        # lane at half the issue rate - measured, no net gain).  One launch occupies `ctas` SMs, so the honest ceiling for THIS
        # launch is those SMs' SFU rate; the other SMs are filled by the other streams.
        units = 128 if dom == "lstm1" else 160
        ctas = int(kernels[dom]["ctas"])
        mufu = 5.0 * 33 * 2 * units * b
        clk_hz = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
        per_clk_sm = mufu / (kernels[dom]["ms_per_launch"] * 1e-3 * clk_hz) / ctas
        roofline["limiter"] = {"resource": "SFU (MUFU.TANH) issue, 16 lanes/clk/SM", "mufu_ops_per_launch": mufu, "ctas": ctas,
                               "achieved_per_clk_per_sm": per_clk_sm, "peak_per_clk_per_sm": 16.0, "frac": per_clk_sm / 16.0}
    return kernels, roofline


def run_forward_workload(ctx, wname, model):
    """Weak-scaled single-network workload: device-resident value, host-fed e2e (three call shapes), kernels + roofline."""
    args, w = ctx.args, WORKLOADS[wname]
    b, n_streams, dev = w["batch"], len(ctx.streams), ctx.device
    in_bytes = b * site_bytes(w)
    pool = max(8, int(140e6 // in_bytes) + 1)
    xs_host = make_inputs(w, pool, seed=100 + 1000 * ctx.rank)        # every rank gets its own sites (weak scaling)
    xs_dev = [torch.from_numpy(x).to(dev) for x in xs_host]
    ys_dev = [torch.empty((b, model.out_dim), dtype=torch.float32, device=dev) for _ in range(2 * n_streams)]
    parity = parity_spot_check(model, w, xs_host[0])                  # the bench never times a wrong kernel
    K = args.steps

    counter = [0]

    def issue_dev(n):
        k = counter[0]
        for i in range(n):
            st = ctx.streams[(k + i) % n_streams]
            with torch.cuda.stream(st):
                model.forward_into(xs_dev[(k + i) % pool], ys_dev[(k + i) % len(ys_dev)])
        counter[0] = k + n

    issue_dev(2 * n_streams)                                          # every stream's workspace exists (allocation, not warm-up)
    torch.cuda.synchronize(dev)
    issue_dev(args.warmup)                                            # W warm-up steps
    launches0 = model.launch_count
    ms, clocks = ctx.timed(issue_dev, K)
    launches = model.launch_count - launches0
    if ctx.dump is not None:
        ctx.dump[wname] = ys_dev[(counter[0] - 1) % len(ys_dev)].cpu().numpy()
    value = b * K * ctx.world / (ms * 1e-3)
    rec = {"value": value, "unit": "sites/s", "scaling": "weak", "steps": K,
           "timed_region_s": ms * 1e-3, "ms_per_step": ms / K, "clocks": clocks,
           "gpu_launches": int(launches), "parity_max_abs_dp": parity, "config": config_of(wname),
           "run": {"streams_in_flight": n_streams, "lstm_subtile_sites": (args.lstm_tile or "auto (64 stream-ordered / 16 synchronous)") if w["kind"] == "pileup" else None,
                   "l2_policy": "inputs rotated over %d distinct device-resident batches (> 126 MB L2)" % pool}}

    # ---- e2e: pinned host tensors in and out through the module API, H2D and D2H inside the timed region
    xs_pin = [torch.from_numpy(x).pin_memory() for x in xs_host[:max(8, n_streams)]]
    ys_pin = [torch.empty((b, model.out_dim), dtype=torch.float32).pin_memory() for _ in range(n_streams)]
    ecount = [0]

    def issue_e2e(n):
        k = ecount[0]
        for i in range(n):
            st = ctx.streams[(k + i) % n_streams]
            with torch.cuda.stream(st):
                model.forward_async(xs_pin[(k + i) % len(xs_pin)], ys_pin[(k + i) % n_streams])
        ecount[0] = k + n

    issue_e2e(2 * n_streams)
    torch.cuda.synchronize(dev)
    e2e_ms, e2e_clocks = ctx.timed(issue_e2e, K)
    last = (ecount[0] - 1)
    ref_y = model(xs_pin[last % len(xs_pin)])                         # the last pipelined result must equal a sync call
    assert float((ref_y - ys_pin[last % n_streams]).abs().max()) < 1e-4
    e2e_value = b * K * ctx.world / (e2e_ms * 1e-3)

    # (b) the predict_stream helper (what a `_torch_predict`-shaped caller switches to)
    def run_stream(n):
        it = (xs_pin[i % len(xs_pin)] for i in range(n))
        cnt = 0
        for y in model.predict_stream(it, streams=n_streams):
            cnt += len(y)
        return cnt
    run_stream(2 * n_streams)
    ctx.barrier()
    t0 = time.perf_counter()
    run_stream(K)
    torch.cuda.synchronize(dev)
    ps_ms = ctx.max_over_ranks([(time.perf_counter() - t0) * 1e3])[0]

    # (c) synchronous per step: y = model(x_pinned), exactly the shape of the reference's _torch_predict
    for i in range(3):
        model(xs_pin[i % len(xs_pin)])
    torch.cuda.synchronize(dev)
    ctx.barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for i in range(K):
        y_host = model(xs_pin[i % len(xs_pin)])
    s1.record()
    torch.cuda.synchronize(dev)
    assert y_host.device.type == "cpu"
    sync_ms = ctx.max_over_ranks([s0.elapsed_time(s1)])[0]
    # (d) pileup only: the window hand-off of c3b_forward_windows - libclair3's per-column count matrix (int64, plp_data.matrix)
    # plus one window start per candidate go over PCIe instead of one [33,18] tensor per candidate; candidates every 4th column
    win = None
    if w["kind"] == "pileup":
        stride_cols = 4
        n_cols = b * stride_cols + 33
        cols_pin = [torch.from_numpy(np.ascontiguousarray(np.resize(x.reshape(-1, 18), (n_cols, 18)).astype(np.int64))).pin_memory()
                    for x in xs_host[:n_streams]]
        starts_pin = torch.arange(0, b * stride_cols, stride_cols, dtype=torch.int64).pin_memory()
        wcount = [0]

        def issue_win(n):
            k = wcount[0]
            for i in range(n):
                st = ctx.streams[(k + i) % n_streams]
                with torch.cuda.stream(st):
                    model.forward_windows(cols_pin[(k + i) % len(cols_pin)], starts_pin, ys_pin[(k + i) % n_streams], sync=False)
            wcount[0] = k + n

        issue_win(2 * n_streams)
        torch.cuda.synchronize(dev)
        win_ms, _ = ctx.timed(issue_win, K)
        win = {"value": b * K * ctx.world / (win_ms * 1e-3), "unit": "sites/s", "steps": K,
               "timed_region_s": win_ms * 1e-3, "h2d_bytes_per_step": n_cols * 18 * 8 + b * 8,
               "mode": "Clair3_P.forward_windows(pinned int64 column matrix [%d,18], pinned window starts) pipelined over %d streams: "
                       "the 33-row windows are gathered on the GPU (candidates every %dth column)" % (n_cols, n_streams, stride_cols)}
    kind = "P" if w["kind"] == "pileup" else "F"
    rec["e2e"] = {"value": e2e_value, "unit": "sites/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": b * model.out_dim * 4,
                  "steps": K, "timed_region_s": e2e_ms * 1e-3, "clocks": e2e_clocks,
                  "mode": "Clair3_%s.forward_async(pinned host x, pinned host y) pipelined over %d streams (H2D + kernels + D2H "
                          "stream-ordered per step, one synchronise at the end)" % (kind, n_streams),
                  "predict_stream": {"value": b * K * ctx.world / (ps_ms * 1e-3), "unit": "sites/s", "steps": K,
                                     "mode": "for Y in model.predict_stream(batches): in-order numpy results, %d batches in flight "
                                             "(host wall clock, includes the per-batch result copy)" % n_streams},
                  "synchronous_per_step": {"value": b * K * ctx.world / (sync_ms * 1e-3), "unit": "sites/s", "steps": K,
                                           "mode": "y = model(x_pinned): H2D, forward, D2H, stream sync every step (the _torch_predict shape)"}}
    if win:
        rec["e2e"]["forward_windows"] = win
    if ctx.rank == 0:
        rec["kernels"], rec["roofline"] = profile_kernels(ctx, model, w, xs_dev, value, clocks)
    del xs_dev, ys_dev
    torch.cuda.empty_cache()
    return rec


def run_cascade(ctx, model_p, model_f):
    """BASELINE configs[3]: >= 1 M pileup sites, then >= 100 k full-alignment sites, host-fed, STRONG-scaled: rank r serves the
    contiguous site range site_range(total, r, N) of each phase (clair3/CallVariantsFromCffiGPU.py:141-156 builds the same
    contiguous per-GPU lists).  Sites are drawn cyclically from pinned pools of distinct batches (> L2 in aggregate)."""
    from clair3_b200 import sharding
    args, dev, n_streams = ctx.args, ctx.device, len(ctx.streams)
    wp, wf = WORKLOADS["pileup"], WORKLOADS["fa"]
    pool_p = [torch.from_numpy(x).pin_memory() for x in make_inputs(wp, 64, seed=5000 + 977 * ctx.rank)]      # 156 MB
    pool_f = [torch.from_numpy(x).pin_memory() for x in make_inputs(wf, 24, seed=6000 + 977 * ctx.rank)]      # 144 MB
    lo_p, hi_p = sharding.site_range(CASCADE_PILEUP_SITES, ctx.rank, ctx.world)
    lo_f, hi_f = sharding.site_range(CASCADE_FA_SITES, ctx.rank, ctx.world)
    # one pinned row per site of the rank's range: a pass leaves every result of the pass for its caller
    yp = torch.empty((hi_p - lo_p, model_p.out_dim), dtype=torch.float32).pin_memory()
    yf = torch.empty((hi_f - lo_f, model_f.out_dim), dtype=torch.float32).pin_memory()

    def batches(lo, hi, b):
        out = []
        s = lo
        while s < hi:
            out.append(min(b, hi - s))
            s += b
        return out
    bp_list, bf_list = batches(lo_p, hi_p, wp["batch"]), batches(lo_f, hi_f, wf["batch"])

    def one_pass():
        for i, n in enumerate(bp_list):
            st = ctx.streams[i % n_streams]
            with torch.cuda.stream(st):
                model_p.forward_async(pool_p[i % len(pool_p)][:n], yp[i * wp["batch"]:i * wp["batch"] + n])
        # phase boundary: full-alignment candidates come out of the pileup calls, so the second phase starts after the first
        evs = []
        for st in ctx.streams:
            ev = torch.cuda.Event()
            ev.record(st)
            evs.append(ev)
        for st in ctx.streams:
            for ev in evs:
                st.wait_event(ev)
        for i, n in enumerate(bf_list):
            st = ctx.streams[i % n_streams]
            with torch.cuda.stream(st):
                model_f.forward_async(pool_f[i % len(pool_f)][:n], yf[i * wf["batch"]:i * wf["batch"] + n])

    def issue(passes):
        for _ in range(passes):
            one_pass()

    issue(args.warmup)             # warm-up passes (workspaces, pinned pages)
    torch.cuda.synchronize(dev)
    passes = args.steps
    ms, clocks = ctx.timed(issue, passes)
    if ctx.dump is not None:
        rp, rf = sample_rows(len(yp)), sample_rows(len(yf))
        ctx.dump.update({"cascade_pileup": yp.numpy()[rp], "cascade_pileup_rows": rp,
                         "cascade_full_alignment": yf.numpy()[rf], "cascade_full_alignment_rows": rf})
    total = CASCADE_PILEUP_SITES + CASCADE_FA_SITES
    value = total * passes / (ms * 1e-3)
    h2d = (hi_p - lo_p) * site_bytes(wp) + (hi_f - lo_f) * site_bytes(wf)
    d2h = (hi_p - lo_p) * model_p.out_dim * 4 + (hi_f - lo_f) * model_f.out_dim * 4
    rec = {"value": value, "unit": "sites/s", "scaling": "strong", "passes": passes, "steps": passes,
           "calls_per_pass": len(bp_list) + len(bf_list), "timed_region_s": ms * 1e-3, "ms_per_pass": ms / passes, "clocks": clocks,
           "sites_per_pass": {"pileup": CASCADE_PILEUP_SITES, "full_alignment": CASCADE_FA_SITES},
           "rank0_range": {"pileup": [lo_p, hi_p], "full_alignment": [lo_f, hi_f]} if ctx.rank == 0 else None,
           "config": config_of("cascade"),
           "e2e": {"value": value, "unit": "sites/s", "h2d_bytes_per_pass_per_rank": h2d, "d2h_bytes_per_pass_per_rank": d2h,
                   "mode": "forward_async from pinned host pools over %d streams, pileup phase then full-alignment phase, one "
                           "synchronise per region; host-fed by definition, so value == e2e" % n_streams},
           "run": {"streams_in_flight": n_streams, "pool": "pileup %d x 1024 + full-alignment %d x 256 distinct pinned batches per rank, "
                                                            "cycled" % (len(pool_p), len(pool_f))}}
    return rec



# ------------------------------------------------------------------------------------------------------- pileup feature counting
PLP_CFG = dict(region=1 << 20, depth=40, read_len=8000, indel_rate=0.04, origin=10000, seed=5)


def run_pileup_counts(ctx):
    """SURVEY.md 8f row N4 (pileup half): calculate_clair3_pileup (src/clair3_pileup.c:142-476) on the GPU from decoded alignment
    records.  A step = one c3b_plp_count over one synthetic region; value = device-resident records, e2e = pinned host records
    in, count matrix / candidates out (H2D + 8 kernels + D2H inside the region).  Unit: aligned bases/s, a base = one
    (read, covered column) pair that the reference's inner loop visits (sum of the per-column depths)."""
    from clair3_b200 import pileup_counts as pc, synth_reads as sr
    from oracle import pileup_oracle as po      # checker + CPU baseline only
    args, dev, cfg = ctx.args, ctx.device, PLP_CFG
    rec, ref, rs = sr.random_alignment(cfg["region"], depth=cfg["depth"], read_len=cfg["read_len"], seed=cfg["seed"],          # the same records on every rank (weak scaling)
                                      
                                       indel_rate=cfg["indel_rate"], origin=cfg["origin"])
    start, end = cfg["origin"], cfg["origin"] + cfg["region"]
    host = pc.BamRecords.from_dict(rec)
    # parity on the bench input (a 65,536-column prefix keeps the CPU side bounded), then the CPU baseline on the same prefix
    n_ctr = min(4, len(ctx.streams))
    counters = [pc.PileupCounter(dev) for _ in range(n_ctr)]
    sample_end = start + 65536
    got = counters[0].count(host, start, sample_end, ref, rs).fetch()
    t0 = time.perf_counter()
    want = po.clair3_pileup(rec, start, sample_end, ref, rs)
    cpu_s = time.perf_counter() - t0
    exact = all(got[k].shape == want[k].shape and np.array_equal(got[k], want[k]) for k in ("matrix", "major", "stats", "cand_cols", "cand_ok"))
    sample_bases = int(want["stats"][:, 0].sum())
    if not exact:
        raise RuntimeError("pileup_counts: GPU result differs from the oracle on the bench input")

    drec = host.to_device(dev, ref)
    full = counters[0].count(drec, start, end, None, rs).fetch()
    bases = int(full["stats"][:, 0].sum())
    n_cols, n_cand = len(full["major"]), len(full["cand_cols"])
    ms_alone, launches_per_call = counters[0].last_ms()
    K = args.steps
    cnt = [0]

    def issue_dev(n):
        k = cnt[0]
        for i in range(n):
            j = (k + i) % n_ctr
            with torch.cuda.stream(ctx.streams[j]):
                counters[j].count(drec, start, end, None, rs)
        cnt[0] = k + n

    issue_dev(2 * n_ctr)
    torch.cuda.synchronize(dev)
    issue_dev(args.warmup)
    ms, clocks = ctx.timed(issue_dev, K)
    value = bases * K * ctx.world / (ms * 1e-3)
    if ctx.dump is not None:                      # what a caller fetches after the last timed count
        got = counters[(cnt[0] - 1) % n_ctr].fetch()
        rows = sample_rows(len(got["major"]))
        ctx.dump.update({"pileup_counts_matrix": got["matrix"][rows], "pileup_counts_major": got["major"][rows],
                         "pileup_counts_stats": got["stats"][rows], "pileup_counts_rows": rows,
                         "pileup_counts_cand_cols": got["cand_cols"], "pileup_counts_cand_ok": got["cand_ok"]})

    # e2e: pinned host records in, results out, synchronous per call (the shape of the reference's per-chunk call)
    pin = pc.BamRecords(**{k: torch.from_numpy(getattr(host, k).view({"uint16": np.int16, "uint32": np.int32}.get(getattr(host, k).dtype.name, getattr(host, k).dtype))).pin_memory().numpy().view(getattr(host, k).dtype)
                           for k, _ in pc._FIELDS})
    ecnt = [0]

    def issue_e2e(n):
        for i in range(n):
            with torch.cuda.stream(ctx.streams[0]):
                counters[0].count(pin, start, end, ref, rs).fetch(pinned=True)
        ecnt[0] += n

    issue_e2e(2)
    e2e_ms, _ = ctx.timed(issue_e2e, K)
    e2e_value = bases * K * ctx.world / (e2e_ms * 1e-3)
    h2d = host.nbytes() + len(ref)
    d2h = n_cols * (18 * 8 + 8 + 24) + n_cand * 9
    pk = peaks()
    # compulsory bytes of one call: the records and reference read once, the emitted arrays written once
    alg_bytes = h2d + d2h + n_cand * 8
    ach = alg_bytes / (ms_alone * 1e-3) / 1e9
    traffic = None
    try:
        ent = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["pileup_counts"]["count_tile"]
        if ent.get("region_columns") == cfg["region"] and ent.get("depth") == cfg["depth"]:
            traffic = ent["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    out = {"metric": "aligned-bases/sec", "value": value, "unit": "bases/s", "scaling": "weak", "steps": K,
           "timed_region_s": ms * 1e-3, "ms_per_step": ms / K, "clocks": clocks,
           "columns_per_s": n_cols * K * ctx.world / (ms * 1e-3),
           "gpu_launches": int(launches_per_call * K), "parity": "bit-exact vs oracle/pileup_oracle.c on the first 65536 columns of the bench input",
           "config": {"workload": "pileup feature counting (calculate_clair3_pileup) over a synthetic %d-column region, mean depth %d, "
                                  "%d reads of ~%d bases (%d CIGAR words), %d aligned bases, %d candidates; %d calls in flight"
                                  % (cfg["region"], cfg["depth"], host.n_reads, cfg["read_len"], len(host.cigar), bases, n_cand, n_ctr)},
           "e2e": {"value": e2e_value, "unit": "bases/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": K,
                   "timed_region_s": e2e_ms * 1e-3,
                   "mode": "PileupCounter.count(pinned host records).fetch(pinned=True): H2D of the records, 8 kernels, D2H of matrix / major / stats / candidates into page-locked buffers, synchronous per call"},
           "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": traffic,
                        "peak_source": pk["which"], "kernel": "all 8 kernels of one call, timed alone with CUDA events on its stream (c3b_plp_last_ms): %.3f ms" % ms_alone,
                        "algorithmic_bytes_per_call": alg_bytes,
                        "note": "achieved = compulsory bytes (records + reference in, emitted arrays out) / the call's device time; traffic = DRAM bytes "
                                "of the dominant kernel (plp_count_tile, 86 % of the call) from the committed ncu capture.  That kernel is issue-bound "
                                "(ncu: 76 % of the issue slots busy, ~470 warp instructions per read and warp: a binary search over the CIGAR prefix "
                                "sums per read and column, single-lane indel bookkeeping), not bandwidth-bound"}}
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = {"value": sample_bases / cpu_s, "unit": "bases/s", "cores": 1, "kind": "port",
                               "sample": "oracle/pileup_oracle.c (plain-C restatement of calculate_clair3_pileup, single thread like the reference's "
                                         "per-chunk call) on the first 65536 columns of the same records: %d aligned bases in %.3f s" % (sample_bases, cpu_s)}
        try:                                          # the reference's deployment shape: one process per chunk on all host cores
            ncores = len(os.sched_getaffinity(0))
            dep = cpu_counts_all_cores(rec, ref, rs, start, end, max(1, min(ncores * 3 // 4, 64)))
            out["cpu_baseline"]["single_thread"] = {"value": out["cpu_baseline"]["value"], "cores": 1}
            out["cpu_baseline"]["deployment_shape"] = dep
            if dep["processes"] > 0 and dep["value"] > out["cpu_baseline"]["value"]:
                out["cpu_baseline"].update({"value": dep["value"], "cores": dep["processes"],
                                            "sample": dep["sample"] + " (oracle/pileup_oracle.c; single thread on the first 65536 columns: %.1f M bases/s)"
                                                      % (sample_bases / cpu_s / 1e6)})
        except Exception as e:                        # noqa: BLE001 - the one-core figure stands
            out["cpu_baseline"]["deployment_shape"] = {"error": "%s: %s" % (type(e).__name__, e)}
    for c in counters:
        c.close()
    del drec
    torch.cuda.empty_cache()
    return out


def cpu_counts_all_cores(rec, ref, rs, start, end, nproc, min_seconds=1.5):
    """The feature counter's CPU baseline in the reference's deployment shape: the region cut into `nproc` chunks, one
    single-threaded oracle process per chunk, all running at once (the reference: one CreateTensorPileupFromCffi process per chunk
    under GNU parallel); each worker counts its chunk repeatedly for >= min_seconds; rate = sum of the workers' rates."""
    import tempfile
    tmp = tempfile.mkdtemp(prefix="c3b_plp_cpu_")
    path = os.path.join(tmp, "records.npz")
    np.savez(path, ref=np.frombuffer(ref.encode() if isinstance(ref, str) else ref, dtype=np.uint8), ref_start=np.int64(rs), **rec)
    cuts = [start + (end - start) * i // nproc for i in range(nproc + 1)]
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
    procs = [subprocess.Popen([sys.executable, "-m", "oracle.pileup_oracle", path, str(cuts[i]), str(cuts[i + 1]), str(min_seconds)],
                              cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for i in range(nproc)]
    total, ok, secs = 0.0, 0, 0.0
    for p in procs:
        try:
            out, _ = p.communicate(timeout=min_seconds * 20 + 120)
            r = json.loads(out.strip().splitlines()[-1])
            if r["seconds"] > 0:
                total += r["bases"] / r["seconds"]
                secs = max(secs, r["seconds"])
                ok += 1
        except Exception:
            p.kill()
    try:
        os.remove(path)
        os.rmdir(tmp)
    except OSError:
        pass
    return {"value": total, "unit": "bases/s", "processes": ok, "threads_each": 1, "seconds": secs,
            "sample": "%d single-thread oracle processes, one contiguous chunk of the bench region each, counted repeatedly for >= %.1f s, rates summed"
                      % (ok, min_seconds)}


def select_workloads(spec, explicit, world):
    """The sub-records one run measures.  The feature counter shards by region with no exchange at all (replicas only), so the
    multi-rank line stays the measured round-2 shape (networks + cascade) and the counter is a single-GPU sub-record unless it is
    asked for by name."""
    names = [x for x in spec.split(",") if x]
    if not explicit and world > 1:
        names = [x for x in names if x != "pileup_counts"]
    return names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="K: steps in every timed region")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workloads", default="pileup,fa,fa_dwell,cascade,pileup_counts")
    ap.add_argument("--workload", default=None, help="alias: run a single workload")
    ap.add_argument("--streams", type=int, default=12)
    ap.add_argument("--lstm-wg", type=int, default=0, help="epilogue warpgroups per LSTM sub-tile (0 = library default)")
    ap.add_argument("--lstm-tile", type=int, default=0,
                    help="sites per LSTM1 sub-tile (16|32|64; 0 = library choice by call shape: 64 for stream-ordered calls, the "
                         "smallest GPU-filling tile for synchronous host-buffer calls)")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value for the pileup model (tuning runs), repeatable")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs of every workload as DIR/<name>.npy (b200 arm, rank 0)")
    args = ap.parse_args()
    explicit = args.workload is not None or any(a.startswith("--workloads") for a in sys.argv[1:])
    args.workloads = select_workloads(args.workload or args.workloads, explicit, int(os.environ.get("WORLD_SIZE", "1")))
    if args.steps <= 0:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the b200 arm's outputs")
    requested_warmup = args.warmup
    if args.warmup < 3:
        args.warmup = 3                                               # the timing rules ask for >= 3 warm-up steps

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch.distributed as dist
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)

    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    ctx = Ctx(args, rank, world, device, sampler)

    need = set(args.workloads)
    if "cascade" in need:
        need |= {"pileup", "fa"}
    models, bcast = {}, {"bytes": 0, "how": None}
    for wname in ("pileup", "fa", "fa_dwell"):
        if wname not in need:
            continue
        w = WORKLOADS[wname]
        m = make_model(w, device, load_real_weights=(rank == 0))
        if w["kind"] == "pileup":
            if args.lstm_wg:
                m.set_option("lstm_wg", args.lstm_wg)
            if args.lstm_tile:
                m.set_option("lstm_tile", args.lstm_tile)
            for kv in args.opt:
                k, v = kv.split("=")
                m.set_option(k, int(v))
        if world > 1:
            from clair3_b200 import sharding
            nbytes, how = sharding.broadcast_weights(m, src=0)        # the one NCCL collective per model, before any timed region
            bcast["bytes"] += nbytes
            bcast["how"] = how
        models[wname] = m

    subs = {}
    for wname in args.workloads:
        if wname == "cascade":
            subs[wname] = run_cascade(ctx, models["pileup"], models["fa"])
        elif wname == "pileup_counts":
            try:                                                      # a widening row: it must not be able to take the headline down
                subs[wname] = run_pileup_counts(ctx)
            except Exception as e:                                    # noqa: BLE001
                subs[wname] = {"error": "%s: %s" % (type(e).__name__, e)}
                torch.cuda.synchronize(device)
        else:
            subs[wname] = run_forward_workload(ctx, wname, models[wname])

    # ---- CPU baseline beside it (rank 0, N = 1 only): bounded samples of the same workloads
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        for wname in args.workloads:
            if wname == "pileup":
                subs[wname]["cpu_baseline"] = cpu_baseline_for("pileup", 10.0, 6.0)
            elif wname == "fa":
                subs[wname]["cpu_baseline"] = cpu_baseline_for("fa", 8.0, 6.0)
            elif wname == "fa_dwell":
                subs[wname]["cpu_baseline"] = cpu_baseline_for("fa_dwell", 5.0, 0.0)
        if "cascade" in subs and "cpu_baseline" in subs.get("pileup", {}) and "cpu_baseline" in subs.get("fa", {}):
            cp, cf = subs["pileup"]["cpu_baseline"], subs["fa"]["cpu_baseline"]
            t = CASCADE_PILEUP_SITES / cp["value"] + CASCADE_FA_SITES / cf["value"]
            subs["cascade"]["cpu_baseline"] = {
                "value": (CASCADE_PILEUP_SITES + CASCADE_FA_SITES) / t, "unit": "sites/s", "cores": max(cp["cores"], cf["cores"]),
                "kind": "port", "sample": "derived from the two bounded CPU samples above: total sites / (pileup sites / pileup rate "
                                           "+ full-alignment sites / full-alignment rate)"}
    if sampler:
        sampler.stop()

    if rank == 0:
        head_name = "pileup" if "pileup" in subs else [n for n in args.workloads if "error" not in subs.get(n, {})][0]
        head = subs[head_name]
        e2e = dict(head["e2e"])
        if "h2d_bytes_per_step" not in e2e:                           # cascade as the head (single-workload runs)
            e2e["h2d_bytes_per_step"] = e2e.get("h2d_bytes_per_pass_per_rank")
            e2e["d2h_bytes_per_step"] = e2e.get("d2h_bytes_per_pass_per_rank")
        line = {
            "metric": "candidate-sites/sec", "value": head["value"], "unit": "sites/s", "n_gpus": world, "steps": args.steps,
            "warmup": requested_warmup, "warmup_steps_run": args.warmup, "ms_per_step": head.get("ms_per_step", head.get("ms_per_pass")),
            "timed_region_s": head["timed_region_s"],
            "higher_is_better": True, "scaling": head["scaling"], "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": head["config"], "run": head.get("run"),
            "clocks": head["clocks"],
            "e2e": e2e,
            "gpu_launches": head.get("gpu_launches", 0) if head_name != "cascade" else int(models["pileup"].launch_count + models["fa"].launch_count),
            "roofline": head.get("roofline"),
            "kernels": head.get("kernels"),
            "cpu_baseline": head.get("cpu_baseline"),
            "parity_max_abs_dp": head.get("parity_max_abs_dp"),
            "weight_broadcast": bcast,
            "workloads": subs,
        }
        if ctx.dump is not None:
            dump_outputs(args.dump_outputs, ctx.dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
