#!/usr/bin/env python
"""bench.py -- MARCONet inference hot path on B200 (metric: SR chars/s, 128-px-high output).

A "step" is one pass of the full hot path (TextContextEncoderV2 -> TSPGAN -> TSPSRNet, the data flow of the
reference's test_sr.py:145-197) over one batch of synthetic 32x512 LR text lines with 16 characters each
(BASELINE.json configs[1]; --lines sets lines per GPU per step).  One process per GPU; lines are independent
(test_sr.py:77) so ranks shard lines with no data-path collective ("weak" scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--lines L] [--chars C] [--dump-outputs DIR]

Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for how every field is produced.  --dump-outputs DIR writes
rank 0's SR images of the last timed step as DIR/sr.npy (float32): inputs and weights are seeded and do not depend on the
host, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# algorithmic work, SURVEY.md section 8d (2*MAC of every conv/linear/matmul of the reference modules)
GF_ENCODER_LINE = 111.692
GF_TSPGAN_CHAR = 41.785
GF_SR_LINE = 484.146
GF_SR_CHAR = 47.245


def gflop_per_line(chars):
    return GF_ENCODER_LINE + GF_SR_LINE + (GF_TSPGAN_CHAR + GF_SR_CHAR) * chars


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region, in-process through NVML (pynvml), every 20 ms;
    falls back to polling nvidia-smi when NVML is unavailable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def run(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                if n is not None:
                    mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                    r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                    flags = [bool(r & n.nvmlClocksEventReasonHwSlowdown), bool(r & n.nvmlClocksEventReasonHwThermalSlowdown),
                             bool(r & n.nvmlClocksEventReasonSwThermalSlowdown), bool(r & n.nvmlClocksEventReasonSwPowerCap)]
                    self.samples.append([str(mhz), str(self.max_mhz)] + ["Active" if f else "Not Active" for f in flags])
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.02 if n is not None else 0.2)

    def summary(self):
        self.stop_flag.set()
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx or None, reasons=sorted(reasons), samples=len(sm),
                    source="nvml" if self.nvml is not None else "nvidia-smi")


def make_inputs(lines, chars, seed):
    from marconet_b200.testing import synth   # seeded synthetic input generators (random tensors only)
    lq = synth.make_lq(lines, seed)
    labels = [synth.make_labels(chars, seed + b) for b in range(lines)]
    locs = synth.make_locs(lines, chars)
    return lq, labels, locs


# --------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port (the reference is Python and cannot travel to the GPU box;
# oracle/restate.py is bit-identical to its modules, tests/test_oracle.py) on all host cores.
# --------------------------------------------------------------------------------------------
_BEST_THREADS = None


def best_cpu_threads():
    """The reference's torch CPU path does not scale to every core of a big host (grouped conv, networks.py:294):
    probe a 1-character TSPGAN forward at a few thread counts and give the baseline its fastest setting."""
    global _BEST_THREADS
    if _BEST_THREADS is None:
        import torch
        from oracle import restate, synth
        sds = synth.make_checkpoints(0)
        ncpu = os.cpu_count() or 1
        cands = sorted({c for c in (ncpu, ncpu // 2, 64, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
        lab, sty = synth.make_labels(1, 0), synth.make_styles(1, 0)
        best = None
        with torch.no_grad():
            for c in cands:
                torch.set_num_threads(c)
                restate.tspgan_forward(sds["tspgan"], sty, lab)
                t0 = time.perf_counter()
                restate.tspgan_forward(sds["tspgan"], sty, lab)
                dt = time.perf_counter() - t0
                if best is None or dt < best[0]:
                    best = (dt, c)
        _BEST_THREADS = best[1]
    return _BEST_THREADS


def cpu_line_seconds(chars, repeats=1, threads=None):
    import torch
    from oracle import restate, synth
    threads = threads or best_cpu_threads()
    torch.set_num_threads(threads)
    sds = synth.make_checkpoints(0)
    lq, labels, locs = make_inputs(1, chars, 0)
    best = None
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            restate.full_line(sds, lq, labels, locs)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return best, threads


def workload_string(lines, chars):
    """One wording for both arms (the driver compares the `config.workload` strings of the two JSON lines)."""
    return (f"{lines} synthetic 32x512 LR line(s) x {chars} chars per GPU per step, "
            f"encoder->TSPGAN->TSPSRNet (BASELINE configs[1])")


PIN = ("oracle/restate.py = the reference's torch CPU path restated op for op; pinned bit-identical (max |diff| = 0.0) to the "
       "unmodified reference modules by tests/test_oracle.py::test_oracle_is_bit_identical_to_reference_modules and against "
       "tests/golden/*.npz generated from them (oracle/make_golden.py, oracle/make_golden2.py)")


def run_reference_arm(args):
    """The reference's own CPU implementation of the path on the box's host cores, one rank only.  The reference is Python and
    cannot travel to the GPU box (no /root/reference there), so the arm runs its pinned restatement (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    chars, lines = args.chars, args.lines
    warm = max(1, args.warmup)
    t_first, threads = cpu_line_seconds(chars, 1)                      # first warm-up step (also sizes the run)
    per_step = max(t_first, 1e-3) * lines
    warm = max(1, min(warm, int(30.0 // per_step)))                    # honour --warmup within a bounded CPU budget
    for _ in range(warm - 1):
        for _ in range(lines):
            cpu_line_seconds(chars, 1)
    steps = args.steps
    times = []
    for _ in range(steps):
        t = 0.0
        for _ in range(lines):                                         # the reference restores one line at a time (test_sr.py:77)
            t += cpu_line_seconds(chars, 1)[0]
        times.append(t)
    ms = 1e3 * sum(times) / len(times)
    value = lines * chars / (ms / 1e3)
    rec = {
        "impl": "reference", "metric": "sr_chars_per_sec", "value": value, "unit": "chars/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_string(lines, chars), "lines_per_step_per_gpu": lines, "chars_per_line": chars,
                   "note": "one CPU process on rank 0 whatever --gpus says: per-N ratios against this arm are only meaningful at N=1"},
        "cpu_baseline": {"value": value, "unit": "chars/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} step(s) of {lines} full {chars}-char line(s), torch {torch.__version__} CPU fp32, {threads} threads "
                                   f"(its fastest setting of those probed). " + PIN},
        "e2e": {"value": value, "unit": "chars/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(rec), flush=True)


# --------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from marconet_b200 import _lib, ops
    from marconet_b200.models import networks
    from marconet_b200.testing import synth   # synthetic checkpoint generator (random weights only)

    _lib.load()   # fail loudly if the CUDA library is missing
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.precision is not None:
        ops.set_default_precision(args.precision)

    sds = synth.make_checkpoints(0)
    nets = {}
    for key, cls in (("tspgan", networks.TSPGAN), ("encoder", networks.TextContextEncoderV2), ("sr", networks.TSPSRNet)):
        m = cls()
        m.load_state_dict(sds[key], strict=True)
        nets[key] = m.eval().to(dev)

    lines, chars = args.lines, args.chars
    lq_h, labels, locs_h = make_inputs(lines, chars, seed=100 * rank)
    lq_pin, locs_pin = lq_h.pin_memory(), locs_h.pin_memory()
    lab_dev = [l.to(dev) for l in labels]
    lq_dev, locs_dev = lq_pin.to(dev), locs_pin.to(dev)

    lab_all = torch.cat(lab_dev, dim=0)
    lab_cpu = torch.cat(labels, dim=0)        # the reference's caller keeps the labels on the CPU (test_sr.py:180 never moves them)

    def step(lq, locs):
        _, _, w = nets["encoder"](lq)
        # one generator call for the characters of all lines of the step (per-character style = its line's w), then per-line views
        _, f64, f32_ = nets["tspgan"](styles=w.repeat_interleave(chars, dim=0), labels=lab_cpu, noise=None)
        p64 = [f64[b * chars:(b + 1) * chars] for b in range(lines)]
        p32 = [f32_[b * chars:(b + 1) * chars] for b in range(lines)]
        return nets["sr"](lq, p64, p32, locs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            out = fn()
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms, out

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step(lq_dev, locs_dev)
        if args.profile:   # exactly one step between cudaProfilerStart/Stop (ncu --profile-from-start off)
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            step(lq_dev, locs_dev)
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
            return
        sampler = ClockSampler(local)
        sampler.start()
        l0 = ops.LAUNCHES
        ms_total, out = timed(lambda: step(lq_dev, locs_dev), args.steps)
        launches = (ops.LAUNCHES - l0) // args.steps
        eager_sr = out.cpu() if args.dump_outputs else None
        graph_sr = None
        # the same step recorded once into a CUDA graph and replayed (SURVEY 8f n1): identical kernels and results, no Python
        # between launches, label/window checks on the device.  Used for `value` when capture works and replays bit-exactly.
        graph_info, g = None, None
        if not args.no_graph:
            try:
                from marconet_b200.graph import GraphedLines
                g = GraphedLines(nets["encoder"], nets["tspgan"], nets["sr"], lines=lines, chars=chars, device=dev)
                g.load(lq_dev, lab_all, locs_dev)
                same = bool(torch.equal(g.replay(), step(lq_dev, locs_dev)))
                g.check()
                graph_info = {"launches_per_replay": int(g.launches), "bit_identical_to_eager": same}
            except Exception as exc:   # capture is an optimisation: report why it was skipped and keep the eager number
                graph_info, g = {"error": f"{type(exc).__name__}: {exc}"[:300]}, None
            ok = torch.tensor([1.0 if (g is not None and graph_info["bit_identical_to_eager"]) else 0.0], device=dev)
            if world > 1:              # timed() contains collectives: every rank replays, or none does
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() > 0.5:
                for _ in range(2):
                    g.replay()
                ms_graph, out = timed(g.replay, args.steps)
                graph_info["ms_per_step"] = ms_graph / args.steps
                graph_sr = out.cpu() if args.dump_outputs else None     # a static buffer: later replays overwrite it
            elif g is not None:
                graph_info["skipped"] = "another rank could not capture" if graph_info["bit_identical_to_eager"] else "replay differs from eager"

        clocks = sampler.summary()      # sampled over the eager and the graph timed regions

        # e2e: host buffers in, SR image out, copies inside the timed region
        sr_host = torch.empty((lines, 3, 128, 2048), dtype=torch.float32).pin_memory()

        def e2e_step():
            lq = lq_pin.to(dev, non_blocking=True)
            locs = locs_pin.to(dev, non_blocking=True)
            sr = step(lq, locs)
            sr_host.copy_(sr, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        e2e_step()
        ms_e2e, _ = timed(e2e_step, args.steps)

        roof = modconv_roofline(nets["tspgan"], chars, dev) if rank == 0 else None
        collective = None
        if not args.no_collective:
            try:
                collective = collective_record(nets, world, rank, dev, args)
            except Exception as exc:      # the sub-records must never cost the headline line
                collective = {"error": f"{type(exc).__name__}: {exc}"[:300]}

        # informational: end to end through GraphedLines (this repo's own extension API) with the same host buffers and copies.
        # Single process only (no collectives inside, so a failure here cannot desynchronise ranks); runs last.
        if world == 1 and g is not None and graph_info and "ms_per_step" in graph_info:
            try:
                def e2e_graph_step():
                    out = g(lq_pin, None, locs_pin)            # H2D into the static buffers + one graph replay
                    sr_host.copy_(out, non_blocking=True)
                    torch.cuda.current_stream().synchronize()

                e2e_graph_step()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                ev0.record()
                for _ in range(args.steps):
                    e2e_graph_step()
                ev1.record()
                torch.cuda.synchronize()
                g.check()
                graph_info["e2e_ms_per_step"] = ev0.elapsed_time(ev1) / args.steps
                graph_info["e2e_chars_per_sec"] = lines * chars / (graph_info["e2e_ms_per_step"] / 1e3)
            except Exception as exc:
                graph_info["e2e_error"] = f"{type(exc).__name__}: {exc}"[:200]

    total_chars = world * lines * chars
    ms_step = ms_total / args.steps
    ms_eager = ms_step
    # ms_per_step of both modes is already the max over ranks, so every rank takes the same branch
    use_graph = bool(graph_info and "ms_per_step" in graph_info and graph_info["ms_per_step"] < ms_step)
    if use_graph:
        ms_step = graph_info["ms_per_step"]
        launches = graph_info["launches_per_replay"]
    value = total_chars / (ms_step / 1e3)
    e2e_value = total_chars / (ms_e2e / args.steps / 1e3)

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, sr=graph_sr if use_graph else eager_sr)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            t, threads = cpu_line_seconds(chars, 1)
            cpu = {"value": chars / t, "unit": "chars/s", "cores": threads, "kind": "port",
                   "sample": f"one full {chars}-char 32x512 line, torch CPU fp32, {threads} threads. " + PIN}
        rec = {
            "metric": "sr_chars_per_sec", "value": value, "unit": "chars/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(lines, chars),
                       "lines_per_step_per_gpu": lines, "chars_per_line": chars, "parallelism": f"line-sharded dp{world}, no collective",
                       "precision": {0: "fp32 CUDA-core", 1: "fp16x3 tcgen05", 2: "bf16x3 tcgen05", 3: "fp16 tcgen05"}[ops.default_precision()],
                       "l2": "weights (352 MB fp32) + activations (>1 GB/line) exceed the 126 MB L2; no flush needed",
                       "launch_mode": "cuda_graph_replay" if use_graph else "module_calls", "eager_ms_per_step": ms_eager,
                       "module_api": "the three reference-facing module calls; each module replays a CUDA graph of its forward from "
                                     "the second call with the same input signature on (MN_MODULE_GRAPHS=0: plain eager launches)"
                                     if ops.MODULE_GRAPHS else "eager launches (MN_MODULE_GRAPHS=0)",
                       "cuda_graph": graph_info,
                       "gflop_per_step_per_gpu": gflop_per_line(chars) * lines,
                       "achieved_tflops_per_gpu": gflop_per_line(chars) * lines / ms_step},
            "ms_per_line": ms_step / lines,
            "e2e": {"value": e2e_value, "unit": "chars/s", "h2d_bytes_per_step": int(lq_pin.numel() * 4 + locs_pin.numel() * 4),
                    "d2h_bytes_per_step": int(sr_host.numel() * 4)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "collective": collective,
        }
        rec["config"]["tc_fallback_shapes"] = len(ops.TC_FALLBACKS)
        print(json.dumps(rec), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(directory, **arrays):
    """Writes each array as directory/<name>.npy in float32.  An array larger than DUMP_BYTES / len(arrays) is replaced by a
    fixed, seeded sample of its flattened elements (same indices on every run of the same shape), in index order."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    budget = (DUMP_BYTES // len(arrays) - 4096) // 4          # elements per file, leaving room for the .npy header
    for name, t in arrays.items():
        a = t.float().numpy()
        if a.size > budget:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, budget, replace=False))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def collective_record(nets, world, rank, dev, args):
    """The north_star's REAL multi-GPU split, driver-visible (SURVEY 8e; VERDICT r1 item 5): characters sharded over ranks with an
    exchange of the prior features the SR decoder consumes (reference consumer: networks.py:442-445, 475-478).

    priors1024  BASELINE configs[2]: 1024 (label, w) pairs, prior generation only, STRONG scaling (1024 characters in total
                whatever N is): block-cyclic character shards, compute only vs + owner-only all-to-all (each line's priors go to
                the rank that owns the line) vs + the round-1 all-gather to every rank.
    lines64     BASELINE configs[3]: 64 lines x 16 characters end to end (64/N lines per rank): line-sharded (no exchange) vs
                character-sharded priors (encoder on owned lines -> all-gather of w (2 KB/line) -> block-cyclic TSPGAN ->
                all-to-all of fea64/fea32 to the line owners -> TSPSRNet on owned lines).
    Every number: CUDA events, barrier + synchronize on both sides, max over ranks.  Collectives are NCCL over NVLink."""
    import torch
    import torch.distributed as dist
    from marconet_b200 import parallel
    from marconet_b200.testing import synth
    W = world
    steps = 3

    def timed(fn):
        for _ in range(2):
            fn()
        if W > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        if W > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item())

    out = {}
    peer = None
    gen, enc, sr = nets["tspgan"], nets["encoder"], nets["sr"]
    chunk = 128                                     # characters per TSPGAN call (bounds activation memory at N=1)
    with torch.no_grad():
        # ---------------- configs[2]: 1024 random (label, w) pairs, prior only
        n = 1024
        if n % (W * W) == 0:
            labels = synth.make_labels(n, 11).to(dev)
            styles = synth.make_styles(n, 11).to(dev)
            own = n // W

            per_call = min(chunk * W, n)
            if W > 1:       # in-kernel exchange: symmetric-memory receive buffers + per-character destination pointers (NVLink peer stores)
                ok = torch.ones(1, device=dev)
                try:
                    peer = parallel.PeerPriorExchange(per_call, dev)
                except Exception as exc:
                    peer, ok = None, torch.zeros(1, device=dev)
                    out["peer_stores_error"] = f"{type(exc).__name__}: {exc}"[:300]
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if ok.item() < 0.5:
                    peer = None

            def run_priors(mode):
                # generated in `chunk`-character calls per rank; every chunk of W*chunk_local characters is its own block-cyclic round
                for c0 in range(0, n, per_call):
                    s_, l_ = styles[c0:c0 + per_call], labels[c0:c0 + per_call]
                    if mode == "all_gather":
                        parallel.generate_priors_sharded(gen, s_, l_)
                    elif mode == "peer":
                        peer.generate(gen, s_, l_)
                    else:
                        parallel.generate_priors_for_owners(gen, s_, l_, exchange=(mode == "all_to_all"))

            ms_c = timed(lambda: run_priors("compute"))
            rec = {"chars_total": n, "chars_per_rank": own, "scaling": "strong", "ms_compute_only": ms_c,
                   "chars_per_sec_compute_only": n / (ms_c / 1e3)}
            if W > 1:
                ms_a2a = timed(lambda: run_priors("all_to_all"))
                ms_ag = timed(lambda: run_priors("all_gather"))
                b = parallel.exchange_bytes_per_rank(n, W)
                rec.update({"ms_with_all_to_all": ms_a2a, "chars_per_sec_with_all_to_all": n / (ms_a2a / 1e3),
                            "all_to_all_bytes_sent_per_rank": b["all_to_all"],
                            "all_to_all_gbps_per_rank": b["all_to_all"] / max(ms_a2a - ms_c, 1e-3) / 1e6,
                            "ms_with_all_gather": ms_ag, "chars_per_sec_with_all_gather": n / (ms_ag / 1e3),
                            "all_gather_bytes_received_per_rank": b["all_gather"],
                            "all_gather_gbps_per_rank": b["all_gather"] / max(ms_ag - ms_c, 1e-3) / 1e6,
                            "exchange": "NCCL all_to_all_single of fea64+fea32 (6 MiB/char) to line owners; all_gather = round-1 variant"})
                if peer is not None:
                    # correctness of the in-kernel exchange: the owned characters must equal the all-to-all result bit for bit
                    a = parallel.generate_priors_for_owners(gen, styles[:per_call], labels[:per_call])
                    b = peer.generate(gen, styles[:per_call], labels[:per_call])
                    same = torch.tensor([1.0 if (torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])) else 0.0], device=dev)
                    dist.all_reduce(same, op=dist.ReduceOp.MIN)
                    ms_peer = timed(lambda: run_priors("peer"))
                    rec.update({"ms_with_peer_stores": ms_peer, "chars_per_sec_with_peer_stores": n / (ms_peer / 1e3),
                                "peer_stores_equal_all_to_all": bool(same.item() > 0.5),
                                "peer_stores": "the tap convolutions' epilogues store fea64/fea32 through per-character pointers into the "
                                               "owners' symmetric-memory buffers (mn_conv_params.y2_ptrs, NVLink stores from the tcgen05 "
                                               "kernel); one device-side barrier per round; no collective moves features"})
            out["priors1024"] = rec
            del labels, styles
        # ---------------- configs[3]: 64 lines x 16 chars end to end
        L, C = 64, 16
        if L % W == 0 and (L * C) % (W * W) == 0:
            lpr = L // W
            lq_all = synth.make_lq(L, 500)
            lq_own = lq_all[rank * lpr:(rank + 1) * lpr].to(dev)
            lab_all = torch.cat([synth.make_labels(C, 500 + b) for b in range(L)], 0).to(dev)
            lab_own = lab_all[rank * lpr * C:(rank + 1) * lpr * C]
            locs_own = synth.make_locs(lpr, C).to(dev)
            lines_per_call = max(1, chunk // C)

            def line_sharded():
                _, _, w = enc(lq_own)
                res = []
                for b0 in range(0, lpr, lines_per_call):             # `chunk` characters (= lines_per_call lines) per TSPGAN / TSPSRNet call
                    b1 = min(lpr, b0 + lines_per_call)
                    _, f64, f32_ = gen(styles=w[b0:b1].repeat_interleave(C, dim=0), labels=lab_own[b0 * C:b1 * C], noise=None)
                    p64 = [f64[i * C:(i + 1) * C] for i in range(b1 - b0)]
                    p32 = [f32_[i * C:(i + 1) * C] for i in range(b1 - b0)]
                    res.append(sr(lq_own[b0:b1], p64, p32, locs_own[b0:b1]))
                return res

            per_call = min(chunk * W, L * C)                # characters per block-cyclic round (all ranks together)
            rounds = (L * C) // per_call
            lines_round = per_call // C                     # a round covers this many consecutive global lines ...
            own_lines = max(1, lines_round // W)            # ... of which this rank owns the rank-th block
            lq_all_dev = lq_all.to(dev)

            def char_sharded(use_peer=False):
                _, _, w = enc(lq_own)
                if W > 1:
                    w_all = torch.empty((L, w.shape[1]), dtype=w.dtype, device=dev)
                    dist.all_gather_into_tensor(w_all, w.contiguous())      # global line order = rank-major blocks of lq_own
                else:
                    w_all = w
                styles = w_all.repeat_interleave(C, dim=0)
                res = []
                for k in range(rounds):
                    c0 = k * per_call
                    if use_peer:
                        f64, f32_ = peer.generate(gen, styles[c0:c0 + per_call], lab_all[c0:c0 + per_call])
                    else:
                        f64, f32_ = parallel.generate_priors_for_owners(gen, styles[c0:c0 + per_call], lab_all[c0:c0 + per_call])
                    g0 = k * lines_round + rank * own_lines                 # first global line of this rank's block in round k
                    p64 = [f64[b * C:(b + 1) * C] for b in range(own_lines)]
                    p32 = [f32_[b * C:(b + 1) * C] for b in range(own_lines)]
                    res.append(sr(lq_all_dev[g0:g0 + own_lines], p64, p32, locs_own[:own_lines]))
                return res

            ms_line = timed(line_sharded)
            rec = {"lines_total": L, "chars_per_line": C, "lines_per_rank": lpr, "ms_line_sharded_no_exchange": ms_line,
                   "chars_per_sec_line_sharded": L * C / (ms_line / 1e3)}
            if W > 1 and lines_ok_for_rounds(L, C, W, chunk):
                ms_char = timed(char_sharded)
                b = parallel.exchange_bytes_per_rank(L * C, W)
                rec.update({"ms_char_sharded_with_all_to_all": ms_char, "chars_per_sec_char_sharded": L * C / (ms_char / 1e3),
                            "all_to_all_bytes_sent_per_rank": b["all_to_all"], "rounds": rounds,
                            "exchange": "all_gather of w (2 KB/line) + NCCL all_to_all_single of fea64/fea32 to line owners"})
                if peer is not None and peer.n == per_call:
                    ms_peer = timed(lambda: char_sharded(True))
                    rec.update({"ms_char_sharded_with_peer_stores": ms_peer, "chars_per_sec_char_sharded_peer_stores": L * C / (ms_peer / 1e3)})
            out["lines64"] = rec
    return out if rank == 0 else None


def lines_ok_for_rounds(L, C, W, chunk):
    """char_sharded() hands every round's owner block to TSPSRNet as whole lines: a round must hold a multiple of W lines."""
    per_call = min(chunk * W, L * C)
    return per_call % C == 0 and (per_call // C) % W == 0 and (L * C) % per_call == 0


def _time_modconv(e, chars, dev, iters):
    import torch
    from marconet_b200 import ops
    x = torch.randn(chars, 32, 32, 512, device=dev)
    dm = torch.rand(chars, 512, device=dev) + 0.5
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)   # 256 MB > L2
    st = torch.cuda.current_stream()
    tot = 0.0
    for i in range(iters + 3):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        ops.conv2d(x, e["w"], 3, 3, pad=(1, 1), bias=e["bias"], out_scale=dm, act=ops.ACT_LRELU02, gain=2 ** 0.5)
        e1.record(st)
        torch.cuda.synchronize()
        if i >= 3:
            tot += e0.elapsed_time(e1)
    ms = tot / iters
    return ms, 2.0 * 512 * 512 * 9 * 32 * 32 * chars


def dram_traffic(chars):
    """roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from an `ncu --set
    full` capture of the CURRENT kernel build summarised in profiles/r2_tc2_dram.json by profiles/summarize_ncu.py (never a
    literal; null when no capture of this build exists)."""
    path = os.path.join(ROOT, "profiles", "r2_tc2_dram.json")
    try:
        d = json.load(open(path))
        if int(d.get("chars", -1)) == int(chars):
            return {"traffic": float(d["dram_bytes_per_launch"]), "traffic_source": "profiles/r2_tc2_dram.json (" + d.get("capture", "ncu --set full") + ")"}
    except Exception:
        pass
    return {"traffic": None}


def modconv_roofline(tspgan, chars, dev, iters=20):
    """Live CUDA-event timing of the dominant kernel: the 3x3 modulated conv 512->512 at 32x32 for `chars`
    characters (reference networks.py:294,299 grouped conv; 4.83 GFLOP per character and launch)."""
    from marconet_b200 import ops
    peaks = load_peaks()
    gen = tspgan.TextGenerator
    pk = gen._get_packed(dev)
    e = pk["styled"][6]                                   # convs.5: 512->512 @ 32x32, no upsample
    ms, flops = _time_modconv(e, chars, dev, iters)
    achieved = flops / (ms * 1e-3) / 1e12
    ms_big, flops_big = _time_modconv(e, 128, dev, 5)     # same kernel with 128 characters: 27.7 waves instead of 3.46
    big = flops_big / (ms_big * 1e-3) / 1e12
    passes = {0: 0, 1: 3, 2: 3, 3: 1}[ops.default_precision()]
    return {"kernel": "mn_conv2d_nhwc modulated 3x3 512->512 @32x32 x%d chars (conv_tc2_kernel<128>)" % chars, "bound": "tensor",
            "achieved": achieved, "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": achieved / peaks["tf_burst"],
            **dram_traffic(chars),
            "algorithmic_gflop_per_launch": flops / 1e9, "ms_per_launch": ms,
            "mma_passes_per_algorithmic_flop": passes,
            "tensor_pipe_frac": (achieved * passes / peaks["tf_burst"]) if passes else 0.0,
            "same_kernel_128_chars": {"achieved": big, "frac": big / peaks["tf_burst"], "ms_per_launch": ms_big,
                                      "tensor_pipe_frac": (big * passes / peaks["tf_burst"]) if passes else 0.0},
            "peak_source": peaks["source"] + ", bf16 dense burst (kernel timed alone, L2 flushed between launches); "
                           "fp32-grade products cost 3 fp16 MMAs each, so the ceiling of this kernel is peak/3 in algorithmic terms"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--lines", type=int, default=1, help="LR lines per GPU per step")
    ap.add_argument("--chars", type=int, default=16)
    ap.add_argument("--precision", type=int, default=None, help="0 fp32 CUDA-core, 1 fp16x3 tcgen05 (default), 2 bf16x3, 3 fp16x1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-collective", action="store_true", help="skip the character-sharded configs[2]/[3] sub-records")
    ap.add_argument("--no-graph", action="store_true", help="skip the CUDA-graph replay measurement (value = eager module calls)")
    ap.add_argument("--profile", action="store_true", help="run one step inside cudaProfilerStart/Stop and exit (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the SR images of rank 0's last timed step as DIR/sr.npy (float32, "
                         "lines x 3 x 128 x 2048; a seeded sample of its values when that exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
