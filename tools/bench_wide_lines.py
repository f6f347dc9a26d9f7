"""Wide-line throughput: GraphedLines(width=Wsr) replay and pipeline.restore_wide_image end to end, for LR widths
Wr in {512, 1024, 2048, 4096} with 16 characters per 512 columns (DESIGN.md "Wide lines").

    python tools/bench_wide_lines.py --out profiles/wide_lines_b200.json [--widths 512,1024,2048,4096] [--repeats 5]

Method: every shape is warmed up first (module graphs recorded, allocator sized); each timed window replays / calls back to
back for at least --window seconds between two CUDA events (the end event is synchronised); --repeats windows per shape give
the median and the spread.  No L2 flush between lines: consecutive lines, as a user restoring a page runs them.  The device
name and its power limit are read in the same run.  Synthetic checkpoints (marconet_b200.testing.synth): the arithmetic and
the shapes are those of the released models.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marconet_b200 import pipeline  # noqa: E402
from marconet_b200.graph import GraphedLines  # noqa: E402
from marconet_b200.models import networks  # noqa: E402
from marconet_b200.testing import synth  # noqa: E402


def device_info(dev):
    info = dict(name=torch.cuda.get_device_name(dev))
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", str(dev.index or 0)], capture_output=True, text=True, timeout=10).stdout.strip()
        pl, mx = [v.strip() for v in out.split(",")[:2]]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(mx))
    except Exception as exc:                         # the number is reported as unknown, never guessed
        info.update(power_limit_w=None, sm_max_mhz=None, query_error=repr(exc))
    return info


def timed_windows(fn, dev, window_s, repeats):
    """ms per call: calls back to back between two CUDA events for >= window_s seconds, ``repeats`` times."""
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize(dev)
    calls = max(3, int(window_s / max(time.perf_counter() - t0, 1e-4)) + 1)
    out = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if ms < window_s * 1e3:                      # window came out short: grow it and measure again
            calls = int(calls * window_s * 1e3 / ms) + 1
            e0.record()
            for _ in range(calls):
                fn()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
        out.append(ms / calls)
    return dict(ms=float(np.median(out)), ms_min=float(min(out)), ms_max=float(max(out)), calls_per_window=calls,
                window_s=float(ms / 1e3), repeats=repeats)


def line_inputs(wr, chars, seed):
    """An h = 32, w = Wr uint8 line (so the LQ width is Wr) with ``chars`` evenly spaced boxes and labels."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (32, wr, 3), dtype=np.uint8)
    pitch = wr / chars
    boxes = [[pitch * i + 2, 2, pitch * (i + 1) - 2, 30] for i in range(chars)]
    labels = synth.make_labels(chars, seed).reshape(-1).tolist()
    return img, labels, boxes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--widths", default="512,1024,2048,4096")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide_lines: no CUDA device (this measures the B200 kernels; there is no CPU path)")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sds = synth.make_checkpoints(0)
    mods = {}
    for key, cls in (("tspgan", networks.TSPGAN), ("encoder", networks.TextContextEncoderV2), ("sr", networks.TSPSRNet)):
        m = cls()
        m.load_state_dict(sds[key], strict=True)
        mods[key] = m.eval().to(dev)
    enc, gen, sr = mods["encoder"], mods["tspgan"], mods["sr"]
    rows = []
    for wr in [int(v) for v in args.widths.split(",")]:
        chars = 16 * wr // 512
        img, labels, boxes = line_inputs(wr, chars, wr)
        geo = pipeline.wide_geometry(32, wr)
        wsr = geo.canvas_width
        row = dict(lq_width=wr, canvas_width=wsr, segments=geo.segments, chars=chars)
        # graph replay: the inputs of the same line loaded once (a page of lines would load each one; the load is three copies)
        with torch.no_grad():
            res = pipeline.restore_wide_image(enc, gen, sr, img, labels, boxes)
        gl = GraphedLines(enc, gen, sr, lines=1, chars=chars, width=wsr, device=dev)
        gl.load(res["lq"], torch.tensor(labels).reshape(-1, 1), res["locs"])
        for _ in range(3):
            gl.replay()
        gl.check()
        g = timed_windows(gl.replay, dev, args.window, args.repeats)
        gl.check()
        row["graph"] = dict(g, chars_per_s=chars / (g["ms"] / 1e3), chars_per_s_min=chars / (g["ms_max"] / 1e3),
                            chars_per_s_max=chars / (g["ms_min"] / 1e3), launches=gl.launches)
        del gl
        # end to end from the host uint8 image (module graphs warm: the second call of a signature records, later ones replay)
        for _ in range(3):
            pipeline.restore_wide_image(enc, gen, sr, img, labels, boxes)
        e = timed_windows(lambda: pipeline.restore_wide_image(enc, gen, sr, img, labels, boxes), dev, args.window, args.repeats)
        row["restore_wide_image"] = dict(e, chars_per_s=chars / (e["ms"] / 1e3), chars_per_s_min=chars / (e["ms_max"] / 1e3),
                                         chars_per_s_max=chars / (e["ms_min"] / 1e3))
        print(json.dumps(row), flush=True)
        rows.append(row)
        torch.cuda.empty_cache()
    out = dict(tool="tools/bench_wide_lines.py", device=device_info(dev), torch=torch.__version__, cuda=torch.version.cuda,
               method=f"CUDA events, >= {args.window} s windows, {args.repeats} windows per shape (median, min, max), shapes warmed "
                      f"up first, no L2 flush between lines", rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["device"]))


if __name__ == "__main__":
    main()
