#!/usr/bin/env python
"""K1 launch-boundary probe: what one more back-to-back launch of the dequant kernel costs, per Flux shape and qtype.

For every (qtype, shape) of the bench.py sweep (plus one 1 GB-output reference shape, [172032, 3072]) it captures CUDA graphs
of n = 1, 2, 4, 8 launches (fp16 math, fp16 out, GGUFB200_DEQUANT_SRC_STABLE, programmatic dependent launch), each launch on
its OWN copy of the packed tensor into its own output (a re-read of the same packed bytes could come from L2), and times
replays of each graph with CUDA events.  A least-squares line T(n) = slope * n + intercept gives
    slope      the time one more launch adds inside a graph, its boundary to the next launch included
    intercept  the fixed cost of a replay (graph start, first ramp, last drain)
    boundary   slope - bytes / R, R = the streaming rate of the reference shape's slope for the same qtype
and the 35-launch step of bench.py (one graph, 5 qtypes x 7 shapes) is timed the same way.

--variants "3=0;3=1" times every figure once per ggufb200_set_tuning setting (needs GGUFB200_ALLOW_TUNING=1, set here),
alternating the settings round by round inside one process.  --trace DIR instead records ONE replay of the 35-launch graph
with torch.profiler per variant and prints each kernel's start / end and the gap to the previous kernel (negative = overlap).

    python tools/probe_k1_boundary.py [--variants "3=0;3=1"] [--rounds 3] [--qtypes Q4_0,Q4_K] [--trace DIR]
"""
import argparse
import json
import os
import sys

os.environ.setdefault("GGUFB200_ALLOW_TUNING", "1")

import numpy as np  # noqa: E402
import torch  # noqa: E402
import gguf  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402
import oracle  # noqa: E402
from bench import FLUX_SHAPES, QTYPES  # noqa: E402

REF_SHAPE = (172032, 3072)
NS = (1, 2, 4, 8)


def parse_variants(s):
    out = []
    for v in filter(None, s.split(";")):
        out.append([(int(kv.split("=")[0]), int(kv.split("=")[1])) for kv in filter(None, v.split(","))])
    return out or [[]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", default="")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--qtypes", default=",".join(QTYPES))
    ap.add_argument("--min-ms", type=float, default=20.0, help="GPU time per timed measurement")
    ap.add_argument("--trace", metavar="DIR", help="profile one replay of the 35-launch step per variant instead")
    args = ap.parse_args()

    lib = ge._sub("_lib")
    L = lib.lib()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    variants = parse_variants(args.variants)
    side = torch.cuda.Stream(dev)
    print(json.dumps({"device": torch.cuda.get_device_name(dev), "variants": [dict(v) for v in variants]}), flush=True)

    def set_variant(v):
        for k, val in v:
            if L.ggufb200_set_tuning(k, val) != 0:
                raise RuntimeError(f"tuning {k}={val} refused")

    def packed_for(qname, shape, seed):
        qt = gguf.GGMLQuantizationType[qname]
        bs, ts = gguf.GGML_QUANT_SIZES[qt]
        N, K = shape
        n_blocks = N * K // bs
        chunk = min(n_blocks, 1 << 15)
        raw = torch.from_numpy(oracle.random_blocks(int(qt), chunk, seed=seed))
        reps = (n_blocks + chunk - 1) // chunk
        return qt, n_blocks, raw.repeat(reps, 1)[:n_blocks].contiguous().to(dev), n_blocks * ts + N * K * 2

    def graph_of(items):
        """items = [(qt, n_blocks, packed, out)]; launches captured on `side`, the same way bench.py captures its step."""
        def run(st):
            for qt, nb, p, o in items:
                rc = L.ggufb200_dequant(int(qt), p.data_ptr(), nb, o.data_ptr(), 0, lib.DEQUANT_SRC_STABLE, st)
                if rc != 0:
                    raise RuntimeError(f"ggufb200_dequant rc={rc}")
        with torch.cuda.stream(side):
            run(side.cuda_stream)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                run(side.cuda_stream)
        return g

    def time_graph(g, est_us):
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        reps = max(5, int(args.min_ms * 1e3 / max(est_us, 1.0)))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e3       # us per replay

    # ---------------- the 35-launch step of bench.py
    step_items, step_bytes = [], 0
    for qi, q in enumerate(QTYPES):
        for si, shape in enumerate(FLUX_SHAPES):
            qt, nb, p, by = packed_for(q, shape, 100 * qi + si)
            step_items.append((qt, nb, p, torch.empty(shape, dtype=torch.float16, device=dev)))
            step_bytes += by
    if args.trace:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.trace, exist_ok=True)
        for vi, v in enumerate(variants):
            set_variant(v)
            g = graph_of(step_items)
            for _ in range(5):
                g.replay()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                g.replay()
                torch.cuda.synchronize()
            path = os.path.join(args.trace, f"k1_step_variant{vi}.pt.trace.json")
            prof.export_chrome_trace(path)
            ev = [e for e in json.load(open(path))["traceEvents"] if e.get("cat") == "kernel"]
            ev.sort(key=lambda e: e["ts"])
            print(f"# variant {dict(v)}: {len(ev)} kernels, first start -> last end "
                  f"{ev[-1]['ts'] + ev[-1]['dur'] - ev[0]['ts']:.1f} us", flush=True)
            prev_end = None
            for i, e in enumerate(ev):
                q, (N, K) = QTYPES[i // len(FLUX_SHAPES)], FLUX_SHAPES[i % len(FLUX_SHAPES)]
                gap = "" if prev_end is None else f"{e['ts'] - prev_end:8.2f}"
                print(f"{i:3d} {q:5s} [{N},{K}]  start {e['ts'] - ev[0]['ts']:9.2f}  dur {e['dur']:8.2f}  gap {gap}", flush=True)
                prev_end = e["ts"] + e["dur"]
            del g
        return

    step_graphs = []
    for v in variants:
        set_variant(v)
        step_graphs.append(graph_of(step_items))
    step_us = [[] for _ in variants]
    for _ in range(args.rounds):
        for vi, v in enumerate(variants):
            set_variant(v)
            step_us[vi].append(time_graph(step_graphs[vi], 600.0))
    for vi, v in enumerate(variants):
        us = float(np.median(step_us[vi]))
        print(json.dumps({"what": "step35", "variant": dict(v), "us": us, "GB/s": step_bytes / us / 1e3,
                          "us_rounds": step_us[vi]}), flush=True)
    del step_graphs, step_items
    torch.cuda.empty_cache()

    # ---------------- graphs of n back-to-back launches per (qtype, shape)
    for qi, q in enumerate(filter(None, args.qtypes.split(","))):
        rate = {}
        for shape in [REF_SHAPE] + FLUX_SHAPES:
            qt, nb, p, by = packed_for(q, shape, 7 + qi)
            copies = [p] + [p.clone() for _ in range(max(NS) - 1)]
            outs = [torch.empty(shape, dtype=torch.float16, device=dev) for _ in range(max(NS))]
            est = by / 6.5e3                                           # us at ~6.5 TB/s
            t = {vi: {n: [] for n in NS} for vi in range(len(variants))}
            graphs = {}
            for vi, v in enumerate(variants):
                set_variant(v)
                for n in NS:
                    graphs[vi, n] = graph_of([(qt, nb, copies[i], outs[i]) for i in range(n)])
            for _ in range(args.rounds):
                for vi, v in enumerate(variants):
                    set_variant(v)
                    for n in NS:
                        t[vi][n].append(time_graph(graphs[vi, n], est * n))
            for vi, v in enumerate(variants):
                ys = np.array([np.median(t[vi][n]) for n in NS])
                slope, icpt = np.polyfit(np.array(NS, dtype=float), ys, 1)
                if shape == REF_SHAPE:
                    rate[vi] = by / slope
                rec = {"what": "b2b", "q": q, "shape": list(shape), "variant": dict(v), "bytes": by,
                       "us_per_replay": {n: float(y) for n, y in zip(NS, ys)}, "slope_us": float(slope), "intercept_us": float(icpt),
                       "slope_GB/s": by / slope / 1e3, "boundary_us": float(slope - by / rate[vi])}
                print(json.dumps(rec), flush=True)
            del graphs, copies, outs, p
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
