#!/usr/bin/env python
"""Seconds per explained query: a loop of ``Explainer(...).run(e)`` against one ``Explainer(...).run_batch(elements)``.

Workloads (the graphs bench.py's query leg uses): the C1 and C2 fixture graphs, the 1/10-scale C3 k-hop query graph and
median-degree / hub queries of the R-MAT 1 M / 20 M graph.  For every batch size: the first call and the warm median, and
a per-phase split from a separate pass in which every NVTX range of run / run_batch is closed by a device synchronise and
timed on the host (flatten, khop, communities, engine_build, masks, masked_forward, fit, aggregate).  The GPU name and
power limit are read in the same run.

  python tools/explain_batch.py --sizes 1,8,64 --out profiles/explain_batch.json
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import defaultdict

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload builders of the query leg)


class PhaseTimer:
    """Host seconds per NVTX range name (last component), each range closed by a device synchronise."""

    def __init__(self):
        self.sec = defaultdict(float)
        self._stack = []
        self._push, self._pop = torch.cuda.nvtx.range_push, torch.cuda.nvtx.range_pop

    def __enter__(self):
        def push(name):
            torch.cuda.synchronize()
            self._stack.append((name.split(":")[-1], time.perf_counter()))
            return self._push(name)

        def pop():
            torch.cuda.synchronize()
            name, t0 = self._stack.pop()
            self.sec[name] += time.perf_counter() - t0
            return self._pop()

        torch.cuda.nvtx.range_push, torch.cuda.nvtx.range_pop = push, pop
        return self

    def __exit__(self, *exc):
        torch.cuda.nvtx.range_push, torch.cuda.nvtx.range_pop = self._push, self._pop


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def workloads(which):
    """name -> (make_explainer, candidate elements in order of use)."""
    from bikg_graph_explainability_public_b200 import Explainer

    out = {}
    for key, case_name in (("c1", "c1_homo_gcn"), ("c2", "c2_hetero_gcn")):
        if key not in which:
            continue
        case, arch, _f, _e, names, _p, _pn = bench._golden_case_inputs(case_name)
        meta = case["meta"]
        flat = names if isinstance(names, list) else list(names.values())[0]

        def mk(meta=meta, case_name=case_name, arch=arch):
            _c, _a, f, e, nm, pw, pn = bench._golden_case_inputs(case_name)
            return Explainer(f, e, arch, dict(meta["params"]), nm, pw, pn, meta["element_type"], meta["problem"])

        out[key] = (mk, [flat[(flat.index(meta["element"]) + 5 * i) % len(flat)] for i in range(64)])
    if "c3_tenth" in which:
        wl, names, pathways, pnames = bench._tenth_query_inputs()
        arch = wl.make_model()
        g = torch.Generator().manual_seed(5)

        def mk(wl=wl, names=names, pathways=pathways, pnames=pnames, arch=arch):
            return Explainer(wl.x.clone(), wl.ei.clone(), arch, dict(bench.QUERY_PARAMS), list(names),
                             [list(p) for p in pathways], list(pnames))

        out["c3_tenth"] = (mk, [names[wl.queries[0]]] + [names[i] for i in torch.randint(0, wl.n, (63,), generator=g).tolist()])
    if "rmat_median" in which or "rmat_hub" in which:
        wl = bench.Workload("c3_rmat")
        names, pathways, pnames = bench._named_communities(wl)
        arch = wl.make_model()
        indeg = torch.bincount(wl.ei[1], minlength=wl.n)
        srt = torch.argsort(indeg, stable=True)

        def mk(wl=wl, names=names, pathways=pathways, pnames=pnames, arch=arch):
            return Explainer(wl.x, wl.ei, arch, dict(bench.QUERY_PARAMS), list(names), [list(p) for p in pathways],
                             list(pnames))

        mid = wl.n // 2
        if "rmat_median" in which:
            out["rmat_median"] = (mk, [names[i] for i in srt[mid - 32: mid + 32].tolist()])
        if "rmat_hub" in which:
            out["rmat_hub"] = (mk, [names[i] for i in srt.flip(0)[:64].tolist()])
    return out


def time_sequential(mk, els):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for e in els:
        mk().run(e, 1)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def time_batch(mk, els):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mk().run_batch(els, 1)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c1,c2,c3_tenth,rmat_median,rmat_hub")
    ap.add_argument("--sizes", default="1,8,64")
    ap.add_argument("--repeats", type=int, default=3, help="calls per arm and size: the first, then the warm median")
    ap.add_argument("--max-seq-seconds", type=float, default=90.0,
                    help="skip the warm repeats of an arm whose first call took longer (large hub batches)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.init()
    dev = torch.cuda.current_device()
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(dev), "torch": torch.__version__, "results": {}}
    sizes = [int(s) for s in args.sizes.split(",")]
    for name, (mk, cands) in workloads(args.workloads.split(",")).items():
        mk().run(cands[0], 1)  # warm-up: library load, kernel images, allocator
        for b in sizes:
            els = cands[:b]
            row = {}
            for arm, fn in (("sequential", time_sequential), ("run_batch", time_batch)):
                ts = [fn(mk, els)]
                while len(ts) < args.repeats and ts[0] < args.max_seq_seconds:
                    ts.append(fn(mk, els))
                with PhaseTimer() as pt:
                    fn(mk, els)
                row[arm] = {"first_s_per_query": ts[0] / b,
                            "warm_s_per_query": float(np.median(ts[1:])) / b if len(ts) > 1 else None,
                            "phase_s_per_query": {k: v / b for k, v in sorted(pt.sec.items())}}
            w = row["run_batch"]["warm_s_per_query"] or row["run_batch"]["first_s_per_query"]
            s = row["sequential"]["warm_s_per_query"] or row["sequential"]["first_s_per_query"]
            row["speedup"] = s / w
            res["results"]["%s/b%d" % (name, b)] = row
            print(json.dumps({"workload": name, "batch": b, **row}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "device": res["device"]}))


if __name__ == "__main__":
    main()
