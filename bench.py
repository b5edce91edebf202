#!/usr/bin/env python
"""Benchmark of the perturbation hot path (BASELINE.json metric: coalition evals/s + masked GTEPS at 1/2/4/8 B200;
s per explained query).

Workload (config.workload = "c3"): BASELINE.json configs[2] -- synthetic homogeneous graph, 1 M nodes / 20 M edges
(uniform), 2 x GCNConv(128) + Linear(128 -> 1), 500 disjoint communities, 4096 coalitions, whole-graph computational
graph, every conv layer over the whole graph ("full" mode = the work the reference does; the engine only materialises,
per coalition, the rows of its ACTIVE nodes -- an inactive node has no active in-edge, so its row is coalition
invariant and never gathered).
A step = one pass of the hot path over the 4096-coalition job.  Strong scaling: the job is fixed, rank r evaluates
coalitions [r * 4096 / N, (r + 1) * 4096 / N) and one all-gather collects the predictions -- at N = 8 a step IS the
north star's "4096-coalition explanation on 8 x B200".  (`--coalitions-per-gpu K` switches to weak scaling.)

value   : coalition evals/s, graph / weights / packed coalition bits resident in HBM, CUDA-event timed, max over ranks.
e2e     : same metric through the C ABI with HOST buffers: the packed coalition matrix (N x W words, the input format of
          xpgnn_forward) in pinned host memory -> H2D -> masked forward -> all-gather -> D2H of the predictions, all timed.
roofline: masked SpMM on coalition-specific activations (layers >= 1; cspmm_seg_kernel of csrc/compact.cu), algorithmic
          bytes per launch (SURVEY.md 8d: 32 coalition-layers x 1.108 GB) / CUDA-event kernel time measured live via
          xpgnn_profile (events on the launching stream); traffic from the committed ncu capture (profiles/traffic.json).
s_per_explained_query: wall time of Explainer(...).run(q, 1) through the drop-in API -- C1 and C2 (the reference's toy
          cases), a k-hop query on the 1/10-scale C3 graph, and hub / median / leaf queries on the R-MAT 1 M / 20 M graph --
          next to the UNMODIFIED reference (oracle/_ref, staged by oracle/stage_ref.py) on the host cores where it can run.
cpu_baseline / --impl reference: the unmodified reference's kernel_output (perturbator + Model.infer; PyG layers from the
          CPU stand-in because torch_geometric is absent) on the host cores, bounded sample; the oracle port when the staged
          reference is missing.  The parity check of the run: exit code 3 when GPU and CPU disagree beyond the bar.
--dump-outputs DIR: the predictions of the last timed step as DIR/predictions.npy, coalition rows x queries (inputs are
          seeded: equal arguments give equal inputs, so two builds can be compared output for output).  --impl reference
          evaluates the first query only, so its file has one column.
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
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[2]: the configuration the metric is quoted on
    "c3": dict(kind="homo_gcn", nodes=1_000_000, edges=20_000_000, features=128, hidden=128, communities=500),
    # R-MAT(0.57, 0.19, 0.19, 0.05) variant of C3: hub rows (SURVEY.md 8d)
    "c3_rmat": dict(kind="homo_gcn", nodes=1_000_000, edges=20_000_000, features=128, hidden=128, communities=500, rmat=True),
    # configs[3]: biomedical-KG shape, 5 node types / 20 relations, 2 x HeteroConv(SAGEConv mean, sum)
    "c4": dict(kind="hetero_sage", nodes=2_000_000, edges=50_000_000, features=64, hidden=128, communities=1000,
               type_frac=(0.4, 0.25, 0.15, 0.1, 0.1), relations=20),
    # configs[4]: scale sweep graph, 64 batched query nodes
    "c5": dict(kind="homo_gcn", nodes=5_000_000, edges=100_000_000, features=128, hidden=128, communities=500, queries=64),
    # configs[1] at scale (SURVEY.md 8d): ONE node type, 3 relations (edges round-robin), HeteroConv(GCNConv) + MLP head
    "c2_100k": dict(kind="hetero_gcn1", nodes=100_000, edges=2_000_000, features=84, hidden=16, communities=50, relations=3),
    # C3 with 10 % of the nodes in a second community (overlapping communities, SURVEY.md 8d)
    "c3_overlap": dict(kind="homo_gcn", nodes=1_000_000, edges=20_000_000, features=128, hidden=128, communities=500, overlap=0.1),
    # half of C3 at the same degree: its per-pass gather working set is 32 MB instead of 64 MB (L2 experiment, profiles/r02_summary.md)
    "c3_half": dict(kind="homo_gcn", nodes=500_000, edges=10_000_000, features=128, hidden=128, communities=250),
    "c3_tenth": dict(kind="homo_gcn", nodes=100_000, edges=2_000_000, features=128, hidden=128, communities=50),
    "c4_small": dict(kind="hetero_sage", nodes=40_000, edges=1_000_000, features=64, hidden=128, communities=40,
                     type_frac=(0.4, 0.25, 0.15, 0.1, 0.1), relations=20),
    "c4_tiny": dict(kind="hetero_sage", nodes=3_000, edges=40_000, features=32, hidden=64, communities=12,
                    type_frac=(0.4, 0.25, 0.15, 0.1, 0.1), relations=9),
    "c2_wide": dict(kind="hetero_gcn1", nodes=2_500, edges=30_000, features=40, hidden=64, communities=10, relations=3),
    "c2_wide2": dict(kind="hetero_gcn1", nodes=2_500, edges=30_000, features=40, hidden=64, communities=10, relations=3, conv_layers=2),
    "tiny": dict(kind="homo_gcn", nodes=20_000, edges=400_000, features=32, hidden=32, communities=20),
}


def rmat_edges(n, e, g, a=0.57, b=0.19, c=0.19):
    bits = int(np.ceil(np.log2(n)))
    src = torch.zeros(e, dtype=torch.int64)
    dst = torch.zeros(e, dtype=torch.int64)
    for _ in range(bits):
        r = torch.rand(e, generator=g)
        src = src * 2 + (r >= a + b).to(torch.int64)                                # quadrants c, d
        dst = dst * 2 + (((r >= a) & (r < a + b)) | (r >= a + b + c)).to(torch.int64)  # quadrants b, d
    return torch.stack([src % n, dst % n])


class Workload:
    """Synthetic inputs of one BASELINE.json configuration (SURVEY.md 8d), flattened to one node id space."""

    def __init__(self, name):
        w = WORKLOADS[name]
        self.name, self.kind = name, w["kind"]
        self.n, self.e, self.f, self.h, self.c = w["nodes"], w["edges"], w["features"], w["hidden"], w["communities"]
        n, e = self.n, self.e
        g = torch.Generator().manual_seed(1234)
        self.type_ptr, self.node_type_names, self.edge_type, self.edge_type_names, self.node_type = [0, n], None, None, None, None
        self.com_of2 = None  # optional second community of a node (overlapping communities)
        if self.kind == "hetero_gcn1":
            self.ei = torch.randint(0, n, (2, e), generator=g)
            self.x = torch.randn(n, self.f, generator=g)
            self.com_of = torch.randperm(n, generator=g) % self.c
            self.node_type_names = ["gene"]
            self.edge_type_names = [("gene", "rel%d" % i, "gene") for i in range(w["relations"])]
            self.edge_type = torch.arange(e, dtype=torch.int64) % w["relations"]
            self.node_type = torch.zeros(n, dtype=torch.float32)
            self.out_type = "gene"
            self.q_in_type = 17
            self.queries = [17]
            self.conv_layers = w.get("conv_layers", 1)
        elif self.kind == "homo_gcn":
            self.ei = rmat_edges(n, e, g) if w.get("rmat") else torch.randint(0, n, (2, e), generator=g)
            self.x = torch.randn(n, self.f, generator=g)
            self.com_of = torch.randperm(n, generator=g) % self.c  # c disjoint, equal communities
            if w.get("overlap"):
                extra = torch.rand(n, generator=g) < w["overlap"]
                second = torch.randint(0, self.c, (n,), generator=g)
                self.com_of2 = torch.where(extra, second, torch.full((n,), -1, dtype=torch.int64))
            q0 = 17
            nq = w.get("queries", 1)
            self.queries = [q0] if nq == 1 else torch.randperm(n, generator=g)[:nq].tolist()
            self.q_in_type = self.queries[0]
        else:
            counts = [int(fr * n) for fr in w["type_frac"]]
            counts[0] += n - sum(counts)
            self.type_ptr = [0]
            for cnt in counts:
                self.type_ptr.append(self.type_ptr[-1] + cnt)
            t = len(counts)
            self.node_type_names = ["t%d" % i for i in range(t)]
            pairs = [(i, i) for i in range(min(4, t))]  # >= 4 same-type relations
            while len(pairs) < w["relations"]:
                pairs.append((int(torch.randint(0, t, (1,), generator=g)), int(torch.randint(0, t, (1,), generator=g))))
            self.edge_type_names = [("t%d" % a_, "rel%d" % i, "t%d" % b_) for i, (a_, b_) in enumerate(pairs)]
            per = e // len(pairs)
            eis, ets = [], []
            for i, (a_, b_) in enumerate(pairs):
                src = torch.randint(self.type_ptr[a_], self.type_ptr[a_ + 1], (per,), generator=g)
                dst = torch.randint(self.type_ptr[b_], self.type_ptr[b_ + 1], (per,), generator=g)
                eis.append(torch.stack([src, dst]))
                ets.append(torch.full((per,), i, dtype=torch.int64))
            self.ei, self.edge_type = torch.cat(eis, 1), torch.cat(ets)
            self.e = int(self.ei.shape[1])
            self.x = torch.randn(n, self.f, generator=g)
            self.node_type = torch.cat([torch.full((cnt,), i, dtype=torch.float32) for i, cnt in enumerate(counts)])
            # type-pure communities (the reference assumes them, README.md:218), sized by type
            per_type = [max(1, round(self.c * cnt / n)) for cnt in counts]
            per_type[0] += self.c - sum(per_type)
            com_of, base = [], 0
            for cnt, k in zip(counts, per_type):
                com_of.append(base + torch.randperm(cnt, generator=g) % k)
                base += k
            self.com_of = torch.cat(com_of)
            self.out_type = "t0"
            self.q_in_type = 17
            self.queries = [self.type_ptr[0] + self.q_in_type]

    @property
    def model_name(self):
        if self.kind == "homo_gcn":
            return "2xGCNConv(%d)+Linear(%d,1)" % (self.h, self.h)
        if self.kind == "hetero_gcn1":
            return "HeteroConv(%d x GCNConv(%d), sum)+MLP(%d-16-32-1)+Sigmoid" % (len(self.edge_type_names), self.h, self.h)
        return "2xHeteroConv(%d x SAGEConv(%d, mean), sum)+Linear(%d,1)+Sigmoid" % (len(self.edge_type_names), self.h, self.h)

    def make_model(self, seed=7):
        """Product-side weight containers (state-dict keys of the PyG layers)."""
        from torch import nn

        from bikg_graph_explainability_public_b200 import nn as xnn

        torch.manual_seed(seed)
        f, h, wl = self.f, self.h, self

        class GCN2(nn.Module):
            def __init__(self):
                super().__init__()
                self.conv = nn.ModuleList([xnn.GCNConv(f, h), nn.ReLU(), xnn.GCNConv(h, h), nn.ReLU()])
                self.fc = nn.ModuleList([xnn.Linear(h, 1)])

        class HeteroSAGE2(nn.Module):
            def __init__(self):
                super().__init__()
                self.out_type = wl.out_type
                self.conv = nn.ModuleList([
                    xnn.HeteroConv({r: xnn.SAGEConv((f, f), h) for r in wl.edge_type_names}), nn.ReLU(),
                    xnn.HeteroConv({r: xnn.SAGEConv((h, h), h) for r in wl.edge_type_names}), nn.ReLU()])
                self.fc = nn.ModuleList([xnn.Linear(h, 1), nn.Sigmoid()])

        class HeteroGCN1(nn.Module):
            def __init__(self):
                super().__init__()
                mods = []
                for li in range(wl.conv_layers):
                    mods += [xnn.HeteroConv({r: xnn.GCNConv(f if li == 0 else h, h) for r in wl.edge_type_names}), nn.ReLU()]
                self.conv = nn.ModuleList(mods)
                self.fc = nn.ModuleList([xnn.Linear(h, 16), nn.ReLU(), xnn.Linear(16, 32), nn.ReLU(), xnn.Linear(32, 1), nn.Sigmoid()])

        return {"homo_gcn": GCN2, "hetero_sage": HeteroSAGE2, "hetero_gcn1": HeteroGCN1}[self.kind]().eval()

    def oracle_model(self, arch):
        """Same weights in the oracle's CPU stand-in layers (for the CPU baseline / parity check)."""
        from oracle import fixture_models as fm

        if self.kind == "homo_gcn":
            m = fm.HomoGCN(self.f, (self.h, self.h), (self.h, 1), final_sigmoid=False)
        elif self.kind == "hetero_gcn1":
            m = fm.HeteroGCNSingleType(self.f, self.edge_type_names, conv_dims=(self.h,) * self.conv_layers,
                                       head_dims=(self.h, 16, 32, 1))
        else:
            m = fm.HeteroSAGE({t: self.f for t in self.node_type_names}, self.edge_type_names, self.out_type,
                              conv_dims=(self.h, self.h), head_dims=(self.h, 1))
        m.load_state_dict(arch.state_dict())
        return m.eval()

    def oracle_eval(self, om, mask_bool_np):
        """Reference algorithm (oracle port) on the host: query prediction of every coalition row of ``mask``."""
        from oracle.xpgnn_oracle import kernel_output

        if self.kind == "homo_gcn":
            _, y = kernel_output(mask_bool_np, self.x, self.ei.numpy(), om, self.queries[0])
        else:
            _, y = kernel_output(mask_bool_np, self.x, self.ei.numpy(), om, self.q_in_type, node_type=self.node_type,
                                 edge_type=self.edge_type.numpy(), node_type_names=self.node_type_names,
                                 edge_type_names=self.edge_type_names, padded_dims=[0] * len(self.node_type_names))
        return y.numpy().reshape(-1)

    def engine(self, dev, precision):
        from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
        from bikg_graph_explainability_public_b200.lowering import lower

        arch = self.make_model()
        if self.kind == "homo_gcn":
            g = GraphSpec(self.x.to(dev), self.ei.to(dev), [0, self.n])
        else:
            g = GraphSpec(self.x.to(dev), self.ei.to(dev), self.type_ptr, self.node_type_names, self.edge_type.to(dev),
                          self.edge_type_names)
        eng = MaskedForward(g, lower(arch), self.queries, prune=False, precision=precision,
                            zero_edge_rule=self.kind == "hetero_sage")  # the zero-edge rule belongs to the multi-node-type branch
        return arch, eng


def make_masks(n_rows, n, c, com_of, seed, com_of2=None):
    """Coalition rows of the reference's family: row i perturbs community i mod C internally (iid node
    bits) and switches every other community on/off as a block (antithetic pairs).  Host version (tests, small runs)."""
    g = torch.Generator().manual_seed(seed)
    half = (n_rows + 1) // 2
    ext = torch.rand(half, c, generator=g) < 0.5
    ext = torch.cat([ext, ~ext])[:n_rows]
    mask = torch.empty((n_rows, n), dtype=torch.uint8)
    has2 = None if com_of2 is None else com_of2 >= 0
    for i in range(n_rows):
        row = ext[i][com_of]
        own = com_of == (i % c)
        if has2 is not None:  # overlapping communities: external activation is an OR over the memberships (masks.py:192),
            row[has2] |= ext[i][com_of2[has2]]  # internal bits overwrite shared nodes (masks.py:338)
            own = own | (com_of2 == (i % c))
        row[own] = torch.rand(int(own.sum()), generator=g) < 0.5
        mask[i] = row
    return mask


def make_packed_masks(lib, n_rows, n, c, com_of, seed, dev, com_of2=None, keep_rows=0):
    """The same row family generated ON THE DEVICE 64 rows at a time and packed into the engine's input format
    (``act[N][W]`` words, bit b of word w of node v = v active in coalition 32 w + b): a 4096 x 1 M job never exists as
    a 4 GB byte matrix.  Returns (act, the first ``keep_rows`` rows as a host bool matrix for the CPU parity sample)."""
    from bikg_graph_explainability_public_b200 import _lib

    g = torch.Generator(device=dev).manual_seed(seed)
    half = (n_rows + 1) // 2
    ext = torch.rand(half, c, generator=g, device=dev) < 0.5
    ext = torch.cat([ext, ~ext])[:n_rows]
    com = com_of.to(dev)
    com2 = None if com_of2 is None else com_of2.to(dev)
    w = -(-n_rows // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device=dev)
    kept = []
    for r0 in range(0, n_rows, 64):
        r1 = min(r0 + 64, n_rows)
        idx = torch.arange(r0, r1, device=dev)
        m = ext[r0:r1][:, com]
        own = com[None, :] == (idx % c)[:, None]
        if com2 is not None:
            has2 = com2 >= 0
            m = m | (ext[r0:r1][:, com2.clamp(min=0)] & has2[None, :])
            own = own | (com2[None, :] == (idx % c)[:, None])
        m = torch.where(own, torch.rand((r1 - r0, n), generator=g, device=dev) < 0.5, m).to(torch.uint8).contiguous()
        wc = -(-(r1 - r0) // 32)
        part = torch.zeros((n, wc), dtype=torch.int32, device=dev)
        _lib.check(lib.xpgnn_pack_mask(m.data_ptr(), r1 - r0, n, part.data_ptr(), wc, None, _lib.stream_ptr()))
        act[:, r0 // 32: r0 // 32 + wc] = part
        if r0 < keep_rows:
            kept.append(m[: max(0, min(keep_rows, r1) - r0)].bool().cpu())
    return act, (torch.cat(kept) if kept else None)


class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ the reference on the host cores
def _reference_modules():
    """The unmodified reference package (oracle/_ref staged copy, or /root/reference in the build container), else None."""
    try:
        from oracle import ref_harness

        if not ref_harness.reference_available():
            return None
        ref_harness.import_reference()
        import pathway_explanations.data as rdata
        import pathway_explanations.explainer as rexp
        import pathway_explanations.model as rmodel
        import pathway_explanations.wlm as rwlm

        return dict(data=rdata, model=rmodel, wlm=rwlm, explainer=rexp, src=ref_harness.REFERENCE_SRC)
    except Exception as ex:  # CUDA visible (cupy branch), staged copy missing, ...
        sys.stderr.write("[bench] unmodified reference not usable here: %r\n" % (ex,))
        return None


def host_eval(wl, om, mask_bool_np, ref=None):
    """Query prediction of every coalition row on the host.  With ``ref`` (homogeneous workloads): the unmodified
    reference's ``wlm.kernel_output`` = ``Data.perturbator`` + ``Model.infer`` + ``extract_node_edge_output``
    (wlm.py:283-436); else the oracle port of the same algorithm.  Returns (y, kind)."""
    if ref is not None and wl.kind == "homo_gcn":
        dc = ref["data"].Data(wl.x, wl.ei)
        mc = ref["model"].Model(om)
        _, y = ref["wlm"].kernel_output(torch.from_numpy(np.ascontiguousarray(mask_bool_np)), dc, mc, "node_prediction",
                                        wl.queries[0])
        return y.numpy().reshape(-1), "reference"
    return wl.oracle_eval(om, mask_bool_np), "port"


def _kind_note(kind):
    return ("unmodified reference wlm.kernel_output (perturbator + Model.infer), package imported from the staged copy "
            "oracle/_ref (or /root/reference in the build container); GCNConv arithmetic from the CPU stand-in of "
            "torch_geometric 2.0.4, which is not installed" if kind == "reference"
            else "oracle port of the reference's block-diagonal path (torch CPU)")


def run_reference(args, rank):
    """Reference arm: the reference's own CPU implementation of the path on the host cores, bounded sample per step."""
    if rank != 0:
        return
    wl = Workload(args.workload)
    torch.set_num_threads(os.cpu_count())
    ref = _reference_modules()
    om = wl.oracle_model(wl.make_model())
    b = args.ref_coalitions
    mask = make_masks(b * (args.steps + args.warmup), wl.n, wl.c, wl.com_of, 99, wl.com_of2).bool().numpy()
    times, kind = [], "port"
    for i in range(args.steps + args.warmup):
        t0 = time.perf_counter()
        y, kind = host_eval(wl, om, mask[i * b:(i + 1) * b], ref)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.reshape(y, (b, -1)))
    t = float(np.sum(times))
    value = b * len(times) / t
    line = {
        "impl": "reference", "metric": "coalition evals/s", "value": value, "unit": "coalition evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / len(times),
        "higher_is_better": True, "scaling": scaling_of(args), "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, wl, args.gpus),
        "masked_gteps": value * 2 * wl.e / 1e9,
        "cpu_baseline": {"value": value, "unit": "coalition evals/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": "%d coalitions per step of the full %s workload; %s" % (b, args.workload, _kind_note(kind))},
        "e2e": {"value": value, "unit": "coalition evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_query_leg and ref is not None:
        line["s_per_explained_query"] = query_leg_reference(ref)
    emit(line)


# ------------------------------------------------------------------------------------------ s per explained query
QUERY_PARAMS = {"interpret_samples": 20, "epochs": 50, "optimizer": "adam", "lr": 0.01, "l1_lambda": 1e-4, "lr_patience": 10,
                "seed": 1}  # the reference's config/configs.json with the toy cases' sample counts (tests/test_explainer.py)


def _golden_case_inputs(name):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import golden_io as gio

    case = gio.load_case(name)
    names, pathways, pnames = gio.fresh_inputs(case)
    if case["meta"]["hetero"]:
        feat = {k: v.clone() for k, v in case["feat"].items()}
        ei = {k: v.clone() for k, v in case["edge_index"].items()}
    else:
        feat, ei = case["feat"].clone(), case["edge_index"].clone()
    return case, gio.build_arch(case), feat, ei, names, pathways, pnames


def _tenth_query_inputs():
    """A k-hop query on the 1/10-scale C3 graph (100 k nodes / 2 M edges, 50 communities given as node indices)."""
    wl = Workload("c3_tenth")
    names, pathways, pnames = _named_communities(wl)
    return wl, names, pathways, pnames


def _named_communities(wl):
    """Node names ``str(i)`` and the workload's communities as lists of member NAMES (the reference's README usage)."""
    order = torch.argsort(wl.com_of, stable=True)
    bounds = torch.searchsorted(wl.com_of[order], torch.arange(wl.c + 1))
    names = [str(i) for i in range(wl.n)]
    pathways = [[names[i] for i in order[bounds[c]:bounds[c + 1]].tolist()] for c in range(wl.c)]
    return names, pathways, ["community_%d" % c for c in range(wl.c)]


def _time_runs(make_explainer, element, repeats=3):
    """Wall seconds of Explainer(...).run(element, 1), construction included; the first run (library load, CUDA context,
    kernel images) is reported separately from the warm median."""
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        ex = make_explainer()
        ex.run(element, 1)
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return {"first_s": ts[0], "warm_s": float(np.median(ts[1:])) if len(ts) > 1 else ts[0]}


def query_leg_reference(ref):
    """The unmodified reference's Explainer.run on the host cores: C1, C2 and the 1/10-scale C3 k-hop query."""
    out = {"cores": torch.get_num_threads(), "impl": "unmodified reference (oracle/_ref), PyG layers from the CPU stand-in"}
    RefExplainer = ref["explainer"].Explainer
    for key, name in (("c1", "c1_homo_gcn"), ("c2", "c2_hetero_gcn")):
        case, arch, feat, ei, names, pathways, pnames = _golden_case_inputs(name)
        meta = case["meta"]

        def mk(case=case, arch=arch, meta=meta, name=name):
            _c, _a, f, e, nm, pw, pn = _golden_case_inputs(name)
            return RefExplainer(f, e, arch, dict(meta["params"]), nm, pw, pn, meta["element_type"], meta["problem"])

        try:
            out[key] = _time_runs(mk, meta["element"])
        except Exception as ex:
            out[key] = {"error": repr(ex)}
    try:
        wl, names, pathways, pnames = _tenth_query_inputs()
        om = wl.oracle_model(wl.make_model())

        def mk2():
            return RefExplainer(wl.x.clone(), wl.ei.clone(), om, dict(QUERY_PARAMS), list(names), [list(p) for p in pathways], list(pnames))

        out["c3_tenth_khop"] = _time_runs(mk2, names[wl.queries[0]], repeats=2)
    except Exception as ex:
        out["c3_tenth_khop"] = {"error": repr(ex)}
    return out


def query_leg_ours(dev):
    """Explainer.run through the drop-in package on one GPU."""
    from bikg_graph_explainability_public_b200 import Explainer, _lib
    from bikg_graph_explainability_public_b200 import nn as xnn

    out = {"impl": "bikg_graph_explainability_public_b200.Explainer on cuda:%d (prune=True, fp32)" % dev.index}
    for key, name in (("c1", "c1_homo_gcn"), ("c2", "c2_hetero_gcn")):
        case, arch, feat, ei, names, pathways, pnames = _golden_case_inputs(name)
        meta = case["meta"]

        def mk(meta=meta, name=name, arch=arch):
            _c, _a, f, e, nm, pw, pn = _golden_case_inputs(name)
            return Explainer(f, e, arch, dict(meta["params"]), nm, pw, pn, meta["element_type"], meta["problem"])

        out[key] = _time_runs(mk, meta["element"], repeats=4)
    wl, names, pathways, pnames = _tenth_query_inputs()
    arch = wl.make_model()

    def mk2():
        return Explainer(wl.x.clone(), wl.ei.clone(), arch, dict(QUERY_PARAMS), list(names), [list(p) for p in pathways], list(pnames))

    out["c3_tenth_khop"] = _time_runs(mk2, names[wl.queries[0]])
    # R-MAT 1 M / 20 M (the realistic degree distribution): hub, median-degree and leaf query, 64 x 64 sample budget
    wl = Workload("c3_rmat")
    names, pathways, pnames = _named_communities(wl)
    arch = wl.make_model()
    indeg = torch.bincount(wl.ei[1], minlength=wl.n)
    srt = torch.argsort(indeg)
    qs = {"rmat_hub": int(srt[-1]), "rmat_median": int(srt[wl.n // 2]), "rmat_leaf": int(srt[0])}
    params = dict(QUERY_PARAMS, interpret_samples=64, epochs=64)
    x_dev, ei_dev = wl.x.to(dev), wl.ei.to(dev)  # the caller's tensors live on the device (device convention, SURVEY.md 8b)
    lib = _lib.load()
    for key, q in qs.items():
        def mk3():
            return Explainer(x_dev, ei_dev, arch, dict(params), names, [list(p) for p in pathways], list(pnames))

        r = _time_runs(mk3, names[q], repeats=3)
        lib.xpgnn_profile(1)  # one more run with per-kernel CUDA events: how much of the wall time is device work
        ex = mk3()
        ex.run(names[q], 1)
        ms, cnt = np.zeros(6), np.zeros(6, dtype=np.int64)
        lib.xpgnn_profile_read(ms.ctypes.data, cnt.ctypes.data)
        lib.xpgnn_profile(0)
        r.update(in_degree=int(indeg[q]), gpu_kernel_ms_per_run=float(ms.sum()), **ex.last_stats)
        out[key] = r
    return out


# ------------------------------------------------------------------------------------------ contract plumbing
def scaling_of(args):
    return "weak" if args.coalitions_per_gpu else "strong"


def per_rank_rows(args, world):
    """Coalition rows of rank r: a 32-aligned share of the job (strong scaling) or a fixed count (weak scaling)."""
    if args.coalitions_per_gpu:
        return [args.coalitions_per_gpu] * world
    words = -(-args.coalitions // 32)
    base, extra = divmod(words, world)
    rows = [32 * (base + (1 if r < extra else 0)) for r in range(world)]
    rows[-1] -= 32 * words - args.coalitions
    return rows


def config_dict(args, wl, world):
    rows = per_rank_rows(args, world)
    return {"workload": args.workload, "nodes": wl.n, "edges": wl.e, "model": wl.model_name, "queries": len(wl.queries),
            "communities": wl.c, "coalitions_per_step": int(sum(rows)), "coalitions_per_gpu_per_step": rows[0],
            "mode": "full (every conv layer over the whole-graph computational graph; per coalition only rows of active "
                    "nodes are materialised, inactive rows are coalition invariant)",
            "l2": "inputs larger than L2 (activation tiles of 16 GiB vs 126 MB L2)", "precision": {
                "fp32": "fp32 (fp32 storage, dense transforms as 3xTF32 tcgen05 MMAs)",
                "bf16": "bf16 transforms (fp32 storage, bf16 tcgen05 MMAs, fp32 accumulate)",
                "bf16_act": "bf16 transforms and bf16 activation storage (fp32 accumulate in the SpMM and the MMAs)",
            }[getattr(args, "precision", "fp32")]}


_REAL_STDOUT = None


def _claim_stdout():
    """Libraries (NCCL's version banner) write to fd 1; the contract is ONE JSON line on stdout.  Point fd 1 at
    stderr for the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much


def dump_outputs(out_dir, y):
    """Writes the predictions of the last timed step (coalition rows x queries) as ``predictions.npy`` (float32) so that
    two builds can be compared output for output; the inputs are seeded, so equal arguments give equal inputs.  Beyond
    DUMP_BYTES a fixed, seeded sample of the rows is written, and their indices as ``prediction_rows.npy`` (float64)."""
    y = np.ascontiguousarray(y, dtype=np.float32)
    os.makedirs(out_dir, exist_ok=True)
    row_bytes = y[0].nbytes + 8
    if y.nbytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(y.shape[0], (DUMP_BYTES - 4096) // row_bytes, replace=False))
        y = y[rows]
        np.save(os.path.join(out_dir, "prediction_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "predictions.npy"), y)


PARITY_BAR = {"fp32": 1e-4, "bf16": 2e-2, "bf16_act": 2e-2}  # BASELINE.json north_star tolerances on the predictions
PARITY_ATOL = 1e-6  # absolute floor for predictions that are themselves ~0 (cancelling head sums): the tests' Y_ATOL


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--coalitions", type=int, default=4096, help="coalition rows of the job = one step (strong scaling over ranks)")
    ap.add_argument("--coalitions-per-gpu", type=int, default=0, help="weak scaling: this many rows per rank and step")
    ap.add_argument("--cpu-coalitions", type=int, default=4, help="coalitions of the CPU baseline / parity sample")
    ap.add_argument("--ref-coalitions", type=int, default=2, help="coalitions per step of --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-query-leg", action="store_true", help="skip s_per_explained_query")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16", "bf16_act"],
                    help="fp32: TF32x3 tensor-core transforms (1e-4 parity bar); bf16: bf16 transforms (2e-2 bar); "
                         "bf16_act: bf16 transforms and bf16 activation storage (2e-2 bar)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the predictions of the last timed step (coalitions x queries; "
                                                         "--impl reference: the first query only) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""  # the reference takes its cupy branch when CUDA is visible (data.py:431)
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist

    from bikg_graph_explainability_public_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    wl = Workload(args.workload)
    n, e, h, c, com_of = wl.n, wl.e, wl.h, wl.c, wl.com_of
    arch, eng = wl.engine(dev, args.precision)
    nq = len(wl.queries)
    rows = per_rank_rows(args, world)
    s_local, s_max, s_total = rows[rank], max(rows), int(sum(rows))
    act, sample = make_packed_masks(lib, s_local, n, c, com_of, 1000 + rank, dev, wl.com_of2,
                                    keep_rows=args.cpu_coalitions if rank == 0 else 0)
    act_host = act.cpu().pin_memory()
    act_in = torch.empty_like(act)
    y_pad = torch.zeros((s_max, nq), dtype=torch.float32, device=dev)
    y_all = torch.empty((world * s_max, nq), dtype=torch.float32, device=dev)

    compute_events = []  # (start, stop) around the rank's own masked forward, without the collective

    def forward(bits, record=False):
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        y = eng(bits, s_local)
        if record:
            e1.record()
            compute_events.append((e0, e1))
        if world > 1:
            y_pad[:s_local] = y
            dist.all_gather_into_tensor(y_all, y_pad)  # the single collective of the path (SURVEY.md 8e)
            return y_all
        return y

    def step_e2e():
        act_in.copy_(act_host, non_blocking=True)
        return forward(act_in).cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        y = forward(act)
    barrier()

    # ---- timed: resident inputs ----
    lib.xpgnn_profile(1)
    launches0 = _lib.launch_count()
    stats0 = eng.stats.cpu().clone()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record()
        for _ in range(args.steps):
            y = forward(act, record=True)
        ev1.record()
        barrier()
    if args.dump_outputs and rank == 0:  # rank 0 holds every rank's rows after the all-gather, each padded to s_max
        y_last = y.cpu().numpy().reshape(world, -1, nq) if world > 1 else y.cpu().numpy()[None]
        y_last = np.concatenate([y_last[r, :rows[r]] for r in range(world)])
    ms_rank = float(ev0.elapsed_time(ev1))
    compute_rank = float(sum(a.elapsed_time(b) for a, b in compute_events))
    ms_all = torch.tensor([ms_rank, compute_rank], device=dev)
    ms_ranks, compute_ranks = [ms_rank], [compute_rank]
    if world > 1:
        gathered = [torch.zeros(2, device=dev) for _ in range(world)]
        dist.all_gather(gathered, ms_all)
        ms_ranks = [float(g[0].item()) for g in gathered]
        compute_ranks = [float(g[1].item()) for g in gathered]
    ms_total = max(ms_ranks)
    launches = _lib.launch_count() - launches0
    active_visits = torch.tensor([float((eng.stats.cpu() - stats0)[1])], device=dev)  # active edge visits of this rank
    if world > 1:
        dist.all_reduce(active_visits, op=dist.ReduceOp.SUM)
    prof_ms = (np.zeros(6), np.zeros(6, dtype=np.int64))
    lib.xpgnn_profile_read(prof_ms[0].ctypes.data, prof_ms[1].ctypes.data)
    lib.xpgnn_profile(0)

    # ---- timed: end to end from the host-resident packed coalition matrix ----
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y_host = step_e2e()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_total = float(e2e_s.item())

    rc = 0
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, y_last)
        evals = s_total * args.steps * nq  # SURVEY.md 8d: coalition rows x queries
        value = evals / (ms_total / 1e3)
        visits = eng.edge_visits_per_coalition  # kept edges x conv layers
        # algorithmic bytes of one coalition-layer (SURVEY.md 8d): col idx + rowptr + bits + read Z once + write
        e_kept = eng.edges_per_layer[0]
        elt = 2 if args.precision == "bf16_act" else 4  # bytes per stored activation element
        b_alg = 4 * e_kept + 4 * (n + 1) + n / 8 + 2 * n * h * elt
        cats = ["masked_degree", "spmm_invariant_l0", "spmm_tile_l1", "dense", "head", "compaction"]
        kern = {k: {"ms": float(prof_ms[0][i]), "launches": int(prof_ms[1][i])} for i, k in enumerate(cats)}
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peaks = json.load(fh)
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        dom = "spmm_tile_l1" if kern["spmm_tile_l1"]["ms"] >= kern["spmm_invariant_l0"]["ms"] else "spmm_invariant_l0"
        share = {k: v["ms"] / max(sum(x["ms"] for x in kern.values()), 1e-9) for k, v in kern.items()}
        tile = eng.tile_coalitions
        roof = {}
        # one pass = one conv layer over one tile of coalitions: ONE launch on homogeneous graphs without hub rows (C3), one
        # launch per relation / destination type on hetero graphs (C4) -- the algorithmic bytes are those of the pass, so
        # the time is the pass's too.  Tiles are counted from the coalitions actually run (a partial last tile counts by
        # its share), the layers' bytes from the per-layer kept-edge counts (sum over the relations of a hetero layer).
        tiles_run = args.steps * s_local / float(tile)
        for k, lays in (("spmm_tile_l1", list(range(1, len(eng.edges_per_layer)))), ("spmm_invariant_l0", [0])):
            if kern[k]["launches"] and lays:
                passes = tiles_run * len(lays)
                avg_ms = kern[k]["ms"] / passes
                b_lay = float(np.mean([4 * eng.edges_per_layer[l] + 4 * (n + 1) + n / 8 + 2 * n * h * elt for l in lays]))
                ach = tile * b_lay / (avg_ms / 1e3) / 1e9
                roof[k] = {"avg_pass_ms": avg_ms, "launches_per_pass": kern[k]["launches"] / passes,
                           "algorithmic_bytes_per_pass": tile * b_lay, "achieved_gbs": ach, "frac": ach / peak}
        traffic, fabric, traffic_src = None, None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                tj = json.load(fh)
            if args.precision == "fp32" and args.workload == "c3":
                traffic = tj.get(dom)
                traffic_src = tj.get("source")
                # the binding resource of the layer >= 1 SpMM is the L2 -> SM fabric, not HBM: report it next to the roofline
                if dom == "spmm_tile_l1" and "spmm_tile_l1_xbar_bytes" in tj and roof.get(dom):
                    ach = tj["spmm_tile_l1_xbar_bytes"] * (tile / 32.0) / (roof[dom]["avg_pass_ms"] / 1e3) / 1e9
                    fabric = {"bytes_per_launch": tj["spmm_tile_l1_xbar_bytes"] * (tile / 32.0), "achieved_gbs": ach,
                              "peak_gbs": tj["l2_fabric_peak_gbs"], "frac": ach / tj["l2_fabric_peak_gbs"],
                              "source": "l1tex__m_xbar2l1tex_read_bytes.sum of one launch (ncu capture named in profiles/traffic.json) / "
                                        "live launch time; peak = tools/gather_probe.cu"}
        except OSError:
            pass
        import ctypes as C
        segv = C.c_int32(0)
        lib.xpgnn_get_option(b"seg", C.byref(segv))
        spmm_name = ("cspmm16_kernel" if args.precision == "bf16_act" else ("cspmm_seg_kernel" if segv.value else "cspmm_kernel"))
        line = {
            "metric": "coalition evals/s", "value": value, "unit": "coalition evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": scaling_of(args), "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": config_dict(args, wl, world),
            "coalition_rows_per_s": value / nq,
            "masked_gteps": value / nq * visits / 1e9,
            "active_gteps": float(active_visits.item()) / (ms_total / 1e3) / 1e9,  # edges that are active in their coalition
            "ms_per_step_by_rank": [m / args.steps for m in ms_ranks],
            # the rank's own masked forward without the all-gather: shows the straggler the collective then waits for
            "compute_ms_per_step_by_rank": [m / args.steps for m in compute_ranks],
            "e2e": {"value": evals / e2e_total, "unit": "coalition evals/s",
                    "h2d_bytes_per_step": int(act_host.numel() * 4), "d2h_bytes_per_step": int(y_host.numel() * 4),
                    "input": "packed coalition matrix [N][W] uint32 (the C ABI's input format) in pinned host memory"},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "roofline": {"bound": "hbm", "kernel": "%s (%s)" % (
                (spmm_name if dom == "spmm_tile_l1" else "l0_ws_kernel") if kern["compaction"]["launches"] else "spmm_masked_kernel", dom),
                         "achieved": roof.get(dom, {}).get("achieved_gbs"), "peak": peak, "unit": "GB/s",
                         "frac": roof.get(dom, {}).get("frac"), "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                         "algorithmic_bytes_per_launch": roof.get(dom, {}).get("algorithmic_bytes_per_pass"), "coalitions_per_launch": tile,
                         "per_kernel": roof, "l2_fabric": fabric},
            "kernels": kern,
            "kernel_share_of_step": share,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, wl, arch, sample, y_host)
            cb, bar = line["cpu_baseline"], PARITY_BAR[args.precision]
            # the bar of the parity tests (tests/test_gpu_parity.py: Y_RTOL / Y_ATOL): |y - y_ref| <= bar * |y_ref| + 1e-6
            ok = bool(np.all(np.abs(np.array(cb["y_gpu"]) - np.array(cb["y_cpu"])) <= bar * np.abs(np.array(cb["y_cpu"])) + PARITY_ATOL))
            line["parity"] = {"max_rel_err": cb["gpu_vs_cpu_max_rel_err"], "max_abs_err": cb["gpu_vs_cpu_max_abs_err"], "rtol": bar,
                              "atol": PARITY_ATOL, "ok": ok, "coalitions": int(sample.shape[0]), "against": cb["kind"]}
            if not ok:
                rc = 3
        if world == 1 and not args.no_query_leg:
            del eng, act, act_in, y_all
            torch.cuda.empty_cache()
            try:
                line["s_per_explained_query"] = query_leg_ours(dev)
            except Exception as ex:
                line["s_per_explained_query"] = {"error": repr(ex)}
                rc = rc or 4
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    if rc:
        sys.stderr.write("[bench] FAILED: %s\n" % ("GPU predictions differ from the CPU reference beyond the parity bar" if rc == 3
                                                   else "query leg raised"))
        sys.exit(rc)


def cpu_baseline(args, wl, arch, sample, y_gpu):
    """The reference (unmodified when staged, else the oracle port) on the host cores over a bounded sample of the same
    workload; also the parity check of the run (bench exits non-zero beyond the bar)."""
    torch.set_num_threads(os.cpu_count())
    m = sample.numpy()
    b = int(m.shape[0])
    om = wl.oracle_model(arch)
    ref = None
    if wl.kind == "homo_gcn":
        # the reference must not see CUDA (cupy branch, data.py:431): run it in a child process with the devices hidden
        ref = "subprocess"
    t0 = time.perf_counter()
    if ref == "subprocess":
        y_ref, kind, dt = _host_eval_subprocess(args, m)
    else:
        y_ref, kind = host_eval(wl, om, m, None)
        dt = time.perf_counter() - t0
    y0 = y_gpu.numpy().reshape(-1, len(wl.queries))[:b, 0].astype(np.float64)
    y_ref = np.asarray(y_ref, dtype=np.float64)
    rel = float(np.max(np.abs(y0 - y_ref) / np.maximum(np.abs(y_ref), 1e-6)))
    return {"value": b / dt, "unit": "coalition evals/s", "cores": os.cpu_count(), "kind": kind,
            "sample": "%d coalitions of the full %s workload in one batch (%.1f s of CPU work); %s" % (b, args.workload, dt, _kind_note(kind)),
            "gpu_vs_cpu_max_rel_err": rel, "gpu_vs_cpu_max_abs_err": float(np.max(np.abs(y0 - y_ref))),
            "y_gpu": [float(v) for v in y0], "y_cpu": [float(v) for v in y_ref]}


def _host_eval_subprocess(args, mask_bool_np):
    """Child process with CUDA hidden: rebuilds the (seeded) workload and model, evaluates the sample rows with the
    unmodified reference (or the port when the staged copy is missing) and returns the predictions and the eval time."""
    import tempfile

    with tempfile.TemporaryDirectory() as td:
        np.save(os.path.join(td, "mask.npy"), mask_bool_np)
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        code = ("import sys, json, time, numpy as np, torch; sys.path.insert(0, %r); import bench;"
                "torch.set_num_threads(%d); wl = bench.Workload(%r); om = wl.oracle_model(wl.make_model());"
                "ref = bench._reference_modules(); m = np.load(%r); t0 = time.perf_counter();"
                "y, kind = bench.host_eval(wl, om, m, ref); dt = time.perf_counter() - t0;"
                "np.save(%r, y); print(json.dumps({'kind': kind, 'dt': dt}))"
                % (ROOT, os.cpu_count(), args.workload, os.path.join(td, "mask.npy"), os.path.join(td, "y.npy")))
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
        if out.returncode != 0:
            raise RuntimeError("CPU baseline child failed: " + out.stderr[-2000:])
        info = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        return np.load(os.path.join(td, "y.npy")), info["kind"], info["dt"]


if __name__ == "__main__":
    main()
