"""The masked forward against a float64 reference: every row, every column, every engine option, the path boundaries.

``masked_forward_f64`` evaluates the lowered plan the kernels receive (``LoweredModel``) in float64, for every
coalition and every row, and a *magnitude pass*: the same forward on |x|, |W|, |b| with ReLU replaced by the identity.
``mag[s, v, c]`` bounds the sum of the absolute values of the terms that make up ``y[s, v, c]``, so the bar
``|y - y64| <= TAU * mag + TINY`` follows the conditioning of each value instead of one global rtol, and it sees
errors that a sigmoid head would shrink.  The CPU tests check the reference itself against the oracle.

The GPU tests read the engine without a head (``n_head = 0``, ``out_col`` swept over the chunk and column-block
boundaries) or through one random projection ``Linear(H, 1)`` without activation, with every node as a query, so
every (coalition, row, column) of the last conv layer reaches the comparison.

Measured on one B200 (1000 W power limit; fp32 plan, default options), the largest ``|y - y64| / mag`` per path:
    compact 8.4e-07 and tile 7.4e-07 (one layer without a head: the 3xTF32 transform Z = X W^T dominates),
    sliced hub rows at the scratch boundary 1.2e-07, hetero 5.8e-09, pruned 2.5e-09 (through the projection head),
    fp32_exact 4.2e-09; bf16_act 3.5e-05.  TAU is about 5x the largest fp32 value, 25x tighter than the 1e-4 bar of
    tests/test_gpu_parity.py before its sigmoid head divides the error by 4 or more.
Two fp32 runs of one plan whose options change only the order of the SpMM additions (``TAU_PAIR``, against the same
magnitudes) differed by at most 2.6e-09 (cw = 16 against 32); TAU_PAIR is about 6x that.

Options whose kernels differ only in scheduling, cache hints, carve-out or how a warp waits -- not in which FMAs run
in which order -- are also checked bitwise against the default (third field of ``OPTION_CASES``):
    l2_stream / l2_gather: the same loads with another ``createpolicy`` eviction priority (compact.cu ``l2_policy``);
    seg_carve: ``cudaFuncAttributePreferredSharedMemoryCarveout`` on the same kernel;
    l0_wait_ns / dense_wait_ns: the suspend-time hint of ``mbarrier.try_wait`` (0: poll + nanosleep) of the warps
    that wait for a stage; the stage contents and the MMA / FMA order do not change;
    act_column: the kernels read the same coalition word from a dense copy instead of the [N][W] matrix;
    l0_ws = 1 against the default 3: the same kernel with the Z pieces staged by cp.async instead of TMA bulk copies.
Every other option that keeps the dense transforms (not in ``TRANSFORM_OPTIONS``) is checked against the default
run under ``TAU_PAIR``.
"""
import math
import os
import sys
from dataclasses import dataclass, replace
from typing import List

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TAU = 4e-6             # fp32 plan against float64 (module docstring: about 5x the largest measured ratio)
TAU_PAIR = 1.5e-8      # two fp32 runs of one plan that differ only in the order of the SpMM sums (module docstring)
TAU_BF16 = 2e-2        # bf16 transforms / storage: the bar of BASELINE.json, against the same magnitudes
TINY = 1e-30
OUT_COLS = (0, 15, 16, 31, 32, 63, 64)  # plus H - 1: chunk (16 / 32 floats) and column-block (64) boundaries


# ------------------------------------------------------------------------------------------------ reference


@dataclass
class Ref64:
    acts: List[torch.Tensor]   # per conv layer [S, N, H] float64 (after its activation)
    mags: List[torch.Tensor]   # magnitude pass of the same
    out: torch.Tensor          # head output [S, N, D] (the last conv layer when there is no head); zero-edge rule applied
    out_mag: torch.Tensor


def _act64(v, m, act):
    if act == "relu":
        return torch.relu(v), m
    if act == "sigmoid":  # |sigmoid(a) - sigmoid(b)| <= |a - b| / 4, plus the rounding of the value itself
        s = torch.sigmoid(v)
        return s, s + 0.25 * m
    assert act is None, act
    return v, m


def _padded(w, k, dev):
    """[out, in] float64 zero-padded to ``k`` input columns (padded hetero features), as the engine stores it."""
    w = w.detach().to(dev, torch.float64)
    return torch.nn.functional.pad(w, (0, k - w.shape[1])) if w.shape[1] < k else w


def _scatter(dst, src, vals, h, n, chunk=1 << 21):
    """out[v] = sum over the edges e with dst[e] = v of vals[e] * h[src[e]] (edge chunks bound the temporary)."""
    out = torch.zeros((n, h.shape[1]), dtype=h.dtype, device=h.device)
    for i in range(0, dst.numel(), chunk):
        out.index_add_(0, dst[i:i + chunk], h[src[i:i + chunk]] * vals[i:i + chunk, None])
    return out


def masked_forward_f64(model, x, edge_index, mask, type_ptr=None, node_type_names=None, edge_type=None,
                       edge_type_names=None, zero_edge_rule=False, device="cpu", keep_acts=True):
    """Float64 forward of a lowered plan under every coalition of ``mask`` [S, N] (bool).

    Edge u->v is active in coalition s iff both endpoints are; features are never masked.  GCN drops the input self
    loops and gives every node one unit loop (deg = 1 + active in-edges, multi-edges counted, weight
    1/sqrt(deg_u deg_v)); SAGE(mean) averages the active in-neighbours (0 without one) through lin_l (+ bias) and adds
    lin_r of the node itself.  Relations into the same destination type are summed; rows of a type no relation of the
    layer writes are 0.  ``zero_edge_rule``: a coalition without any active input edge outputs 0 (model.py:213-215)."""
    dev = torch.device(device)
    x = torch.as_tensor(x).to(dev, torch.float64)
    ei = torch.as_tensor(edge_index).to(dev, torch.int64)
    m_all = torch.as_tensor(mask).to(dev, torch.bool)
    s_cnt, n = m_all.shape
    f_in = x.shape[1]
    tnames = node_type_names
    et = None if edge_type is None else torch.as_tensor(edge_type).to(dev, torch.int64)

    def rng(t):
        if tnames is None or t is None:
            return 0, n
        i = tnames.index(t)
        return type_ptr[i], type_ptr[i + 1]

    # per-relation edge lists and float64 weights, per layer
    layers, h_in = [], f_in
    for conv in model.convs:
        rels = []
        for r in conv.relations:
            src, dst = ei[0], ei[1]
            if r.key is not None:
                sel = et == edge_type_names.index(r.key)
                src, dst = src[sel], dst[sel]
            if r.kind == "gcn":
                keep = src != dst
                src, dst = src[keep], dst[keep]
            s_t, d_t = (r.key[0], r.key[-1]) if r.key is not None else (None, None)
            w = _padded(r.w_nbr, h_in, dev)
            wr = None if r.w_root is None else _padded(r.w_root, h_in, dev)
            b = None if r.b_nbr is None else r.b_nbr.detach().to(dev, torch.float64)
            rels.append((r.kind, src, dst, rng(d_t), w, wr, b))
        layers.append((rels, conv.out_dim, conv.act))
        h_in = conv.out_dim
    head = [(w.detach().to(dev, torch.float64), None if b is None else b.detach().to(dev, torch.float64), a)
            for w, b, a in model.head]
    d_out = head[-1][0].shape[0] if head else model.convs[-1].out_dim

    acts = [torch.zeros((s_cnt, n, c.out_dim), dtype=torch.float64, device=dev) for c in model.convs] if keep_acts else []
    mags = [torch.zeros_like(a) for a in acts]
    out = torch.zeros((s_cnt, n, d_out), dtype=torch.float64, device=dev)
    out_mag = torch.zeros_like(out)
    for s in range(s_cnt):
        m = m_all[s]
        h, hm = x, x.abs()
        for li, (rels, h_out, act) in enumerate(layers):
            o = torch.zeros((n, h_out), dtype=torch.float64, device=dev)
            om = torch.zeros_like(o)
            for kind, src, dst, (lo, hi), w, wr, b in rels:
                a = m[src] & m[dst]
                sa, da = src[a], dst[a]
                cnt = torch.bincount(da, minlength=n).to(torch.float64)
                rows = slice(lo, hi)
                if kind == "gcn":
                    dis = (1.0 + cnt).rsqrt()
                    vals = dis[sa] * dis[da]
                    z, zm = h @ w.T, hm @ w.abs().T
                    agg = _scatter(da, sa, vals, z, n) + (dis * dis)[:, None] * z
                    aggm = _scatter(da, sa, vals, zm, n) + (dis * dis)[:, None] * zm
                else:
                    vals = 1.0 / cnt.clamp(min=1.0)[da]
                    agg = _scatter(da, sa, vals, h, n) @ w.T
                    aggm = _scatter(da, sa, vals, hm, n) @ w.abs().T
                    if wr is not None:
                        agg, aggm = agg + h @ wr.T, aggm + hm @ wr.abs().T
                if b is not None:
                    agg, aggm = agg + b, aggm + b.abs()
                o[rows] += agg[rows]
                om[rows] += aggm[rows]
            h, hm = _act64(o, om, act)
            if keep_acts:
                acts[li][s], mags[li][s] = h, hm
        for w, b, act in head:
            h, hm = h @ w.T, hm @ w.abs().T
            if b is not None:
                h, hm = h + b, hm + b.abs()
            h, hm = _act64(h, hm, act)
        if zero_edge_rule and not bool((m[ei[0]] & m[ei[1]]).any()):
            h, hm = torch.zeros_like(h), torch.zeros_like(hm)
        out[s], out_mag[s] = h, hm
    return Ref64(acts, mags, out, out_mag)


# ------------------------------------------------------------------------------------------------ CPU: the reference itself


def _fixture_case(seed, kind, n=400, e=3000, f=20, hidden=(24, 24), s=60):
    """Random multigraph with duplicate edges and input self loops, iid coalitions incl. all-on / all-off rows."""
    from oracle import fixture_models as fm

    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, f, generator=g)
    ei = torch.randint(0, n, (2, e), generator=g)
    ei = torch.cat([ei, ei[:, :30], torch.arange(10).repeat(2, 1)], 1)
    arch = (fm.HomoGCN(f, hidden, (hidden[-1], 8, 1), seed=seed) if kind == "gcn"
            else fm.HomoSAGE(f, hidden, (hidden[-1], 1), seed=seed)).eval()
    mask = torch.rand(s, n, generator=g) < 0.5
    mask[0] = True
    mask[1] = False
    return x, ei, arch, mask


@pytest.mark.parametrize("kind,hidden", [("gcn", (24,)), ("gcn", (24, 24)), ("gcn", (16, 32, 24)), ("sage", (24, 24)),
                                         ("sage", (32,))])
def test_reference_matches_oracle_homogeneous(kind, hidden):
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask = _fixture_case(3, kind, hidden=hidden)
    ref = masked_forward_f64(lower(arch), x, ei, mask)
    for q in (0, 5, 399):  # node 5 carries an input self loop
        _, y_or = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
        y_or = y_or.double().reshape(-1)
        np.testing.assert_allclose(ref.out[:, q, 0].numpy(), y_or.numpy(), rtol=1e-6, atol=1e-7)
    assert bool((ref.out_mag >= ref.out.abs()).all())


def test_reference_matches_oracle_hetero():
    """c4_tiny: 5 node types, 9 SAGE relations, 2 layers, several relations into one type, and the zero-edge rule."""
    sys.path.insert(0, ROOT)
    import bench
    from bikg_graph_explainability_public_b200.lowering import lower

    wl = bench.Workload("c4_tiny")
    mask = bench.make_masks(12, wl.n, wl.c, wl.com_of, 3).bool()
    mask[5] = False   # no active edge: the zero-edge rule
    mask[6] = True
    arch = wl.make_model()
    y_or = wl.oracle_eval(wl.oracle_model(arch), mask.numpy())
    ref = masked_forward_f64(lower(arch), wl.x, wl.ei, mask, wl.type_ptr, wl.node_type_names, wl.edge_type,
                             wl.edge_type_names, zero_edge_rule=True)
    np.testing.assert_allclose(ref.out[:, wl.queries[0], 0].numpy(), y_or, rtol=1e-6, atol=1e-7)
    assert float(ref.out[5].abs().max()) == 0.0


def test_reference_magnitude_bounds_perturbed_weights():
    """The magnitude pass is a bound: perturbing every weight by a relative 1e-6 moves no value by more than
    about 1e-6 x mag (first order, ReLU kinks aside)."""
    from bikg_graph_explainability_public_b200.lowering import lower

    x, ei, arch, mask = _fixture_case(4, "gcn", hidden=(32, 32), s=20)
    model = _headless(lower(arch))
    ref = masked_forward_f64(model, x, ei, mask)
    g = torch.Generator().manual_seed(1)

    def jitter(t):
        return None if t is None else t * (1 + 1e-6 * (2 * torch.rand(t.shape, generator=g, dtype=torch.float64) - 1))

    pert = _headless(model)
    for c in pert.convs:
        c.relations = [replace(r, w_nbr=jitter(r.w_nbr.double()), b_nbr=jitter(r.b_nbr.double())) for r in c.relations]
    ref2 = masked_forward_f64(pert, x, ei, mask)
    ratio = float(((ref2.out - ref.out).abs() / (ref.out_mag + TINY)).max())
    assert 1e-8 < ratio <= 3e-6, ratio


# ------------------------------------------------------------------------------------------------ GPU helpers


def _headless(model):
    from bikg_graph_explainability_public_b200.lowering import LoweredModel

    return LoweredModel(convs=[replace(c, relations=list(c.relations)) for c in model.convs], head=[],
                        n_message_passing=model.n_message_passing)


def _with_projection(model, seed=0):
    """The same conv stack followed by one random Linear(H, 1) without activation: y = p . h + b mixes every column."""
    g = torch.Generator().manual_seed(seed)
    h = model.convs[-1].out_dim
    m = _headless(model)
    m.head = [(torch.randn(1, h, generator=g) / math.sqrt(h), torch.randn(1, generator=g), None)]
    return m


def _random_stack(kind, f, widths, seed, acts=None):
    """Lowered homogeneous stack with random weights (ReLU between layers, none after the last unless given)."""
    from bikg_graph_explainability_public_b200.lowering import LoweredConv, LoweredModel, LoweredRelation

    g = torch.Generator().manual_seed(seed)
    convs, d = [], f
    for i, h in enumerate(widths):
        w = torch.randn(h, d, generator=g) / math.sqrt(d)
        b = 0.1 * torch.randn(h, generator=g)
        wr = torch.randn(h, d, generator=g) / math.sqrt(d) if kind == "sage" else None
        act = (acts[i] if acts is not None else ("relu" if i < len(widths) - 1 else None))
        convs.append(LoweredConv([LoweredRelation(kind, None, w, b, wr)], h, act=act))
        d = h
    return LoweredModel(convs=convs, head=[], n_message_passing=len(widths))


def _pack(lib, mask):
    from bikg_graph_explainability_public_b200 import _lib

    s, n = mask.shape
    m8 = mask.to(torch.uint8).cuda().contiguous()
    w = -(-s // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
    _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, None, _lib.stream_ptr()))
    return act


def _ratio(y, y64, mag):
    y = torch.as_tensor(y).to(y64.device, torch.float64)
    return float(((y - y64).abs() / (mag + TINY)).max()) if y.numel() else 0.0


def _check(y, y64, mag, tau=None, what=""):
    """|y - y64| <= tau * mag + TINY elementwise (tau: TAU); reports the worst element."""
    tau = TAU if tau is None else tau
    y = torch.as_tensor(y).to(y64.device, torch.float64)
    assert y.shape == y64.shape, (what, tuple(y.shape), tuple(y64.shape))
    assert bool(torch.isfinite(y).all()), (what, "non-finite output")
    err = (y - y64).abs()
    bad = err > tau * mag + TINY
    if bool(bad.any()):
        i = tuple(int(t) for t in torch.nonzero(bad)[0])
        raise AssertionError("%s: %d values outside tau=%g; first at %s: y=%r y64=%r mag=%r, max ratio %.3g"
                             % (what, int(bad.sum()), tau, i, float(y[i]), float(y64[i]), float(mag[i]), _ratio(y, y64, mag)))


def _rich_graph(seed=0, n=3000, f=32, e=12000, s=75):
    """A graph that reaches every branch of the kernels: rows with no in-edge, medium rows (80 - 240 active in-edges),
    hub rows above 1024 and above 4096 in-edges (one and several layer-0 slices; > 256 active: CTA-level rows of the
    compact SpMM), multi-edges and input self loops; S = 75 coalitions (three words, the last one partial) incl. an
    all-on row, an all-off row, a sparse row, and coalitions in which the hubs and the first query are inactive."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, f, generator=g)
    ei = torch.randint(0, n, (2, e), generator=g)
    ei = ei[:, (ei[1] < 100) | (ei[1] >= 150)]          # rows 100 .. 149: no in-edge
    parts = [ei, ei[:, :40], torch.arange(200, 210).repeat(2, 1)]  # duplicates, self loops
    for r in range(20):                                  # medium rows: 160 .. 480 in-edges, about a quarter active
        k = 160 + 16 * r
        parts.append(torch.stack([torch.randint(0, n, (k,), generator=g), torch.full((k,), 300 + r)]))
    for hub, k in ((7, 1100), (8, 1500), (9, 4100), (10, 5000), (11, 9000)):
        parts.append(torch.stack([torch.randint(0, n, (k,), generator=g), torch.full((k,), hub)]))
    ei = torch.cat(parts, 1)
    mask = torch.rand(s, n, generator=g) < 0.5
    mask[0] = True
    mask[1] = False
    mask[2] = torch.rand(n, generator=g) < 0.05
    mask[3:10, 7:12] = False                             # hubs inactive
    mask[10:17, 7:12] = True
    mask[17:22, 0] = False
    return x, ei, mask


QUERY = 0


class Case:
    """One graph + coalitions + float64 reference of a model, on the GPU."""

    def __init__(self, lib, model, x, ei, mask, graph_kw=None, zero_edge_rule=False):
        from bikg_graph_explainability_public_b200.engine import GraphSpec

        self.lib, self.model, self.x, self.ei, self.mask = lib, model, x, ei, mask
        self.s, self.n = mask.shape
        gk = dict(graph_kw or {})
        self.zero_edge_rule = zero_edge_rule
        self.graph = GraphSpec(x.cuda(), ei.cuda(), gk.get("type_ptr", [0, self.n]), gk.get("node_type_names"),
                               None if gk.get("edge_type") is None else gk["edge_type"].cuda(), gk.get("edge_type_names"))
        self.ref = masked_forward_f64(model, x, ei, mask, gk.get("type_ptr"), gk.get("node_type_names"), gk.get("edge_type"),
                                      gk.get("edge_type_names"), zero_edge_rule, device="cuda", keep_acts=False)
        self.act = _pack(lib, mask)

    def run(self, queries=None, out_col=0, s0=0, n_s=None, model=None, **kw):
        from bikg_graph_explainability_public_b200.engine import MaskedForward

        q = list(range(self.n)) if queries is None else list(queries)
        eng = MaskedForward(self.graph, model or self.model, q, zero_edge_rule=self.zero_edge_rule, out_col=out_col, **kw)
        y = eng(self.act, self.s, s0, n_s)
        torch.cuda.synchronize()
        return y

    def expect(self, queries=None, out_col=0, s0=0, n_s=None):
        q = torch.arange(self.n) if queries is None else torch.as_tensor(list(queries))
        n_s = self.s - s0 if n_s is None else n_s
        q = q.to(self.ref.out.device)
        return self.ref.out[s0:s0 + n_s][:, q, out_col], self.ref.out_mag[s0:s0 + n_s][:, q, out_col]

    def check(self, y, tau=None, what="", **sel):
        y64, mag = self.expect(**sel)
        _check(y, y64, mag, tau, what)


# ------------------------------------------------------------------------------------------------ GPU: every row, every column


@pytest.mark.gpu
@pytest.mark.parametrize("kind,widths", [("gcn", (128, 128, 128)), ("sage", (128, 64, 128)), ("gcn", (64, 192))])
def test_every_row_every_column(kind, widths, lib, knobs):
    """Stacks of one, two, three layers (prefixes of the same weights), no head, every node a query: y[s, v] is column
    ``out_col`` of the last layer at row v, swept over the chunk / column-block boundaries; then one projection head
    over all columns.  Compact path, tile path (compact=0), pruned tile path on a few queries (prune_l0 0 and 1)."""
    from bikg_graph_explainability_public_b200.data import khop_subgraph

    x, ei, mask = _rich_graph(1)
    full = _random_stack(kind, x.shape[1], widths, seed=11)
    for depth in range(1, len(widths) + 1):
        model = _headless(full)
        model.convs = model.convs[:depth]
        h = widths[depth - 1]
        c = Case(lib, model, x, ei, mask)
        for col in sorted(set(OUT_COLS + (h - 1,))):
            if col < h:
                c.check(c.run(out_col=col), what="compact depth %d col %d" % (depth, col), out_col=col)
        knobs(compact=0)
        for col in (0, h - 1):
            c.check(c.run(out_col=col), what="tile depth %d col %d" % (depth, col), out_col=col)
        knobs(compact=1)
    cp = Case(lib, _with_projection(full), x, ei, mask)
    cp.check(cp.run(), what="projection head")
    knobs(compact=0)
    cp.check(cp.run(), what="projection head, tile path")
    for q in (QUERY, 11, 120):  # a plain row, the largest hub, a row without in-edges
        hop = khop_subgraph(ei.cuda(), x.shape[0], q, len(widths) + 1)[4]
        for pl0 in (1, 0):
            knobs(prune_l0=pl0)
            y = cp.run([q], prune=True, hop=hop)
            cp.check(y, what="pruned q=%d prune_l0=%d" % (q, pl0), queries=[q])


@pytest.mark.gpu
def test_fp32_exact_every_row(lib):
    """precision="fp32_exact" (exact fp32 FMA transforms) on the same rows and columns."""
    x, ei, mask = _rich_graph(2)
    c = Case(lib, _with_projection(_random_stack("gcn", x.shape[1], (128, 128), seed=5)), x, ei, mask)
    c.check(c.run(precision="fp32_exact"), what="fp32_exact")


# ------------------------------------------------------------------------------------------------ GPU: every option value

# (option values, model kind, extra options, bitwise against the default run of the same model)
OPTION_CASES = [
    ({"compact": 0}, "gcn", False),
    ({"cw": 16}, "gcn", False),
    ({"cw": 16}, "sage", False),
    ({"l0_lists": 1}, "gcn", False),
    ({"l0_lists": 1}, "sage", False),
    ({"seg": 0, "occ": 6}, "gcn", False),
    ({"seg": 0, "occ": 8}, "gcn", False),
    ({"seg": 4}, "gcn", False), ({"seg": 6}, "gcn", False), ({"seg": 7}, "sage", False), ({"seg": 8}, "gcn", False),
    ({"seg": 12}, "gcn", False), ({"seg": 16}, "gcn", False), ({"seg": 116}, "gcn", False), ({"seg": 124}, "gcn", False),
    ({"seg": 216}, "gcn", False), ({"seg": 232}, "gcn", False), ({"seg": 316}, "gcn", False), ({"seg": 332}, "gcn", False),
    ({"seg": 432}, "gcn", False), ({"seg": 516}, "gcn", False), ({"seg": 532}, "gcn", False),
    ({"seg": 8, "seg_occ": 7}, "gcn", False), ({"seg": 8, "seg_occ": 8}, "gcn", False),
    ({"seg": 6, "seg_occ": 6}, "gcn", False), ({"seg": 6, "seg_occ": 7}, "gcn", False),
    ({"seg": 4, "seg_occ": 10}, "gcn", False),
    ({"seg_skew": 4}, "gcn", False),
    ({"seg_tma": 1}, "gcn", False),
    ({"seg": 8, "seg_pf": 8}, "gcn", False), ({"seg": 8, "seg_pf": 12}, "gcn", False),
    ({"seg": 8, "seg_pf": 16}, "gcn", False), ({"seg": 4, "seg_pf": 8}, "sage", False),
    ({"seg_carve": 50}, "gcn", True),
    ({"l2_stream": 0}, "gcn", True), ({"l2_stream": 2}, "gcn", True),
    ({"l2_gather": 1}, "gcn", True), ({"l2_gather": 2}, "gcn", True),
    ({"sched_static": 1}, "gcn", False),
    ({"act_column": 0}, "gcn", True), ({"act_column": 0}, "sage", True),
    ({"l0_slices": 0}, "gcn", False),
    ({"long_rows": 0}, "gcn", False), ({"long_rows": 0}, "sage", False),
    ({"l0_ws": 0}, "gcn", False), ({"l0_ws": 1}, "gcn", True), ({"l0_ws": 2}, "sage", False),
    ({"l0_wait_ns": 0}, "gcn", True),
    ({"dense_wait_ns": 0}, "gcn", True), ({"dense_wait_ns": 0}, "sage", True),
    ({"dense_simt": 1}, "gcn", False),
    ({"compact": 0, "fused": 1}, "gcn", False),
    ({"compact": 0, "fused": 1, "fused_sb": 8}, "gcn", False),
]


# options that change the dense transforms (or route layers through other ones), not only the order of the SpMM sums
TRANSFORM_OPTIONS = {"dense_simt", "compact", "fused", "fused_sb", "l0_lists"}


@pytest.fixture(scope="module")
def option_cases(lib):
    x, ei, mask = _rich_graph(3)
    cases, base = {}, {}
    for kind in ("gcn", "sage"):
        cases[kind] = Case(lib, _with_projection(_random_stack(kind, x.shape[1], (128, 128), seed=21), seed=2), x, ei, mask)
        base[kind] = cases[kind].run().cpu()
    return cases, base


@pytest.mark.gpu
@pytest.mark.parametrize("opts,kind,bitwise", OPTION_CASES, ids=lambda v: str(v) if isinstance(v, (dict, str)) else "")
def test_option_value_matches_reference(opts, kind, bitwise, option_cases, knobs):
    cases, base = option_cases
    c = cases[kind]
    _check(base[kind], *c.expect(), what="default options")
    knobs(**opts)
    y = c.run()
    c.check(y, what=str(opts))
    if bitwise:
        np.testing.assert_array_equal(y.cpu().numpy(), base[kind].numpy(), err_msg=str(opts))
    elif not set(opts) & TRANSFORM_OPTIONS:
        _check(y, base[kind].to(y.device, torch.float64), c.expect()[1], TAU_PAIR, "%s vs default" % opts)


@pytest.mark.gpu
@pytest.mark.parametrize("occ16", [4, 6, 8])
def test_bf16_storage_occupancy_variants(occ16, lib, knobs):
    """occ16 selects the CTAs / SM of the bf16-storage SpMM (precision="bf16_act", GCN, widths % 64): bf16 bar."""
    x, ei, mask = _rich_graph(4)
    c = Case(lib, _with_projection(_random_stack("gcn", x.shape[1], (128, 128), seed=3)), x, ei, mask)
    knobs(occ16=occ16)
    c.check(c.run(precision="bf16_act"), tau=TAU_BF16, what="bf16_act occ16=%d" % occ16)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", [{}, {"l0_multi": 0}, {"l1_multi": 1}, {"compact_hetero": 0}])
def test_hetero_options_match_reference(opts, lib, knobs):
    """c4_tiny graph (5 node types, 9 SAGE relations, several into one type), zero-edge rule, every node a query,
    projection head: the hetero compact path and its options, and the per-relation tile path."""
    sys.path.insert(0, ROOT)
    import bench
    from bikg_graph_explainability_public_b200.lowering import lower

    wl = bench.Workload("c4_tiny")
    mask = bench.make_masks(70, wl.n, wl.c, wl.com_of, 3).bool()
    mask[5] = False
    mask[6] = True
    model = _with_projection(lower(wl.make_model()), seed=4)
    gk = dict(type_ptr=wl.type_ptr, node_type_names=wl.node_type_names, edge_type=wl.edge_type,
              edge_type_names=wl.edge_type_names)
    c = Case(lib, model, wl.x, wl.ei, mask, gk, zero_edge_rule=True)
    knobs(**opts)
    y = c.run()
    c.check(y, what="hetero %s" % opts)
    assert float(y[5].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------ GPU: path boundaries


def _slice_boundary_graph(n, hubs, query_from_hubs, seed):
    """``hubs`` destination rows with 1100 in-edges each from random sources other than the row (one layer-0 slice
    item each); with ``query_from_hubs`` the last node also receives one in-edge from every hub."""
    g = torch.Generator().manual_seed(seed)
    rows = torch.arange(hubs)
    dst = rows.repeat_interleave(1100)
    src = torch.randint(0, n - 1, (dst.numel(),), generator=g)
    src += (src >= dst).to(src.dtype)      # never the row itself
    parts = [torch.stack([src, dst])]
    if query_from_hubs:
        parts.append(torch.stack([rows, torch.full((hubs,), n - 1)]))
    return torch.cat(parts, 1)


def _layer0_items(ei, n, rows):
    """Slice items of the layer-0 hub rows among ``rows`` (compact_l0.cu l0_long_items_kernel): a row with more than
    kLongRow = 1024 in-edges (self loops dropped) is cut into ceil(deg / kL0Slice) slices of 4096; and the scratch
    capacity l0_slice_scratch_items(E) = min(E / 1024 + E / 4096 + 2, kL0SliceScratchItems = 16384)."""
    keep = ei[0] != ei[1]
    deg = torch.bincount(ei[1][keep], minlength=n)[rows]
    e = int(keep.sum())
    return int(((deg + 4095) // 4096)[deg > 1024].sum()), min(e // 1024 + e // 4096 + 2, 16384)


@pytest.mark.gpu
@pytest.mark.parametrize("over", [0, 1])
def test_slice_scratch_boundary_compact(over, lib, knobs):
    """Compact path, layer 0 with 16 384 (sliced) / 16 385 (more items than the scratch holds: unsliced) hub rows,
    about 18 M edges, every node a query through a projection head."""
    n = 20000
    ei = _slice_boundary_graph(n, 16384 + over, False, seed=over)
    items, cap = _layer0_items(ei, n, torch.arange(n))
    assert cap == 16384 and items == 16384 + over, (items, cap)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(n, 32, generator=g)
    mask = torch.rand(12, n, generator=g) < 0.5
    mask[0] = True
    mask[1] = False
    c = Case(lib, _with_projection(_random_stack("gcn", 32, (128,), seed=1)), x, ei, mask)
    y = c.run()
    c.check(y, what="compact, %d slice items" % items)
    knobs(l0_slices=0)
    y0 = c.run()
    c.check(y0, what="compact, l0_slices=0")
    if over:  # above the cap the call already ran unsliced
        np.testing.assert_array_equal(y.cpu().numpy(), y0.cpu().numpy())
    else:     # the same Z, the same terms: sliced and unsliced differ in the order of the additions only
        _check(y, y0.double(), c.expect()[1], TAU_PAIR, "sliced vs unsliced")


@pytest.mark.gpu
@pytest.mark.parametrize("over", [0, 1])
def test_slice_scratch_boundary_pruned(over, lib, knobs):
    """Pruned tile path (engine.cu: prune_l0, 2 layers): layer 0 runs the rows within one hop of the query; its hub
    rows are the 16 380 / 16 381 in-neighbours (1100 in-edges, one item each) and the query itself (16 380 / 16 381
    in-edges: 4 slices), i.e. 16 384 / 16 385 items."""
    from bikg_graph_explainability_public_b200.data import khop_subgraph

    n = 20000
    q = n - 1
    ei = _slice_boundary_graph(n, 16380 + over, True, seed=10 + over)
    hop = khop_subgraph(ei.cuda(), n, q, 3)[4]
    rows0 = torch.nonzero((hop >= 0) & (hop <= 1)).flatten().cpu()
    items, cap = _layer0_items(ei, n, rows0)
    assert cap == 16384 and items == 16384 + over, (items, cap)
    g = torch.Generator().manual_seed(19)
    x = torch.randn(n, 32, generator=g)
    mask = torch.rand(12, n, generator=g) < 0.5
    mask[0] = True
    mask[1] = False
    mask[3, q] = False
    c = Case(lib, _with_projection(_random_stack("gcn", 32, (128, 64), seed=2)), x, ei, mask)
    y = c.run([q], prune=True, hop=hop)
    c.check(y, what="pruned, %d slice items" % items, queries=[q])
    knobs(l0_slices=0)
    y0 = c.run([q], prune=True, hop=hop)
    c.check(y0, what="pruned, l0_slices=0", queries=[q])
    if over:
        np.testing.assert_array_equal(y.cpu().numpy(), y0.cpu().numpy())
    else:
        _check(y, y0.double(), c.expect(queries=[q])[1], TAU_PAIR, "sliced vs unsliced")


@pytest.mark.gpu
@pytest.mark.parametrize("widths", [(256, 64), (320, 64), (48, 48), (24, 32), (64, 24)])
def test_layer_width_boundaries(widths, lib, knobs):
    """256 / 320 in layer 0 (hub rows sliced only up to 4 column blocks; 320 runs the compact path unsliced), 48
    (forces 16-float chunks), 24 (not a multiple of 16: tile path), on the hub graph, both conv kinds."""
    x, ei, mask = _rich_graph(5, s=40)
    for kind in ("gcn", "sage"):
        c = Case(lib, _with_projection(_random_stack(kind, x.shape[1], widths, seed=7)), x, ei, mask)
        c.check(c.run(), what="%s %s" % (kind, widths))
        knobs(compact=0)
        c.check(c.run(), what="%s %s tile path" % (kind, widths))
        knobs(compact=1)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [256, 320])
def test_hetero_width_boundary(hidden, lib):
    """Hetero compact path up to 256 columns; at 320 it hands the plan to the per-relation tile path."""
    sys.path.insert(0, ROOT)
    import bench
    from bikg_graph_explainability_public_b200.lowering import LoweredConv, LoweredModel, LoweredRelation

    wl = bench.Workload("c4_tiny")
    g = torch.Generator().manual_seed(hidden)
    convs, d = [], wl.f
    for i in range(2):
        rels = [LoweredRelation("sage", r, torch.randn(hidden, d, generator=g) / math.sqrt(d), 0.1 * torch.randn(hidden, generator=g),
                                torch.randn(hidden, d, generator=g) / math.sqrt(d)) for r in wl.edge_type_names]
        convs.append(LoweredConv(rels, hidden, act="relu" if i == 0 else None, hetero=True))
        d = hidden
    model = _with_projection(LoweredModel(convs=convs, head=[], n_message_passing=2 * len(wl.edge_type_names)), seed=1)
    mask = bench.make_masks(40, wl.n, wl.c, wl.com_of, 5).bool()
    gk = dict(type_ptr=wl.type_ptr, node_type_names=wl.node_type_names, edge_type=wl.edge_type,
              edge_type_names=wl.edge_type_names)
    c = Case(lib, model, wl.x, wl.ei, mask, gk, zero_edge_rule=True)
    c.check(c.run(), what="hetero width %d" % hidden)


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 31, 32, 33, 64])
def test_coalition_counts_and_ranges(s, lib):
    """S = 1, 31, 32, 33, 64, and sub-ranges (s0 on a word boundary) that end inside a word, and n_s = 0."""
    x, ei, mask = _rich_graph(6, s=max(s, 3))
    mask = mask[:s]
    c = Case(lib, _with_projection(_random_stack("gcn", x.shape[1], (64, 64), seed=8)), x, ei, mask)
    c.check(c.run(), what="S=%d" % s)
    for s0 in range(0, s, 32):
        for n_s in sorted({1, min(17, s - s0), s - s0}):
            c.check(c.run(s0=s0, n_s=n_s), what="S=%d range (%d, %d)" % (s, s0, n_s), s0=s0, n_s=n_s)
    assert c.run(s0=0, n_s=0).shape == (0, c.n)
