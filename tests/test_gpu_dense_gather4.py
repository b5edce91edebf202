"""The layer >= 1 transforms that load their A operand by TMA gather4 (option dense_tma = 1, csrc/dense_tc.cu) against the
register loaders (dense_tma = 0), bit for bit: the gathered fp32 rows are the tensor core's hi operand, so the MMAs see
the same operands in the same order.  Every masked-forward case below takes the gather4 form for its layer >= 1
transforms (TF32x3, chunk-major 32-float input, tile-table rows); the last two cases take the register loaders either way."""
import math
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stack(kind, f, widths, acts, seed):
    from bikg_graph_explainability_public_b200.lowering import LoweredConv, LoweredModel, LoweredRelation

    g = torch.Generator().manual_seed(seed)
    convs, d = [], f
    for h, act in zip(widths, acts):
        w = torch.randn(h, d, generator=g) / math.sqrt(d)
        b = 0.1 * torch.randn(h, generator=g)
        wr = torch.randn(h, d, generator=g) / math.sqrt(d) if kind == "sage" else None
        convs.append(LoweredConv([LoweredRelation(kind, None, w, b, wr)], h, act=act))
        d = h
    return LoweredModel(convs=convs, head=[], n_message_passing=len(widths))


def _project(model, seed):
    """The same stack followed by one random Linear(H, 1): the query value mixes every column of the last layer."""
    from bikg_graph_explainability_public_b200.lowering import LoweredModel

    g = torch.Generator().manual_seed(seed)
    h = model.convs[-1].out_dim
    head = [(torch.randn(1, h, generator=g) / math.sqrt(h), torch.randn(1, generator=g), None)]
    return LoweredModel(convs=model.convs, head=head, n_message_passing=model.n_message_passing)


def _graph(n, f, e, s, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, f, generator=g)
    ei = torch.randint(0, n, (2, e), generator=g)
    hub = torch.stack([torch.randint(0, n, (1500,), generator=g), torch.full((1500,), 3)])  # one hub row
    ei = torch.cat([ei, hub], 1)
    mask = torch.rand(s, n, generator=g) < 0.6
    mask[0] = True
    return x, ei, mask


def _pack(lib, mask):
    from bikg_graph_explainability_public_b200 import _lib

    s, n = mask.shape
    m8 = mask.to(torch.uint8).cuda().contiguous()
    w = -(-s // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
    _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, None, _lib.stream_ptr()))
    return act


def _forward(lib, model, x, ei, mask, out_col=0, graph_kw=None, zero_edge_rule=False):
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward

    gk = graph_kw or {}
    s, n = mask.shape
    graph = GraphSpec(x.cuda(), ei.cuda(), gk.get("type_ptr", [0, n]), gk.get("node_type_names"),
                      None if gk.get("edge_type") is None else gk["edge_type"].cuda(), gk.get("edge_type_names"))
    eng = MaskedForward(graph, model, list(range(n)), zero_edge_rule=zero_edge_rule, out_col=out_col)
    y = eng(_pack(lib, mask), s, 0, s)
    torch.cuda.synchronize()
    return y.cpu().numpy()


def _both(knobs, run, **opts):
    """run() with dense_tma = 1 and = 0 (other options as given); asserts bitwise equality, returns the dense_tma = 1 result."""
    knobs(dense_tma=1, **opts)
    y1 = run()
    knobs(dense_tma=0)
    y0 = run()
    np.testing.assert_array_equal(y1, y0)
    assert np.isfinite(y1).all()
    return y1


def _dense_kernels(run):
    """Names of the dense_tc kernel instantiations that run() launches."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if "dense_tc_kernel" in e.name}


@pytest.mark.parametrize("s", [1, 31, 32, 33])
def test_gather4_coalition_counts(s, lib, knobs):
    """GCN 128 -> 128 -> 128 (C3's stack) on 3000 nodes (partial last 128-row tile of every slot), ReLU, bias, the
    pre-scale of the next GCN layer on the first layer >= 1 transform; last-layer columns around the 32-float chunk
    boundaries and one projection over all columns."""
    x, ei, mask = _graph(3000, 64, 15000, s, seed=s)
    model = _stack("gcn", 64, (128, 128, 128), ("relu", "relu", None), seed=1)
    for col in (0, 31, 32, 127):
        _both(knobs, lambda: _forward(lib, model, x, ei, mask, out_col=col))
    _both(knobs, lambda: _forward(lib, _project(model, 2), x, ei, mask))


def test_gather4_path_is_taken(lib, knobs):
    x, ei, mask = _graph(3000, 64, 15000, 33, seed=7)
    model = _project(_stack("gcn", 64, (128, 128), ("relu", None), seed=3), 4)
    knobs(dense_tma=1)
    on = _dense_kernels(lambda: _forward(lib, model, x, ei, mask))
    knobs(dense_tma=0)
    off = _dense_kernels(lambda: _forward(lib, model, x, ei, mask))
    assert any("dense_tc_kernel<0, true>" in k for k in on), on
    assert not any("true" in k for k in off), off


@pytest.mark.parametrize("n", [129, 1000, 4096, 5000])
def test_gather4_node_counts(n, lib, knobs):
    """Node counts with one row past a tile, a partial tile, whole tiles, and a partial tile after many."""
    x, ei, mask = _graph(n, 32, 5 * n, 40, seed=n)
    model = _project(_stack("gcn", 32, (64, 128), ("relu", None), seed=n), 5)
    _both(knobs, lambda: _forward(lib, model, x, ei, mask))


@pytest.mark.parametrize("widths", [(64, 64), (128, 128), (256, 64), (64, 256)])
def test_gather4_widths(widths, lib, knobs):
    """K (= the layer >= 1 input width) of 64, 128, 256 and outputs of 64, 128, 256 columns; sigmoid on the last layer."""
    x, ei, mask = _graph(2000, 32, 10000, 36, seed=sum(widths))
    model = _stack("gcn", 32, widths, ("relu", "sigmoid"), seed=6)
    for col in (0, widths[-1] - 1):
        _both(knobs, lambda: _forward(lib, model, x, ei, mask, out_col=col))
    _both(knobs, lambda: _forward(lib, _project(model, 7), x, ei, mask))


def test_gather4_sage_root(lib, knobs):
    """SAGE: the root transform accumulates into the neighbour transform's output (accumulate), then ReLU."""
    x, ei, mask = _graph(2500, 48, 12000, 35, seed=9)
    model = _project(_stack("sage", 48, (128, 64, 128), ("relu", "relu", None), seed=8), 9)
    _both(knobs, lambda: _forward(lib, model, x, ei, mask))


def test_gather4_hetero(lib, knobs):
    """c4_tiny: 5 node types, 9 SAGE relations, several into one type, zero-edge rule: per-relation layer >= 1 transforms."""
    sys.path.insert(0, ROOT)
    import bench
    from bikg_graph_explainability_public_b200.lowering import lower

    wl = bench.Workload("c4_tiny")
    mask = bench.make_masks(70, wl.n, wl.c, wl.com_of, 3).bool()
    model = _project(lower(wl.make_model()), 10)
    gk = dict(type_ptr=wl.type_ptr, node_type_names=wl.node_type_names, edge_type=wl.edge_type,
              edge_type_names=wl.edge_type_names)
    for opts in ({}, {"l1_multi": 1}):
        _both(knobs, lambda: _forward(lib, model, wl.x, wl.ei, mask, graph_kw=gk, zero_edge_rule=True), **opts)


def test_register_loaders_where_gather4_does_not_apply(lib, knobs):
    """16-float chunks (cw = 16) take the register loaders with either value of the option."""
    x, ei, mask = _graph(2000, 32, 10000, 33, seed=11)
    model = _project(_stack("gcn", 32, (128, 128), ("relu", None), seed=12), 13)
    _both(knobs, lambda: _forward(lib, model, x, ei, mask), cw=16)
    knobs(dense_tma=1)
    assert not any("true" in k for k in _dense_kernels(lambda: _forward(lib, model, x, ei, mask)))


def test_dense_rows_row_major(lib, knobs):
    """xpgnn_dense_rows: row-major input without a tile table, the same result with either value of the option."""
    from bikg_graph_explainability_public_b200 import _lib

    g = torch.Generator(device="cuda").manual_seed(14)
    m, k, n = 3000, 128, 128
    a = torch.randn(m, k, device="cuda", generator=g)
    w = torch.randn(n, k, device="cuda", generator=g) / k ** 0.5
    b = torch.randn(n, device="cuda", generator=g)

    def run():
        out = torch.zeros((m, n), device="cuda")
        _lib.check(lib.xpgnn_dense_rows(a.data_ptr(), m, k, k, w.data_ptr(), b.data_ptr(), n, 1, out.data_ptr(), n, 0, 2,
                                        _lib.stream_ptr()))
        torch.cuda.synchronize()
        return out.cpu().numpy()

    _both(knobs, run)
