"""GPU parity tests: CUDA path (through the C ABI) vs the reference goldens and the oracle.

Bars (BASELINE.json north_star): coalition masks and k-hop indices bit-exact; perturbed
predictions within 1e-4 relative (fp32); importances within 1e-3 with identical community ranking.
"""
import copy
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

import golden_io as gio

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Y_RTOL, Y_ATOL = 1e-4, 1e-6      # perturbed predictions (fp32 path)
W_TOL = 1e-3                      # importances / community scores


def _run_product(case, prune):
    from bikg_graph_explainability_public_b200 import Explainer

    meta = case["meta"]
    names, pathways, pnames = gio.fresh_inputs(case)
    if meta["hetero"]:
        feat = {k: v.clone() for k, v in case["feat"].items()}
        ei = {k: v.clone() for k, v in case["edge_index"].items()}
    else:
        feat, ei = case["feat"].clone(), case["edge_index"].clone()
    arch = gio.build_arch(case)
    if "rng_state" in case["z"].files:
        torch.set_rng_state(torch.from_numpy(case["z"]["rng_state"].copy()))
    nt, et = case.get("node_types"), case.get("edge_types")
    ex = Explainer(feat, ei, arch, dict(meta["params"]), names, pathways, pnames, meta["element_type"], meta["problem"],
                   None if nt is None else nt.clone(), None if et is None else et.clone())
    ex.options = dict(prune=prune, keep_last=True)
    cfg, pdf = ex.run(meta["element"], meta["times"])
    return ex, cfg, pdf


@pytest.mark.parametrize("prune", [False, True])
@pytest.mark.parametrize("name", gio.CASES)
def test_explainer_matches_reference_golden(name, prune):
    case = gio.load_case(name)
    z, meta = case["z"], case["meta"]
    ex, cfg, pdf = _run_product(case, prune)
    last = ex._last
    r = meta["times"] - 1  # intermediates of the last repeat are kept

    # k-hop subgraph: bit exact
    assert np.array_equal(last["sub_edge_index"].cpu().numpy(), z["sub_edge_index"])
    assert last["sub_ind"] == int(z["sub_ind"])
    # coalition masks: bit exact, incl. the shuffle and the row -> community map
    co = last["coalitions"]
    gm = gio.golden_mask(case, r)
    assert co.n_coalitions == gm.shape[0] and co.batch_size == int(z["batch_size_%d" % r])
    assert np.array_equal(co.dense().cpu().numpy(), gm)
    if "pathway_rows_%d" % r in z.files:
        assert np.array_equal(co.pathway_rows.cpu().numpy(), z["pathway_rows_%d" % r])
    assert np.array_equal(co.popcount.cpu().numpy(), gm.sum(1))
    # surrogate init continues the same CPU stream: bit exact
    assert np.array_equal(last["w0"].cpu().numpy(), z["w0_%d" % r])
    # SHAP kernel weights: float64, same operation order -> exact
    assert np.array_equal(last["kernel"].cpu().numpy(), z["kernel_%d" % r])
    # perturbed predictions
    y_ref = z["y_%d" % r].reshape(-1)
    np.testing.assert_allclose(last["y"].cpu().numpy(), y_ref, rtol=Y_RTOL, atol=Y_ATOL)
    # importances, ranking
    ref_mean = dict(zip([str(x) for x in z["cfg_names"]], z["cfg_mean"]))
    got = np.array([ref_mean[str(k)] for k in cfg.index])
    np.testing.assert_allclose(cfg["config_value_mean"].values, got, atol=W_TOL, rtol=W_TOL)
    ref_std = dict(zip([str(x) for x in z["cfg_names"]], z["cfg_std"]))
    np.testing.assert_allclose(cfg["config_value_std"].values, np.array([ref_std[str(k)] for k in cfg.index]),
                               atol=W_TOL, rtol=W_TOL)
    if "pw_names" in z.files:
        assert [str(x) for x in pdf.index] == [str(x) for x in z["pw_names"]], "community ranking differs"
        np.testing.assert_allclose(pdf["score"].values, z["pw_score"], atol=W_TOL, rtol=W_TOL)
    else:
        assert pdf is None


def test_mask_stream_goldens():
    """Reference ``Mask`` outputs on shapes the end-to-end cases do not reach: N > 4000 truncation,
    capped rows, dead-mask repair (C = 2, 3).  SHA-256 of the bool matrix must match."""
    from bikg_graph_explainability_public_b200.masks import generate_coalitions

    with open(os.path.join(gio.GOLDEN, "mask_stream.json")) as f:
        specs = json.load(f)
    for sp in specs:
        params = dict(interpret_samples=sp["interpret_samples"], epochs=sp["epochs"])
        torch.manual_seed(sp["seed"] + 2)
        co = generate_coalitions(sp["n"], copy.deepcopy(sp["communities"]), params)
        m = co.dense().cpu().numpy()
        assert m.shape[0] == sp["rows"] and co.batch_size == sp["batch_size"], sp["name"]
        assert hashlib.sha256(np.ascontiguousarray(m).tobytes()).hexdigest() == sp["sha256_mask"], sp["name"]
        assert hashlib.sha256(co.pathway_rows.cpu().numpy().astype(np.int32).tobytes()).hexdigest() == sp["sha256_rows"]
        # the CPU generator must have advanced by exactly the draws the reference consumed
        from oracle.mt19937 import MT19937

        mt = MT19937(sp["seed"] + 2)
        mt.raw(sp["consumed"])
        now = torch.get_rng_state().numpy()
        assert np.array_equal(mt.to_torch_state(now), now), sp["name"]


def test_shap_kernel_goldens():
    from bikg_graph_explainability_public_b200.kernels import Kernel

    z = np.load(os.path.join(gio.GOLDEN, "shap_kernel.npz"))
    for key in [k[len("kernel_"):] for k in z.files if k.startswith("kernel_")]:
        rows, n = (int(v) for v in z["shape_" + key])
        m = np.unpackbits(z["mask_" + key], axis=1)[:, :n].astype(bool)
        k = Kernel(torch.from_numpy(m)).compute().cpu().numpy()
        assert np.array_equal(k, z["kernel_" + key]), key


def test_mt19937_stream_matches_torch():
    from bikg_graph_explainability_public_b200.rng import DeviceStream

    for seed, n in ((0, 5), (7, 624), (11, 625), (123, 100000), (2 ** 31 + 5, 3000)):
        torch.manual_seed(seed)
        torch.rand(seed % 17)  # arbitrary position inside the state block
        st = DeviceStream(torch.device("cuda"))
        d = st.draw(n)[:n].cpu().numpy().view(np.uint32)
        ref = torch.randint(0, 2, (n,), dtype=torch.bool).numpy()
        assert np.array_equal((d & 1).astype(bool), ref)
        st.hand_back()
        a = torch.randint(0, 2 ** 31 - 1, (97,))
        torch.manual_seed(seed)
        torch.rand(seed % 17)
        torch.randint(0, 2, (n,), dtype=torch.bool)
        assert torch.equal(a, torch.randint(0, 2 ** 31 - 1, (97,)))


def test_randperm_matches_torch(lib):
    from bikg_graph_explainability_public_b200 import _lib
    from bikg_graph_explainability_public_b200.rng import DeviceStream

    for n in (1, 2, 3, 1002, 50000, 60000):  # 60000 > shared-memory capacity -> global path
        torch.manual_seed(n)
        st = DeviceStream(torch.device("cuda"))
        d = st.draw(max(n - 1, 1))
        perm = torch.empty(n, dtype=torch.int32, device="cuda")
        _lib.check(lib.xpgnn_randperm(d.data_ptr(), n, perm.data_ptr(), _lib.stream_ptr()))
        assert torch.equal(perm.cpu().long(), torch.randperm(n))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_khop_matches_oracle(seed):
    from bikg_graph_explainability_public_b200.data import khop_subgraph
    from oracle.xpgnn_oracle import k_hop_subgraph

    g = torch.Generator().manual_seed(seed)
    n, e = 5000, 20000
    ei = torch.randint(0, n, (2, e), generator=g)
    ei[:, :50] = ei[:, 50:100]            # duplicates
    ei[1, 100:130] = ei[0, 100:130]       # self loops
    for hops in (0, 1, 2, 3):
        q = int(torch.randint(0, n, (1,), generator=g))
        subset, sub_ei, sub_ind, mask, hop, _ = khop_subgraph(ei.cuda(), n, q, hops)
        s2, e2, i2, m2 = k_hop_subgraph(ei.numpy(), q, hops)
        assert np.array_equal(subset.cpu().numpy(), s2)
        assert np.array_equal(sub_ei.cpu().numpy(), e2)
        assert int(sub_ind) == i2
        if m2.sum() > 0:
            assert np.array_equal(mask.cpu().numpy(), m2)


def test_khop_isolated_query_gets_self_loop():
    from bikg_graph_explainability_public_b200.data import khop_subgraph

    ei = torch.tensor([[0, 1], [1, 2]]).cuda()
    subset, sub_ei, sub_ind, mask, hop, _ = khop_subgraph(ei, 4, 0, 2)  # node 0 has no in-edge
    assert subset.tolist() == [0] and sub_ei.tolist() == [[0], [0]] and int(sub_ind) == 0


def test_khop_rejects_out_of_range_edges():
    """An endpoint outside [0, N) raises IndexError (PyG would too) instead of reading / writing out of bounds."""
    from bikg_graph_explainability_public_b200.data import khop_subgraph

    ei = torch.tensor([[0, 1, 7, 2], [1, 2, 3, -1]])
    with pytest.raises(IndexError):
        khop_subgraph(ei.cuda(), 5, 2, 2)
    subset, sub_ei, *_ = khop_subgraph(ei[:, :2].cuda(), 5, 2, 2)
    assert subset.cpu().tolist() == [0, 1, 2]


def test_csr_is_stable_and_drops_self_loops():
    from bikg_graph_explainability_public_b200.engine import build_csr

    g = torch.Generator().manual_seed(5)
    n, e = 300, 4000
    ei = torch.randint(0, n, (2, e), generator=g)
    for drop in (False, True):
        rowptr, col = build_csr(ei[0].cuda(), ei[1].cuda(), n, drop)
        rowptr, col = rowptr.cpu().numpy(), col.cpu().numpy()
        src, dst = ei[0].numpy(), ei[1].numpy()
        keep = (src != dst) if drop else np.ones(e, bool)
        order = np.argsort(dst[keep], kind="stable")
        assert rowptr[-1] == keep.sum()
        assert np.array_equal(col[: rowptr[-1]], src[keep][order])
        assert np.array_equal(np.diff(rowptr), np.bincount(dst[keep], minlength=n))


def _random_model_case(seed, kind, n=400, e=3000, f=20, hidden=(24, 24), s=150):
    """Engine vs oracle layers on a random multigraph with arbitrary (iid) coalitions."""
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
    q = int(torch.randint(0, n, (1,), generator=g))
    return x, ei, arch, mask, q


@pytest.mark.parametrize("kind", ["gcn", "sage"])
@pytest.mark.parametrize("seed", [0, 1])
def test_engine_matches_oracle_on_random_coalitions(kind, seed, lib):
    from bikg_graph_explainability_public_b200 import _lib
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(seed, kind)
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    m8 = mask.to(torch.uint8).cuda().contiguous()
    w = -(-s // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
    pop = torch.zeros(s, dtype=torch.int32, device="cuda")
    _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, pop.data_ptr(), _lib.stream_ptr()))
    assert np.array_equal(pop.cpu().numpy(), mask.sum(1).numpy())
    eng = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q])
    y = eng(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y, y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    # sub-range evaluation (what a rank of a sharded run does) gives the same rows
    y2 = eng(act, s, 64, 40)[:, 0].cpu().numpy()
    np.testing.assert_array_equal(y2, y[64:104])
    # a smaller coalition tile (memory-limited graphs) gives the same numbers
    eng8 = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q], tile_coalitions=8)
    np.testing.assert_allclose(eng8(act, s)[:, 0].cpu().numpy(), y, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("hidden", [(32, 32), (64, 128, 64), (128, 128)])
def test_fused_spmm_dense_matches_oracle(hidden, lib, knobs):
    """Layers >= 1 through the fused SpMM + tcgen05 (TF32x3) kernel, vs the oracle and vs the unfused path."""
    from bikg_graph_explainability_public_b200 import _lib
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(3, "gcn", n=700, e=6000, f=40, hidden=hidden, s=75)
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    m8 = mask.to(torch.uint8).cuda().contiguous()
    w = -(-s // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
    _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, None, _lib.stream_ptr()))
    ys = {}
    knobs(compact=0)  # the compact path would take these shapes first
    for fused in ("1", "0"):
        knobs(fused=int(fused))
        eng = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q])
        ys[fused] = eng(act, s)[:, 0].cpu().numpy()
        np.testing.assert_allclose(ys[fused], y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    np.testing.assert_allclose(ys["1"], ys["0"], rtol=2e-5, atol=1e-6)
    # 8-slot tiles in coalition-major order and a memory-limited 8-coalition tile give the same numbers
    knobs(fused=1)
    knobs(fused_sb=8)
    eng = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q], tile_coalitions=8)
    np.testing.assert_allclose(eng(act, s)[:, 0].cpu().numpy(), ys["1"], rtol=2e-5, atol=1e-6)


def _pack(lib, mask):
    from bikg_graph_explainability_public_b200 import _lib

    s, n = mask.shape
    m8 = mask.to(torch.uint8).cuda().contiguous()
    w = -(-s // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
    _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, None, _lib.stream_ptr()))
    return act


@pytest.mark.gpu
@pytest.mark.parametrize("kind,hidden,env", [
    ("gcn", (128, 128), {}),                          # row-outer layer 0 + list-driven layer 1 (the C3 shape)
    ("gcn", (128, 128), {"l0_lists": 1}),       # list-driven layer 0 with per-source weights
    ("gcn", (128, 128), {"sched_static": 1}),
    ("sage", (128, 128), {}),
    ("sage", (128, 128), {"l0_lists": 1}),
    ("gcn", (128,), {}),                              # single conv layer
    ("gcn", (16,), {}),                               # 16-wide chunks, SIMT transforms
    ("gcn", (32, 48), {}),
    ("sage", (64, 128, 64), {}),
    ("gcn", (192, 128), {}),                          # three 64-column blocks in the row-outer kernel
])
def test_compact_path_matches_oracle(kind, hidden, env, lib, knobs):
    """Compact path (compact.cu: active rows only, per-coalition compacted edge lists, chunk-major
    activations) vs the oracle and vs the tile path of engine.cu, incl. coalitions in which the query
    node is inactive (isolated chain in the head), a partial last word and memory-limited tiles."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(7, kind, n=900, e=9000, f=40, hidden=hidden, s=75)
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    y_ref = y_ref.numpy().reshape(-1)
    assert (~mask[:, q]).sum() > 5 and mask[:, q].sum() > 5   # both the active and the isolated query branch
    act = _pack(lib, mask)
    for k, v in env.items():
        knobs(**{k: v})
    g = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    eng = MaskedForward(g, lower(arch), [q, (q + 1) % n, 5])
    y = eng(act, s).cpu().numpy()
    np.testing.assert_allclose(y[:, 0], y_ref, rtol=Y_RTOL, atol=Y_ATOL)
    _, y_ref2 = kernel_output(mask.numpy(), x, ei.numpy(), arch, 5)
    np.testing.assert_allclose(y[:, 2], y_ref2.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    # sub-range (a rank's shard) and a memory-limited tile
    np.testing.assert_array_equal(eng(act, s, 32, 43).cpu().numpy(), y[32:75])
    eng8 = MaskedForward(g, lower(arch), [q, (q + 1) % n, 5], tile_coalitions=8)
    np.testing.assert_allclose(eng8(act, s).cpu().numpy(), y, rtol=1e-6, atol=1e-7)
    # the tile path of engine.cu computes every row; same predictions
    knobs(compact=0)
    legacy = MaskedForward(g, lower(arch), [q, (q + 1) % n, 5])
    np.testing.assert_allclose(legacy(act, s).cpu().numpy(), y, rtol=2e-5, atol=1e-6)


@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_compact_path_hub_rows(kind, lib, knobs):
    """Destination rows above the long-row threshold (1024 in-edges) are processed by whole CTAs in the compact
    path (hub rows of power-law graphs), in layer 0 cut into slices of 4096 in-edges whose partial sums a second kernel
    adds in slice order; same predictions as the oracle and as the tile path."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(9, kind, n=4000, e=30000, f=32, hidden=(128, 128), s=40)
    g = torch.Generator().manual_seed(5)
    n = x.shape[0]
    hubs = [q, 7, 1234]
    extra = [torch.stack([torch.randint(0, n, (k,), generator=g), torch.full((k,), h)]) for h, k in zip(hubs, (9000, 4100, 1100))]  # 3, 2 and 1 slices of 4096 in-edges in layer 0
    ei = torch.cat([ei] + extra, 1)
    s = mask.shape[0]
    mask[2, q] = True
    mask[3, q] = False
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    act = _pack(lib, mask)
    gs = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    y = MaskedForward(gs, lower(arch), [q, 7])(act, s).cpu().numpy()
    np.testing.assert_allclose(y[:, 0], y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    _, y_ref7 = kernel_output(mask.numpy(), x, ei.numpy(), arch, 7)
    np.testing.assert_allclose(y[:, 1], y_ref7.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    # pruned mode (what Explainer.run uses): the last layer is ONE hub row -- its in-edges are sliced over many CTAs
    from bikg_graph_explainability_public_b200.data import khop_subgraph
    hop = khop_subgraph(ei.cuda(), n, q, 3)[4]
    yp = MaskedForward(gs, lower(arch), [q], prune=True, hop=hop)(act, s).cpu().numpy()
    np.testing.assert_allclose(yp[:, 0], y[:, 0], rtol=2e-5, atol=1e-6)
    yp2 = MaskedForward(gs, lower(arch), [q], prune=True, hop=hop)(act, s).cpu().numpy()
    np.testing.assert_array_equal(yp2, yp)  # slices are added in a fixed order
    np.testing.assert_array_equal(MaskedForward(gs, lower(arch), [q, 7])(act, s).cpu().numpy(), y)  # slices add in a fixed order
    knobs(l0_slices=0)   # one CTA per hub row
    np.testing.assert_allclose(MaskedForward(gs, lower(arch), [q, 7])(act, s).cpu().numpy(), y, rtol=2e-5, atol=1e-6)
    knobs(long_rows=0)   # hub rows through the row-per-warp kernels
    np.testing.assert_allclose(MaskedForward(gs, lower(arch), [q, 7])(act, s).cpu().numpy(), y, rtol=2e-5, atol=1e-6)
    knobs(compact=0)
    np.testing.assert_allclose(MaskedForward(gs, lower(arch), [q, 7])(act, s).cpu().numpy(), y, rtol=2e-5, atol=1e-6)


@pytest.mark.parametrize("kind", ["gcn", "sage"])
@pytest.mark.parametrize("seg", ["0", "4", "6", "7", "8", "12", "16", "116", "124", "216", "232", "316", "332", "432", "516", "532", "8t"])
def test_segmented_spmm_variants(kind, seg, lib, knobs):
    """Layers >= 1 through the segmented SpMM (cspmm_seg_kernel: a warp sums the gather stream of a 32-row block in four
    pieces cut at row boundaries) with 4 .. 16 gathers in flight per lane, through its shared-memory ring variant (116 / 124:
    cp.async into 16 / 24 slots per group), through the warp-specialised kernel of compact_bulk.cu (2xx bulk copies, 3xx / 4xx
    cp.async, 5xx TMA gather4; 16- and 32-stage rings: rows longer than the ring), through the hybrid launch ("8t": gather4
    kernel next to the segmented one) and through the row-lockstep kernel (0): medium hubs
    (80-240 active in-edges, below the long-row threshold) make blocks longer than one staging round, rows cut by piece
    and round boundaries, empty rows (SAGE) and a short last block; vs the oracle, bitwise repeatable."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(21, kind, n=3001, e=9000, f=32, hidden=(128, 128, 64), s=45)
    g = torch.Generator().manual_seed(77)
    n = x.shape[0]
    hubs = [q, 5, 6, 7, 8, 1500, 2999, 3000]
    extra = [torch.stack([torch.randint(0, n, (k,), generator=g), torch.full((k,), h)])
             for h, k in zip(hubs, (900, 400, 800, 333, 950, 700, 600, 850))]
    ei = torch.cat([ei] + extra, 1)
    s = mask.shape[0]
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    act = _pack(lib, mask)
    knobs(seg=int(seg.rstrip("t")), seg_tma=int(seg.endswith("t")))  # "t": TMA gather4 kernel next to the segmented kernel
    gs = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    eng = MaskedForward(gs, lower(arch), [q, 5, 3000])
    y = eng(act, s).cpu().numpy()
    np.testing.assert_allclose(y[:, 0], y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    _, y_ref5 = kernel_output(mask.numpy(), x, ei.numpy(), arch, 5)
    np.testing.assert_allclose(y[:, 1], y_ref5.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    if not seg.endswith("t"):  # hybrid: rows longer than a staging round are summed in a different order by the two kernels
        np.testing.assert_array_equal(eng(act, s).cpu().numpy(), y)


@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_compact_path_without_edges(kind, lib):
    """Only self loops in the input: GCN drops them (zero edges left, every node is its own unit loop), SAGE keeps
    them.  Empty coalitions and empty rows through the compaction, the SpMM and the tile table."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle import fixture_models as fm
    from oracle.xpgnn_oracle import kernel_output

    g = torch.Generator().manual_seed(2)
    n, f, s = 300, 24, 40
    x = torch.randn(n, f, generator=g)
    ei = torch.arange(n).repeat(2, 1)
    arch = (fm.HomoGCN(f, (32, 32), (32, 8, 1), seed=1) if kind == "gcn" else fm.HomoSAGE(f, (32, 32), (32, 1), seed=1)).eval()
    mask = torch.rand(s, n, generator=g) < 0.5
    mask[0] = True
    mask[1] = False
    q = 11
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    y = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q])(_pack(lib, mask), s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y, y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)


def test_compact_path_is_deterministic(lib):
    """Dynamic work scheduling and the CTA-level reductions of hub rows add in a fixed order: bitwise equal runs."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower

    x, ei, arch, mask, q = _random_model_case(4, "gcn", n=5000, e=60000, f=32, hidden=(128, 128), s=64)
    g = torch.Generator().manual_seed(8)
    n = x.shape[0]
    ei = torch.cat([ei, torch.stack([torch.randint(0, n, (4000,), generator=g), torch.full((4000,), q)])], 1)
    act = _pack(lib, mask)
    eng = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q, 3])
    y0 = eng(act, 64).cpu().numpy()
    for _ in range(3):
        np.testing.assert_array_equal(eng(act, 64).cpu().numpy(), y0)


@pytest.mark.parametrize("seed", list(range(8)))
def test_compact_path_randomized(seed, lib, knobs):
    """Random configurations (conv kind, depth / widths, hubs, coalition count, tile size, query set): compact path vs
    the oracle and vs the tile path."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    rng = np.random.default_rng(100 + seed)
    kind = ["gcn", "sage"][seed % 2]
    hidden = [(64,), (128, 64), (32, 32, 32), (16, 48), (128, 128), (64, 192), (256, 128), (48,)][seed]
    n = int(rng.integers(300, 3000))
    e = int(rng.integers(2 * n, 12 * n))
    s = int(rng.integers(1, 100))
    x, ei, arch, mask, q = _random_model_case(50 + seed, kind, n=n, e=e, f=int(rng.choice([20, 32, 64])), hidden=hidden, s=max(s, 2))
    g = torch.Generator().manual_seed(seed)
    if seed % 3 != 2:  # hub rows above the long-row thresholds
        for hub, k in ((q, 1500), (int(rng.integers(0, n)), 2600)):
            ei = torch.cat([ei, torch.stack([torch.randint(0, n, (k,), generator=g), torch.full((k,), hub)])], 1)
    mask = mask[:max(s, 2)]
    s = mask.shape[0]
    mask[rng.integers(0, s)] = torch.rand(n, generator=g) < 0.05   # a sparse coalition
    queries = [q] + rng.integers(0, n, size=int(rng.integers(0, 3))).tolist()
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    act = _pack(lib, mask)
    gs = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    tile = [None, 8, 4, 16][seed % 4]
    y = MaskedForward(gs, lower(arch), queries, tile_coalitions=tile)(act, s).cpu().numpy()
    np.testing.assert_allclose(y[:, 0], y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    knobs(compact=0)
    y_tile = MaskedForward(gs, lower(arch), queries)(act, s).cpu().numpy()
    np.testing.assert_allclose(y_tile, y, rtol=3e-5, atol=1e-6)
    knobs(compact=1)
    if kind == "gcn" and all(h % 64 == 0 for h in hidden):  # bf16 activation storage where it applies
        y16 = MaskedForward(gs, lower(arch), queries, precision="bf16_act", tile_coalitions=tile)(act, s).cpu().numpy()
        np.testing.assert_allclose(y16, y, rtol=2e-2, atol=2e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_layer0_kernel_variants_agree(kind, lib, knobs):
    """The layer-0 row kernels (option l0_ws = 0 one warp per row, 1 warp specialised with column blocks, 2 warp
    specialised with slot x column tiles, 3 = 1 with the Z pieces staged by TMA bulk copies) do the same FMAs in the same order: outputs agree to rounding of the epilogue,
    on a graph with isolated rows, rows longer than one stage (> 16 / > 32 in-edges) and more than 16 active slots."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(11, kind, n=3000, e=60000, f=32, hidden=(128, 128), s=64)
    ei[1, :6000] = ei[1, :6000] % 50          # 50 rows with ~120 extra in-edges: several stages per pass
    mask[:, ::7] = True                       # every 7th node active in all 32 slots of a word: two slot blocks
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    y_ref = y_ref.numpy().reshape(-1)
    act = _pack(lib, mask)
    g = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    ys = []
    for mode in ("0", "1", "2", "3"):
        knobs(l0_ws=int(mode))
        y = MaskedForward(g, lower(arch), [q, 3])(act, s).cpu().numpy()
        np.testing.assert_allclose(y[:, 0], y_ref, rtol=Y_RTOL, atol=Y_ATOL)
        ys.append(y)
    np.testing.assert_allclose(ys[1], ys[0], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(ys[2], ys[0], rtol=2e-6, atol=1e-7)
    np.testing.assert_array_equal(ys[3], ys[1])  # same kernel, another copy engine


@pytest.mark.parametrize("name", ["c4_tiny", "c2_wide", "c2_wide2"])
def test_hetero_compact_path_matches_oracle(name, lib, knobs):
    """Hetero compact path (per-relation compaction, relations into one destination type accumulate, merged root
    transform, isolated chain of typed queries, zero-edge rule) vs the oracle and vs the per-relation tile path."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    wl = bench.Workload(name)
    s = 70
    mask = bench.make_masks(s, wl.n, wl.c, wl.com_of, 3).bool()
    mask[5] = False                      # a coalition without any active edge (zero-edge rule of the multi-type branch)
    mask[6] = True
    arch, eng = wl.engine(torch.device("cuda", 0), "fp32")
    om = wl.oracle_model(arch)
    y_ref = wl.oracle_eval(om, mask.numpy())
    act = _pack(lib, mask)
    y = eng(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y, y_ref, rtol=Y_RTOL, atol=Y_ATOL)
    np.testing.assert_array_equal(eng(act, s, 32, 38)[:, 0].cpu().numpy(), y[32:70])
    knobs(l1_multi=0)   # layers >= 1 aggregate-first relation by relation instead of transform-first per type
    np.testing.assert_allclose(eng(act, s)[:, 0].cpu().numpy(), y, rtol=3e-5, atol=1e-6)
    knobs(l0_multi=0)   # layer 0 relation by relation (accumulate / finish) instead of one pass per type
    np.testing.assert_allclose(eng(act, s)[:, 0].cpu().numpy(), y, rtol=3e-5, atol=1e-6)
    knobs(compact_hetero=0)
    _, eng_tile = wl.engine(torch.device("cuda", 0), "fp32")
    np.testing.assert_allclose(eng_tile(act, s)[:, 0].cpu().numpy(), y, rtol=3e-5, atol=1e-6)


@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_bf16_transform_mode_within_tolerance(kind, lib):
    """precision="bf16": dense transforms on tcgen05 with bf16 operands (fp32 accumulate, fp32 storage).
    Bar from BASELINE.json north_star: predictions within 2e-2 relative."""
    from bikg_graph_explainability_public_b200 import _lib
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(5, kind, n=2000, e=16000, f=64, hidden=(64, 128), s=40)
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    m8 = mask.to(torch.uint8).cuda().contiguous()
    w = -(-s // 32)
    act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
    _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, None, _lib.stream_ptr()))
    eng = MaskedForward(GraphSpec(x.cuda(), ei.cuda(), [0, n]), lower(arch), [q], precision="bf16")
    y = eng(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y, y_ref.numpy().reshape(-1), rtol=2e-2, atol=2e-3)


def test_bf16_activation_storage_within_tolerance(lib):
    """precision="bf16_act": bf16 tensor-core transforms and bf16 storage of the per-coalition activations in the
    compact path (fp32 accumulation everywhere).  Bar from BASELINE.json north_star: predictions within 2e-2 relative."""
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(6, "gcn", n=3000, e=30000, f=64, hidden=(128, 128), s=70)
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    act = _pack(lib, mask)
    g = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    y = MaskedForward(g, lower(arch), [q], precision="bf16_act")(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y, y_ref.numpy().reshape(-1), rtol=2e-2, atol=2e-3)
    y32 = MaskedForward(g, lower(arch), [q], precision="fp32")(act, s)[:, 0].cpu().numpy()
    assert np.max(np.abs(y - y32)) > 0, "the bf16 storage path was not taken"
    # memory-limited tiles and sub-ranges give the same numbers
    y8 = MaskedForward(g, lower(arch), [q], precision="bf16_act", tile_coalitions=8)(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y8, y, rtol=1e-6, atol=1e-7)


def test_fp32_exact_transforms_option(lib):
    """precision="fp32_exact": the dense transforms run as exact fp32 FMAs (not 3xTF32 tensor-core products): tighter
    against the oracle than the 1e-4 bar needs, and the engine option it sets is restored after every call."""
    import ctypes as C

    from bikg_graph_explainability_public_b200 import _lib
    from bikg_graph_explainability_public_b200.engine import GraphSpec, MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower
    from oracle.xpgnn_oracle import kernel_output

    x, ei, arch, mask, q = _random_model_case(9, "gcn", n=3000, e=30000, f=64, hidden=(128, 128), s=40)
    s, n = mask.shape
    _, y_ref = kernel_output(mask.numpy(), x, ei.numpy(), arch, q)
    act = _pack(lib, mask)
    g = GraphSpec(x.cuda(), ei.cuda(), [0, n])
    y = MaskedForward(g, lower(arch), [q], precision="fp32_exact")(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y, y_ref.numpy().reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    y_tc = MaskedForward(g, lower(arch), [q], precision="fp32")(act, s)[:, 0].cpu().numpy()
    np.testing.assert_allclose(y_tc, y, rtol=Y_RTOL, atol=Y_ATOL)
    v = C.c_int32(-1)
    _lib.check(lib.xpgnn_get_option(b"dense_simt", C.byref(v)))
    assert v.value == 0


def test_wlm_fit_matches_closed_form(lib):
    """Fit kernels vs the oracle's torch-autograd port on random data, both target layouts."""
    from bikg_graph_explainability_public_b200 import _lib
    from bikg_graph_explainability_public_b200.masks import CoalitionSet
    from bikg_graph_explainability_public_b200.wlm import fit_surrogate
    from oracle.xpgnn_oracle import shap_kernel, train_wlm

    g = torch.Generator().manual_seed(3)
    params = dict(optimizer="adam", lr=0.01, lr_patience=10, l1_lambda=1e-4)
    for n, s, b in ((15, 1002, 20), (3000, 257, 33)):
        mask = torch.rand(s, n, generator=g) < 0.5
        y = torch.rand(s, generator=g)
        kern = shap_kernel(mask.numpy())
        w0 = (torch.rand(n, generator=g) - 0.5) * 0.2
        w = -(-s // 32)
        act = torch.zeros((n, w), dtype=torch.int32, device="cuda")
        pop = torch.zeros(s, dtype=torch.int32, device="cuda")
        m8 = mask.to(torch.uint8).cuda().contiguous()
        _lib.check(lib.xpgnn_pack_mask(m8.data_ptr(), s, n, act.data_ptr(), w, pop.data_ptr(), _lib.stream_ptr()))
        co = CoalitionSet(act, pop, s, n, b)
        for broadcast in (True, False):
            batches = [(mask[i:i + b].numpy(), kern[i:i + b], y[i:i + b].reshape(-1, 1) if broadcast else y[i:i + b])
                       for i in range(0, s, b)]
            w_ref, losses_ref = train_wlm(batches, w0.numpy(), params)
            w_dev, losses = fit_surrogate(co, y.cuda(), torch.from_numpy(kern).cuda(), w0.cuda(), params, broadcast)
            np.testing.assert_allclose(w_dev.cpu().numpy(), w_ref.numpy(), atol=2e-5, rtol=1e-3)
            np.testing.assert_allclose(losses, losses_ref, rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("name", ["c3_tenth", "c4_small"])
def test_parity_at_bench_scale(name, lib, knobs):
    """The bench workloads at 1/10 (C3: 100 k nodes / 2 M edges, 2 x GCN(128)) and 1/50 (C4: 5 node types / 20 relations /
    40 k nodes / 1 M edges, 2 x HeteroConv(SAGE)) scale: compact / hetero-compact path, tile path and pruned tile path
    against the oracle on 8 coalitions of the bench's row family incl. an all-off row, an all-on row and rows in which the
    query node is inactive.  Bar: 1e-4 relative (BASELINE.json north_star, fp32)."""
    sys.path.insert(0, ROOT)
    import bench
    from bikg_graph_explainability_public_b200.data import khop_subgraph
    from bikg_graph_explainability_public_b200.engine import MaskedForward
    from bikg_graph_explainability_public_b200.lowering import lower

    wl = bench.Workload(name)
    dev = torch.device("cuda", 0)
    arch, eng = wl.engine(dev, "fp32")
    q = wl.queries[0]
    mask = bench.make_masks(8, wl.n, wl.c, wl.com_of, 77, wl.com_of2).bool()
    mask[1] = False
    mask[2] = True
    mask[3, q] = False
    mask[4, q] = True
    assert (~mask[:, q]).sum() >= 2 and mask[:, q].sum() >= 2
    y_ref = wl.oracle_eval(wl.oracle_model(arch), mask.numpy())
    act = _pack(lib, mask)

    def rel(y):
        return float(np.max(np.abs(y - y_ref) / np.maximum(np.abs(y_ref), 1e-6)))

    y = eng(act, 8)[:, 0].cpu().numpy()
    assert rel(y) <= 1e-4, ("compact path", rel(y))
    hop = khop_subgraph(wl.ei.cuda(), wl.n, q, len(eng.edges_per_layer) + 1)[4]
    pruned = MaskedForward(eng.graph, lower(arch), [q], prune=True, hop=hop, zero_edge_rule=wl.kind == "hetero_sage")
    yp = pruned(act, 8)[:, 0].cpu().numpy()
    assert rel(yp) <= 1e-4, ("pruned tile path", rel(yp))
    knobs(compact=0)
    tile = MaskedForward(eng.graph, lower(arch), [q], prune=False, zero_edge_rule=wl.kind == "hetero_sage")
    yt = tile(act, 8)[:, 0].cpu().numpy()
    assert rel(yt) <= 1e-4, ("tile path", rel(yt))


def test_bench_dump_outputs_are_the_timed_predictions(lib, tmp_path):
    """``bench.py --dump-outputs`` writes the predictions of its timed path: one row per coalition of the job (40 rows:
    the second 32-row word is partial), equal to the oracle on the same seeded coalitions, regenerated here with
    bench.make_packed_masks and bench's seed of rank 0."""
    import subprocess

    sys.path.insert(0, ROOT)
    import bench

    rows = 40
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--coalitions", str(rows),
                          "--steps", "2", "--warmup", "1", "--no-query-leg", "--no-cpu-baseline", "--dump-outputs",
                          str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    y = np.load(tmp_path / "predictions.npy")
    wl = bench.Workload("tiny")
    assert y.shape == (rows, len(wl.queries)) and y.dtype == np.float32
    _, sample = bench.make_packed_masks(lib, rows, wl.n, wl.c, wl.com_of, 1000, torch.device("cuda", 0), wl.com_of2,
                                        keep_rows=rows)
    y_ref = wl.oracle_eval(wl.oracle_model(wl.make_model()), sample.numpy())
    np.testing.assert_allclose(y[:, 0], y_ref, rtol=Y_RTOL, atol=Y_ATOL)
