"""Explainer.run_batch: many queries through one k-hop call, one engine and one batched surrogate fit.

The multi-query k-hop and the batched fit must be bit-identical to their single-query entry points; run_batch must
give what a loop of run gives (masks, SHAP weights, sub-graphs exact; predictions within the fp32 bar) and leave the
global CPU generator where that loop leaves it.  The community resolution test runs without a GPU.
"""
import copy
import random

import numpy as np
import pytest
import torch

import golden_io as gio

Y_RTOL, Y_ATOL = 1e-4, 1e-6
W_TOL = 1e-3


# ---------------------------------------------------------------- community resolution (CPU)
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_community_index_matches_resolve_indices(seed):
    from bikg_graph_explainability_public_b200.pathways import CommunityIndex, Pathways

    rng = random.Random(seed)
    n = 300
    pool = ["g%d" % rng.randrange(180) for _ in range(n)]  # about 40 % of the names repeat
    names = pool if seed != 2 else [int(x[1:]) for x in pool]  # non-str names go through numpy's str conversion
    comms = [[rng.choice(pool) for _ in range(rng.randrange(1, 25))] + ["absent%d" % i] for i in range(40)]
    if seed == 2:
        comms = [[int(m[1:]) if m.startswith("g") else m for m in c] for c in comms]
    cnames = ["c%d" % i for i in range(len(comms))]
    index = CommunityIndex(comms, cnames, names)
    for _ in range(30):
        subset = np.sort(np.array(rng.sample(range(n), rng.randrange(1, n))))
        sub_names = np.array(names, dtype=str)[subset].tolist()
        want = Pathways(copy.deepcopy(comms), cnames).resolve_indices(sub_names)
        assert index.resolve(subset) == want
    assert index.resolve(np.array([], dtype=np.int64)) == ([], [])


# ---------------------------------------------------------------- multi-query k-hop
def _random_graph(seed, n=3000, e=12000):
    g = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, n, (2, e), generator=g)
    ei[:, :60] = ei[:, 60:120]           # duplicate edges
    ei[1, 200:240] = ei[0, 200:240]      # self loops
    isolated = n - 1                      # no edge touches the last node
    ei[ei == isolated] = 0
    return ei, n, isolated, g


def _check_multi_vs_single(ei, n, queries, hops):
    from bikg_graph_explainability_public_b200.data import khop_subgraph, khop_subgraph_multi

    mk = khop_subgraph_multi(ei.cuda(), n, queries, hops)
    assert len(mk) == len(queries)
    for q, node in enumerate(queries):
        subset, sub_ei, sub_ind, mask, hop, _ = khop_subgraph(ei.cuda(), n, node, hops)
        s2, e2, i2, lev2, eid2 = mk.block(q)
        assert torch.equal(s2, subset)
        assert torch.equal(e2, sub_ei)
        assert i2 == int(sub_ind)
        assert torch.equal(lev2, hop[subset])
        kept = torch.nonzero(mask).flatten()
        if kept.numel():
            assert torch.equal(eid2, kept)
        else:
            assert eid2.tolist() == [-1]
    return mk


@pytest.mark.gpu
@pytest.mark.parametrize("hops", [0, 1, 2, 3])
@pytest.mark.parametrize("nq", [1, 2, 31, 63, 64])
def test_khop_multi_matches_single_calls(nq, hops):
    ei, n, isolated, g = _random_graph(nq * 7 + hops)
    queries = torch.randint(0, n, (nq,), generator=g).tolist()
    if nq >= 2:
        queries[-1] = queries[0]      # a repeated query
    if nq >= 31:
        queries[5] = isolated         # self-loop rule
    _check_multi_vs_single(ei, n, queries, hops)


@pytest.mark.gpu
def test_khop_multi_without_edges_and_bad_edges():
    from bikg_graph_explainability_public_b200.data import khop_subgraph_multi

    mk = _check_multi_vs_single(torch.zeros((2, 0), dtype=torch.int64), 10, [3, 3, 7], 2)
    assert mk.edge_index.tolist() == [[0, 1, 2], [0, 1, 2]]
    ei = torch.tensor([[0, 1, 7, 2], [1, 2, 3, -1]])
    with pytest.raises(IndexError):
        khop_subgraph_multi(ei.cuda(), 5, [2, 1], 2)
    with pytest.raises(IndexError):
        khop_subgraph_multi(ei[:, :2].cuda(), 5, [2, 5], 2)
    _check_multi_vs_single(ei[:, :2], 5, [2, 0], 2)


# ---------------------------------------------------------------- batched surrogate fit
@pytest.mark.gpu
@pytest.mark.parametrize("broadcast_y", [0, 1])
@pytest.mark.parametrize("shapes", [
    [(40, 100, 20)],                                                # Q = 1
    [(40, 100, 20), (2500, 333, 64), (7, 50, 80), (300, 256, 64)],  # S % 32 != 0, S < batch, S % batch == 0, N > 2048
    [(5000, 1000, 97), (3, 31, 31), (4100, 65, 8), (64, 4000, 1000), (129, 1, 1)],
])
def test_wlm_fit_batch_matches_single_fits(shapes, broadcast_y, lib):
    from bikg_graph_explainability_public_b200 import _lib

    g = torch.Generator().manual_seed(len(shapes) * 10 + broadcast_y)
    w_max = max(-(-s // 32) for _, s, _ in shapes) + 1
    n_u = sum(n for n, _, _ in shapes)
    s_max = max(s for _, s, _ in shapes)
    nq = len(shapes)
    act = torch.randint(-2 ** 31, 2 ** 31 - 1, (n_u, w_max), generator=g, dtype=torch.int64).to(torch.int32).cuda()
    y = torch.rand((s_max, nq), generator=g).cuda()
    descs, kerns, w0s, losses, want = [], [], [], [], []
    n0 = koff = woff = 0
    for q, (n, s, b) in enumerate(shapes):
        kern = (torch.rand(s, generator=g, dtype=torch.float64) + 0.01).cuda()
        w0 = (torch.rand(n, generator=g) - 0.5).cuda()
        loss_q = torch.zeros(-(-s // b), dtype=torch.float64, device="cuda")
        d = _lib.FitQuery()
        d.act_off, d.y_off, d.kern_off, d.w_off, d.n, d.s, d.batch, d.losses = n0 * w_max, q, koff, woff, n, s, b, loss_q.data_ptr()
        descs.append(d)
        kerns.append(kern)
        w0s.append(w0)
        losses.append(loss_q)
        # the single fit on the query's own act / y
        a_q = act[n0:n0 + n, : -(-s // 32)].contiguous()
        y_q = y[:s, q].contiguous()
        w_q = w0.clone()
        l_q = torch.zeros_like(loss_q)
        _lib.check(lib.xpgnn_wlm_fit(a_q.data_ptr(), a_q.shape[1], n, s, b, y_q.data_ptr(), kern.data_ptr(), w_q.data_ptr(), 0.01,
                                     1e-4, 1e-2, broadcast_y, l_q.data_ptr(), _lib.stream_ptr()))
        want.append((w_q, l_q))
        n0 += n
        koff += s
        woff += n
    kern_all, w_all = torch.cat(kerns), torch.cat(w0s)
    arr = (_lib.FitQuery * nq)(*descs)
    launches = _lib.launch_count()
    _lib.check(lib.xpgnn_wlm_fit_batch(act.data_ptr(), w_max, y.data_ptr(), nq, kern_all.data_ptr(), w_all.data_ptr(), arr, nq,
                                       0.01, 1e-4, 1e-2, broadcast_y, _lib.stream_ptr()))
    assert _lib.launch_count() - launches == 3 * max(-(-s // b) for _, s, b in shapes)
    woff = 0
    for q, (n, s, b) in enumerate(shapes):
        assert torch.equal(w_all[woff:woff + n], want[q][0]), q
        assert torch.equal(losses[q], want[q][1]), q
        woff += n


# ---------------------------------------------------------------- run_batch vs a loop of run
BATCH_CASES = ["c1_homo_gcn", "c1_homo_gcn_times3", "gcn2_random", "sage2_shapley", "c2_hetero_gcn", "c2_dict_out"]


def _inputs(case, isolated):
    """Fresh copies of the case's inputs; ``isolated`` appends a node without edges (in the first community, so that a
    community-mode query on it has a community; no other query's graph contains it)."""
    meta = case["meta"]
    names, pathways, pnames = gio.fresh_inputs(case)
    if meta["hetero"]:
        feat = {k: v.clone() for k, v in case["feat"].items()}
        ei = {k: v.clone() for k, v in case["edge_index"].items()}
    else:
        feat, ei = case["feat"].clone(), case["edge_index"].clone()
        if isolated:
            feat = torch.cat([feat, feat[:1]])
            names = names + ["isolated"]
            if pathways is not None:
                pathways[0] = pathways[0] + ["isolated"]
    return feat, ei, names, pathways, pnames


def _elements(case):
    meta = case["meta"]
    names = meta["names"] if isinstance(meta["names"], list) else list(meta["names"].values())[0]
    if meta["hetero"]:
        ei = torch.cat(list(case["edge_index"].values()), 1)
    else:
        ei = case["edge_index"]
    deg = torch.bincount(ei[1], minlength=len(names))
    hub = names[int(deg.argmax())]
    other = names[(names.index(meta["element"]) + 7) % len(names)]
    els = [meta["element"], hub, other, meta["element"]]
    if not meta["hetero"]:
        # the one-type dict path of run cannot explain an isolated node (its edge types select no self loop), so the
        # isolated query is a homogeneous-graph case
        els.insert(2, "isolated")
    return els


def _explainer(case, isolated, prune, extra_opts=None):
    from bikg_graph_explainability_public_b200 import Explainer

    meta = case["meta"]
    feat, ei, names, pathways, pnames = _inputs(case, isolated)
    with torch.random.fork_rng(devices=[]):  # building the module draws its default init from the global generator
        arch = gio.build_arch(case)
    ex = Explainer(feat, ei, arch, dict(meta["params"]), names, pathways, pnames, meta["element_type"], meta["problem"])
    ex.options = dict(prune=prune, keep_last=True, **(extra_opts or {}))
    return ex


def _initial_rng(case):
    if "rng_state" in case["z"].files:
        return torch.from_numpy(case["z"]["rng_state"].copy())
    torch.manual_seed(1234)
    return torch.get_rng_state()


def _sequential(case, elements, prune):
    isolated = "isolated" in elements
    torch.set_rng_state(_initial_rng(case))
    out, lasts = [], []
    for e in elements:
        ex = _explainer(case, isolated, prune)
        out.append(ex.run(e, case["meta"]["times"]))
        lasts.append(ex._last)
    return out, lasts, torch.get_rng_state()


def _assert_same_explanation(got, want, last_got, last_want, tag):
    cg, pg = got
    cw, pw = want
    co_g, co_w = last_got["coalitions"], last_want["coalitions"]
    assert co_g.n_coalitions == co_w.n_coalitions and co_g.batch_size == co_w.batch_size, tag
    assert torch.equal(co_g.dense(), co_w.dense()), tag
    assert torch.equal(co_g.popcount, co_w.popcount), tag
    if co_w.pathway_rows is not None:
        assert torch.equal(co_g.pathway_rows, co_w.pathway_rows), tag
    assert torch.equal(last_got["w0"].cpu(), last_want["w0"].cpu()), tag
    assert torch.equal(last_got["kernel"], last_want["kernel"]), tag
    assert torch.equal(last_got["sub_edge_index"], last_want["sub_edge_index"]), tag
    assert last_got["sub_ind"] == last_want["sub_ind"], tag
    assert last_got["subset_names"] == last_want["subset_names"], tag
    yg, yw = last_got["y"].cpu().numpy(), last_want["y"].cpu().numpy()
    print("%s: max |y_batch - y_run| = %.3g" % (tag, float(np.max(np.abs(yg - yw))) if yw.size else 0.0))
    np.testing.assert_allclose(yg, yw, rtol=Y_RTOL, atol=Y_ATOL, err_msg=tag)
    assert sorted(map(str, cg.index)) == sorted(map(str, cw.index)), tag
    cg = cg.loc[cw.index]
    for col in ("config_value_mean", "config_value_std"):
        np.testing.assert_allclose(cg[col].values, cw[col].values, atol=W_TOL, rtol=W_TOL, err_msg=tag)
    if pw is None:
        assert pg is None, tag
    else:
        assert [str(x) for x in pg.index] == [str(x) for x in pw.index], tag + ": community order differs"
        np.testing.assert_allclose(pg["score"].values, pw["score"].values, atol=W_TOL, rtol=W_TOL, err_msg=tag)


def _assert_meets_golden(case, cfg, pdf, last):
    """The golden element's explanation against the reference fixture (the bars of test_explainer_matches_reference_golden)."""
    z, meta = case["z"], case["meta"]
    r = meta["times"] - 1
    assert np.array_equal(last["sub_edge_index"].cpu().numpy(), z["sub_edge_index"])
    assert last["sub_ind"] == int(z["sub_ind"])
    co = last["coalitions"]
    gm = gio.golden_mask(case, r)
    assert co.n_coalitions == gm.shape[0] and co.batch_size == int(z["batch_size_%d" % r])
    assert np.array_equal(co.dense().cpu().numpy(), gm)
    if "pathway_rows_%d" % r in z.files:
        assert np.array_equal(co.pathway_rows.cpu().numpy(), z["pathway_rows_%d" % r])
    assert np.array_equal(last["w0"].cpu().numpy(), z["w0_%d" % r])
    assert np.array_equal(last["kernel"].cpu().numpy(), z["kernel_%d" % r])
    np.testing.assert_allclose(last["y"].cpu().numpy(), z["y_%d" % r].reshape(-1), rtol=Y_RTOL, atol=Y_ATOL)
    ref_mean = dict(zip([str(x) for x in z["cfg_names"]], z["cfg_mean"]))
    np.testing.assert_allclose(cfg["config_value_mean"].values, np.array([ref_mean[str(k)] for k in cfg.index]),
                               atol=W_TOL, rtol=W_TOL)
    ref_std = dict(zip([str(x) for x in z["cfg_names"]], z["cfg_std"]))
    np.testing.assert_allclose(cfg["config_value_std"].values, np.array([ref_std[str(k)] for k in cfg.index]),
                               atol=W_TOL, rtol=W_TOL)
    if "pw_names" in z.files:
        assert [str(x) for x in pdf.index] == [str(x) for x in z["pw_names"]], "community ranking differs"
        np.testing.assert_allclose(pdf["score"].values, z["pw_score"], atol=W_TOL, rtol=W_TOL)
    else:
        assert pdf is None


@pytest.mark.gpu
@pytest.mark.parametrize("prune", [False, True])
@pytest.mark.parametrize("name", BATCH_CASES)
def test_run_batch_matches_sequential_run(name, prune):
    case = gio.load_case(name)
    elements = _elements(case)
    want, lasts, rng_after = _sequential(case, elements, prune)
    torch.set_rng_state(_initial_rng(case))
    ex = _explainer(case, "isolated" in elements, prune)
    got = ex.run_batch(elements, case["meta"]["times"])
    assert torch.equal(torch.get_rng_state(), rng_after)
    assert len(got) == len(elements) and len(ex._last_batch) == len(elements) and len(ex.last_stats) == len(elements)
    for i, e in enumerate(elements):
        _assert_same_explanation(got[i], want[i], ex._last_batch[i], lasts[i], "%s[%d]=%s" % (name, i, e))
    _assert_meets_golden(case, got[0][0], got[0][1], ex._last_batch[0])


@pytest.mark.gpu
def test_run_batch_groups():
    """70 queries need two k-hop groups; a forced group size of 5 must give the same explanations as 64."""
    case = gio.load_case("gcn2_random")
    names = case["meta"]["names"]
    elements = [names[(7 * i) % len(names)] for i in range(70)]
    results = []
    for group in (64, 5):
        torch.set_rng_state(_initial_rng(case))
        ex = _explainer(case, False, True, dict(group_size=group))
        results.append((ex.run_batch(elements), ex._last_batch, torch.get_rng_state()))
    (a, la, ra), (b, lb, rb) = results
    assert torch.equal(ra, rb)
    assert {s["queries_per_engine_call"] for s in ex.last_stats} == {5}
    for i in range(len(elements)):
        _assert_same_explanation(b[i], a[i], lb[i], la[i], "group 5 vs 64 [%d]" % i)


@pytest.mark.gpu
@pytest.mark.parametrize("name,problem", [("gcn2_graph", None), ("c4_hetero_sage", None), ("gcn2_5arg", None),
                                          ("c1_homo_gcn", "edge_prediction")])
def test_run_batch_rejects_unsupported_inputs(name, problem):
    from bikg_graph_explainability_public_b200 import Explainer

    case = gio.load_case(name)
    meta = case["meta"]
    feat, ei, names, pathways, pnames = _inputs(case, False)
    nt, et = case.get("node_types"), case.get("edge_types")
    ex = Explainer(feat, ei, gio.build_arch(case), dict(meta["params"]), names, pathways, pnames, meta["element_type"],
                   problem or meta["problem"], nt, et)
    with pytest.raises(NotImplementedError):
        ex.run_batch([meta["element"]])
