"""``Explainer(...).run(query_node, repeats)`` -- the drop-in boundary.

Same constructor, assertions, side effects and return values as the reference's
``pathway_explanations.explainer.Explainer`` (``explainer.py:25-546``), with the perturbation hot
path (k-hop cut, coalition masks, perturbed forward, SHAP weights, surrogate fit, community
scores) running in CUDA kernels through ``libxpgnn_b200.so``.  There is no CPU fallback: without
a CUDA device or without the built library, ``run`` raises.
"""
import operator
import random

import numpy as np
import torch

from . import _lib
from .data import MAX_QUERIES_PER_KHOP, Data, khop_subgraph_multi
from .engine import GraphSpec, MaskedForward, require_cuda
from .kernels import shap_weights
from .lowering import lower
from .masks import Mask
from .model import Model
from .pathways import CommunityIndex, Pathways, _first_index, all_str
from .shard import sharded_eval
from .wlm import LinearRegression, fit_surrogate, optimizer_assertions


def set_seed(seed=100):
    """explainer.py:14-22 (the CPU generator seeded with ``seed + 2`` is the stream that matters)."""
    random.seed(seed)
    np.random.seed(seed + 1)
    torch.manual_seed(seed + 2)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(seed + 3)
        torch.cuda.manual_seed_all(seed + 4)
    torch.backends.cudnn.enabled = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False


def build_engine(feat, edge_index, arch, element_index, node_type=None, edge_type=None, node_type_names=None,
                 edge_type_names=None, padded_dims=None, out_type=None, hop=None, prune=False, precision="fp32",
                 query_flat=None, model=None, queries=None):
    """Lower ``arch`` and bind it to the (flattened) computational graph.

    ``element_index`` follows the reference: the row of the model output that is read
    (``model.py:247,325``), i.e. an index *inside the output node type* for hetero graphs.
    ``model``: an already lowered plan (``lowering.lower_candidates``); ``queries``: flat node ids to read instead of
    the single element (probe check)."""
    dev = require_cuda()
    if model is None:
        model = lower(arch)
    n = int(feat.shape[0])
    if node_type_names is None:
        if model.hetero:
            raise NotImplementedError("a HeteroConv model needs dict inputs (node / edge types)")
        graph = GraphSpec(feat, edge_index, [0, n])
        n_types = 1
        q = int(element_index) if query_flat is None else int(query_flat)
    else:
        nt = node_type.to(torch.int64).cpu()
        if nt.numel() > 1 and bool((nt[1:] < nt[:-1]).any()):
            raise ValueError("node types must be contiguous blocks (flattened hetero graph)")
        counts = torch.bincount(nt, minlength=len(node_type_names)).tolist()
        type_ptr = [0]
        for c in counts:
            type_ptr.append(type_ptr[-1] + int(c))
        graph = GraphSpec(feat, edge_index, type_ptr, list(node_type_names), edge_type.to(torch.int64),
                          [tuple(e) for e in edge_type_names])
        n_types = int((torch.tensor(counts) > 0).sum())
        if query_flat is not None:
            q = int(query_flat)
        else:
            t = out_type if out_type is not None else getattr(arch, "out_type", None) or node_type_names[0]
            q = type_ptr[node_type_names.index(t)] + int(element_index)
    if model.out_dim != 1:
        raise NotImplementedError("the surrogate needs a scalar prediction per node (model output width 1)")
    multi = n_types >= 2
    eng = MaskedForward(graph, model, [q] if queries is None else list(queries), prune=prune and hop is not None, hop=hop,
                        zero_edge_rule=multi and queries is None, precision=precision)
    # (B,1) targets broadcast against (B,) predictions in the reference loss (wlm.py:517); the
    # multi-node-type branch yields (B,) targets (model.py:251) and the plain weighted MSE
    eng.broadcast_y = not multi
    return eng


def _forward_arity(arch):
    import inspect

    return len(inspect.getfullargspec(arch.forward).args)  # model.py:104: 3 = (self, x, edge_index), 5 = + node / edge types


def verify_lowering(arch, feat_dims, node_type_names=None, edge_type_names=None, out_type=None, seed=12345):
    """Pick the lowered plan that IS ``arch``: the reference calls ``arch(feat, edge_index)`` as a black box
    (``model.py:104-112``), the engine runs a lowered plan, so every candidate plan (``lowering.lower_candidates``) is
    evaluated by the engine on a small random probe graph with no node removed and compared with ``arch`` itself on the
    same graph, all output rows.  Returns ``(plan, status)``, status = "verified" or "unverified: ..." when ``arch``
    cannot be called (weight containers of ``nn.py``: their plan is their definition).  Raises ``NotImplementedError``
    when no candidate reproduces ``arch`` -- a model with skip connections, functional ops the lowering does not know, or
    layers applied in an order the plan does not reflect must not be explained with a different function."""
    from .lowering import lower_candidates

    cands = lower_candidates(arch)
    g = torch.Generator().manual_seed(seed)
    par = next(arch.parameters(), None)
    adev = par.device if par is not None else torch.device("cpu")
    hetero = node_type_names is not None
    if not hetero:
        n, e = 48, 220
        x = torch.randn(n, int(feat_dims), generator=g)
        ei = torch.randint(0, n, (2, e), generator=g)
        ei = torch.cat([ei, ei[:, :7], torch.arange(5).repeat(2, 1)], 1)  # duplicate edges and self loops
        args = (x.to(adev), ei.to(adev))
        if _forward_arity(arch) == 5:
            args = args + (torch.zeros(n, device=adev), torch.zeros(ei.shape[1], device=adev))
    else:
        counts = [20 + 3 * i for i in range(len(node_type_names))]
        x_dict = {t: torch.randn(c, int(feat_dims[t]), generator=g) for t, c in zip(node_type_names, counts)}
        ei_dict = {}
        for r in edge_type_names:
            r = tuple(r)
            ns, nd = counts[node_type_names.index(r[0])], counts[node_type_names.index(r[-1])]
            ei_dict[r] = torch.stack([torch.randint(0, ns, (60,), generator=g), torch.randint(0, nd, (60,), generator=g)])
        args = ({t: v.to(adev) for t, v in x_dict.items()}, {r: v.to(adev) for r, v in ei_dict.items()})
    was_training = arch.training
    arch.eval()
    try:
        with torch.no_grad():
            ref = arch(*args)
    except NotImplementedError as ex:
        # nn.py layers hold weights only, and a Module without a forward (torch: 'missing the required "forward" function')
        # cannot be called either: there is no black box to compare with, the plan is the model's definition
        if "weight container" in str(ex) or 'missing the required "forward"' in str(ex):
            return cands[-1], "unverified: arch cannot be called (weight containers / no forward), its plan is its definition"
        raise
    finally:
        arch.train(was_training)
    # rows of the reference output <-> flat probe node ids
    if hetero:
        raw = Data(x_dict, ei_dict)
        ntn, etn, feat, ei, node_types, edge_types, nptr, _eptr, pads = raw.preprocess_hetero_graph()
        if isinstance(ref, dict):  # model.py:255-292: outputs of the node types, stacked in dict order
            rows, flat = [], []
            for t, v in ref.items():
                rows.append(v)
                lo = nptr[ntn.index(t)]
                flat += list(range(lo, lo + v.shape[0]))
            ref = torch.vstack(rows)
        else:
            t = out_type if out_type is not None else getattr(arch, "out_type", None) or ntn[0]
            lo = nptr[ntn.index(t)]
            flat = list(range(lo, lo + ref.shape[0]))
    else:
        ntn = etn = node_types = edge_types = pads = None
        feat, ei = x, ei
        flat = list(range(ref.shape[0]))
    ref = ref.detach().float().cpu().reshape(len(flat), -1)[:, 0].numpy()
    dev = require_cuda()
    act = torch.ones((int(feat.shape[0]), 1), dtype=torch.int32, device=dev)
    worst = []
    for cand in cands:
        try:
            eng = build_engine(feat.to(dev), ei.to(dev), arch, 0, node_types, edge_types, ntn, etn, pads, out_type=out_type,
                               model=cand, queries=flat)
        except NotImplementedError as ex:
            worst.append("%s: %s" % (cand.how, ex))
            continue
        y = eng(act, 1)[0].cpu().numpy()
        err = float(np.max(np.abs(y - ref) / np.maximum(np.abs(ref), 1e-3)))
        if err <= 2e-4:
            return cand, "verified"
        worst.append("%s: max rel. deviation %.3g on the probe graph" % (cand.how, err))
    raise NotImplementedError(
        "arch.forward is not the layer sequence the engine can lower (%s); supported: chains of GCNConv / SAGEConv(mean) / "
        "HeteroConv(sum) with ReLU / Sigmoid, then Linear layers" % "; ".join(worst))


_TOO_LARGE = (torch.OutOfMemoryError, torch.AcceleratorError, _lib.XpgnnError)


class _GroupTooLarge(Exception):
    """The union of a group of queries does not fit the device; the group is split."""


def _does_not_fit(ex):
    """A device allocation failed or the engine's workspace does not fit: a smaller group of queries may."""
    return isinstance(ex, torch.OutOfMemoryError) or "does not fit" in str(ex) or "out of memory" in str(ex)


def sync_rng_across_ranks():
    """One process per GPU: every rank replays the coalition stream of the CPU generator, so the generators must agree.
    ``set_seed`` guarantees that only for ``times == 1`` (explainer.py:342); rank 0's state is made authoritative."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    box = [torch.get_rng_state()]
    dist.broadcast_object_list(box, src=0)
    torch.set_rng_state(box[0])


def check_ranks_agree(act):
    """Ranks evaluate slices of ONE coalition matrix; raise if theirs differ (mismatched masks would pair predictions
    with the wrong rows and the replicated fit would silently train on wrong targets)."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    a = act.view(-1)
    n = int(a.numel())
    wcol = (torch.arange(int(act.shape[1]), device=act.device, dtype=torch.int64) % 8191) + 1
    h = torch.stack([torch.sum(a, dtype=torch.int64), torch.sum(torch.sum(act, dim=0, dtype=torch.int64) * wcol),
                     torch.sum(act[:: max(n // (1 << 20) // max(int(act.shape[1]), 1), 1)].to(torch.int64) * 31 % 1000003),
                     torch.tensor(n, device=act.device, dtype=torch.int64)])
    lo, hi = h.clone(), h.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    if not torch.equal(lo, hi):
        raise RuntimeError("ranks generated different coalition masks (per-rank seeding?): Explainer.run needs the same "
                           "global CPU generator state on every rank")


class Explainer:
    #: engine knobs (extension).  precision "fp32": fp32 storage and accumulation, dense transforms as 3xTF32 tensor-core
    #: products (error ~1e-6 relative, inside the 1e-4 bar); "fp32_exact": exact fp32 FMA transforms (slower, for audits);
    #: "bf16" / "bf16_act": the 2e-2 bar.  verify: compare the
    #: lowered plan with ``arch`` itself on a probe graph before explaining (see ``verify_lowering``).
    #: group_size (``run_batch``): queries per k-hop call and per engine, at most 64.
    engine_options = dict(prune=True, precision="fp32", verify=True, group_size=MAX_QUERIES_PER_KHOP)

    def __init__(self, feat, edge_index, arch, params, names, pathways=None, pathway_names=None, element_type=None,
                 problem="node_prediction", node_types=None, edge_types=None):
        self.initial_assertions(feat, edge_index, arch, params, names, pathways, pathway_names, element_type, problem)
        problem = problem.lower().strip()
        self.feat, self.edge_index, self.arch, self.params, self.names = feat, edge_index, arch, params, names
        self.pathways, self.pathway_names, self.element_type = pathways, pathway_names, element_type
        self.problem, self.node_types, self.edge_types = problem, node_types, edge_types
        self.last_stats = {}

    @staticmethod
    def initial_assertions(feat, edge_index, arch, params, names, pathways, pathway_names, element_type, problem):
        """explainer.py:106-189, same messages."""
        if pathways is not None:
            assert isinstance(pathways, list) or isinstance(pathways, dict), "Pathways is not list or dict"
        if pathway_names is not None:
            assert isinstance(pathway_names, list) or isinstance(
                pathway_names, dict
            ), "Pathway names is not list or dict"
            assert len(pathway_names) == len(
                pathways
            ), "Length of list with pathway names and list with pathway indexes do not match"
        assert isinstance(feat, torch.Tensor) or isinstance(feat, dict), "Feature matrix is not torch tensor or dict"
        assert isinstance(edge_index, torch.Tensor) or isinstance(
            edge_index, dict
        ), "Edge index matrix is not torch tensor or dict"
        assert isinstance(names, list) or isinstance(names, dict), "Element names is not list or dict"
        assert isinstance(params, dict), "Hyperparameters given is not dictionary"
        assert isinstance(problem, str), "Problem type given is not string"
        if element_type is not None:
            assert isinstance(element_type, str) or isinstance(
                element_type, tuple
            ), "Element type is not string (node) nor tuple (edge)"
            if "node" in problem:
                assert isinstance(feat, dict), "Feature given is not a dict of node types"
                assert (
                    element_type in list(feat.keys())
                ), "Node type '{}' is not among input node types in heterogeneous graph".format(element_type)
            elif "edge" in problem:
                assert isinstance(edge_index, dict), "Edge index given is not a dict of edge index types"
                assert (
                    element_type in list(edge_index.keys())
                ), "Edge type '{}' is not among input node types in heterogeneous graph".format(element_type)

    @staticmethod
    def extract_index(element, names=None):
        """explainer.py:191-226."""
        if names is None:
            assert isinstance(element, int) or isinstance(
                element, float
            ), "No element names have been given and the node name given is not numeric"
            return int(element)
        assert element in names, "Element name '{}' is not present in the graph".format(element)
        if type(element) is str and all_str(names):
            return names.index(element)  # first match, as np.where(...)[0][0]
        return int(np.where(np.array(names, dtype=str) == element)[0][0])

    def filter_hetero_names(self, names, node_type, edge_type, node_type_names, edge_type_names):
        """explainer.py:228-286."""
        names_array = np.array(names, dtype=str)
        if isinstance(self.element_type, str):
            sel = torch.where(node_type == node_type_names.index(self.element_type))[0]
        elif isinstance(self.element_type, tuple):
            sel = torch.where(edge_type == edge_type_names.index(self.element_type))[0]
        else:
            sel = torch.where(node_type == 1)[0]
        return names_array[sel.cpu().numpy()].tolist()

    @staticmethod
    def weight_stacking(weights):
        """explainer.py:288-314: mean and population std over repeats (device kernel)."""
        lib = _lib.load()
        stack = torch.vstack([w.reshape(1, -1) for w in weights]).to(require_cuda(), torch.float32).contiguous()
        t, n = stack.shape
        mean, std = torch.empty(n, device=stack.device), torch.empty(n, device=stack.device)
        _lib.check(lib.xpgnn_repeat_stats(stack.data_ptr(), t, n, mean.data_ptr(), std.data_ptr(), _lib.stream_ptr()))
        return mean, std

    def run(self, element, times=1):
        """explainer.py:316-546.  Returns (config_val_df, pathway_df)."""
        import gc

        # The host side handles lists of up to millions of names; every generation-2 collection of the cyclic GC walks all of
        # them (measured: up to 0.4 s per explained query at 1 M names).  Nothing here creates reference cycles.
        gc_was_enabled = gc.isenabled()
        gc.disable()
        try:
            return self._run(element, times)
        finally:
            if gc_was_enabled:
                gc.enable()

    def _run(self, element, times):
        dev = require_cuda()
        _lib.load()
        if "edge" in self.problem:
            # the reference itself cannot run them: comp_graph raises UnboundLocalError on homogeneous graphs (data.py:359,
            # ``ind_filter``), Mask reads an attribute that is never set (masks.py:294, ``self.edge_size``)
            raise NotImplementedError("edge problems: the reference path is not runnable (data.py:359, masks.py:294); not built")
        graph_problem = "graph" in self.problem
        if times == 1:
            set_seed(self.params["seed"])
        nvtx = torch.cuda.nvtx
        nvtx.range_push("xpgnn:run:flatten")
        raw = Data(self.feat, self.edge_index)
        if self.pathways is not None:
            raw_pathways = Pathways(self.pathways, self.pathway_names)
        (ntn, etn, self.feat, self.edge_index, node_types, edge_types, nptr, eptr, pads) = raw.preprocess_hetero_graph()
        typed_homo = False
        if node_types is None and self.node_types is not None:  # explainer.py:365-371: caller-provided type vectors of a
            node_types = self.node_types.clone()                 # homogenised graph (5-argument forward, model.py:110-112)
            typed_homo = True
        if edge_types is None and self.edge_types is not None:
            edge_types = self.edge_types.clone()
            typed_homo = True
        self.names, _ = raw.hetero2homo_names(self.names)
        if self.pathways is not None:
            self.pathways, self.pathway_names, ptypes = raw_pathways.hetero2homo(self.problem, nptr, eptr)
            pathway_class = Pathways(self.pathways, self.pathway_names, ptypes)

        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:khop")
        self.feat = self.feat.to(dev)
        self.edge_index = self.edge_index.to(dev)
        data_class = Data(self.feat, self.edge_index)
        relations = len(etn) if etn is not None else 0
        n_hops = Model(self.arch).get_hops(relations)
        ind = self.extract_index(element, self.names)
        if graph_problem:
            # explainer.py:427-447: no computational-graph cut -- the whole graph, every community as given, the prediction
            # read at the element's own row (wlm.py:435-436); every conv layer runs over the whole graph ("full" mode)
            sub_feat, sub_ei, sub_names = self.feat, self.edge_index.to(torch.int64), self.names
            sub_ind = torch.tensor([ind])
            sub_nt = None if node_types is None else node_types.to(dev)
            sub_et = None if edge_types is None else edge_types.to(dev)
            hop = None
        else:
            sub_feat, sub_ei, sub_names, sub_ind, sub_nt, sub_et = data_class.comp_graph(
                ind, n_hops, self.problem, self.names, node_types, edge_types)
            hop = data_class.last_hop
        query_flat = hop_query = int(sub_ind[0])  # hop levels are distances to this node

        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:communities")
        sub_pathway_inds = sub_pathway_names = None
        if self.pathways is not None and graph_problem:  # explainer.py:447-449, 464-470: communities kept as given
            sub_pathway_names = self.pathway_names
            first = self.pathways[0][0]
            sub_pathway_inds = Pathways(self.pathways, sub_pathway_names).names2inds(sub_names) if isinstance(first, str) else self.pathways
            sub_pathway_class = Pathways(sub_pathway_inds, sub_pathway_names)
        elif self.pathways is not None:
            # pathways.py:33-136 (comp_graph + names2inds) in one vectorised pass; see Pathways.resolve_indices
            sub_pathway_inds, sub_pathway_names = pathway_class.resolve_indices(sub_names)
            if not sub_pathway_inds:
                raise IndexError("list index out of range")  # explainer.py:467: no community reaches the computational graph
            sub_pathway_class = Pathways(sub_pathway_inds, sub_pathway_names)
        if not graph_problem and (self.element_type is not None or self.node_types is not None or self.edge_types is not None):
            filtered = self.filter_hetero_names(sub_names, sub_nt, sub_et, ntn, etn)
            sub_ind = torch.tensor([self.extract_index(element, filtered)])
        del self.feat, self.edge_index  # explainer.py:476: the object is single use

        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:engine_build")
        elements = int(sub_feat.shape[0])
        opts = dict(type(self).engine_options)
        opts.update(getattr(self, "options", {}))
        out_type = self.element_type if isinstance(self.element_type, str) else None
        self.arch.eval()
        plan = None
        self.lowering_status = "not checked"
        if opts.get("verify", True):  # the plan must be the function the reference would call (model.py:104-112)
            fd = int(sub_feat.shape[1]) if ntn is None else {t: int(sub_feat.shape[1]) - int(pads[i]) for i, t in enumerate(ntn)}
            plan, self.lowering_status = verify_lowering(self.arch, fd, ntn, etn, out_type)
        if typed_homo:
            # The reference hands the type vectors to arch.forward and then reads row ``sub_ind`` -- the query's index among
            # the type-1 nodes (explainer.py:280-284) -- of the full output (wlm.py:435-436).  The engine lowers models whose
            # plan reproduces arch on the probe graph (i.e. that do not branch on the types) and reads the same row.
            sub_nt = sub_et = None
            query_flat = int(sub_ind[0])
        engine = build_engine(sub_feat, sub_ei, self.arch, int(sub_ind[0]), sub_nt, sub_et, ntn, etn, pads,
                              out_type=out_type, hop=hop if not typed_homo or query_flat == int(hop_query) else None,
                              prune=opts["prune"], precision=opts["precision"], query_flat=query_flat, model=plan)
        # ---- all repeats' coalitions first: the masks, the surrogate init and the DataLoader seed draw of repeat r + 1
        # depend on the RNG stream only (masks -> randperm -> N init draws -> 2 draws, explainer.py:490-523 / wlm.py:210),
        # never on the predictions, so every repeat's rows go through ONE sharded engine call ----
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:masks")
        sync_rng_across_ranks()
        sets = []
        for _ in range(times):
            coalitions, _rows = Mask(sub_feat, sub_ei, sub_pathway_inds, self.params, self.problem).mask_generator()
            wlrm = LinearRegression(elements)           # kaiming-uniform init: next N draws of the CPU stream
            torch.empty((), dtype=torch.int64).random_()  # iter(DataLoader) base seed (wlm.py:210)
            sets.append((coalitions, wlrm.layer.weight.detach().reshape(-1)))
        if times == 1:
            act_all, n_all = sets[0][0].act, sets[0][0].n_coalitions
        else:  # repeats side by side along the word axis; a repeat's last word is padded with all-off rows
            act_all = torch.cat([c.act for c, _ in sets], dim=1).contiguous()
            n_all = 32 * int(act_all.shape[1])
        check_ranks_agree(act_all)
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:masked_forward")
        y_all = sharded_eval(engine, act_all, n_all)[:, 0]
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:fit")
        config_vals, word0 = [], 0
        for coalitions, w0 in sets:
            y = y_all[32 * word0: 32 * word0 + coalitions.n_coalitions]
            word0 += coalitions.words
            kern = shap_weights(coalitions.popcount, elements, coalitions.batch_size)
            w, losses = fit_surrogate(coalitions, y, kern, w0, self.params, broadcast_y=engine.broadcast_y, want_losses=False)
            config_vals.append(w)
            self.last_stats = dict(n_sub=elements, e_sub=int(sub_ei.shape[1]), coalitions=coalitions.n_coalitions,
                                   batch_size=coalitions.batch_size, tile_coalitions=engine.tile_coalitions,
                                   repeats_per_engine_call=times, lowering=self.lowering_status)
            if opts.get("keep_last", False):  # tests / debugging only: pins the coalition draws and predictions in HBM
                self._last = dict(coalitions=coalitions, y=y, kernel=kern, w0=w0, subset_names=sub_names,
                                  sub_edge_index=sub_ei, sub_ind=query_flat)
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run:aggregate")
        mean, std = self.weight_stacking(config_vals)
        config_val_df = Data.config_val_dataframe(mean, std, sub_names)
        pathway_df = None
        if self.pathways is not None:
            pathway_df = sub_pathway_class.aggregate(mean, sub_pathway_inds)
        nvtx.range_pop()
        return config_val_df, pathway_df

    # ------------------------------------------------------------------ many queries
    def run_batch(self, elements, times=1):
        """Explain several query nodes: returns ``[Explainer(<same constructor args>).run(e, times) for e in elements]``,
        run from the same global CPU generator state, which it also leaves as that loop does.

        The query-independent work runs once: flattening, the plan check (``verify_lowering``), the name -> index map and
        the community members' ids.  The queries' computational graphs are cut together (``khop_subgraph_multi``), laid
        side by side as one block-diagonal graph and evaluated by ONE engine call over all their coalitions; their
        surrogates are fitted together (``xpgnn_wlm_fit_batch``).  Queries go in groups of at most ``group_size`` (64),
        in input order; a group whose engine does not fit the device is split.

        Node problems on homogeneous graphs and on dict graphs with one node type.  Raises ``NotImplementedError`` for
        graph and edge problems, graphs with two or more node types and caller-provided node / edge type vectors.
        With ``options["keep_last"]`` the intermediates ``run`` keeps in ``_last`` go to the list ``_last_batch``;
        ``last_stats`` is a list with one dict per query."""
        import gc

        gc_was_enabled = gc.isenabled()
        gc.disable()
        try:
            return self._run_batch(list(elements), times)
        finally:
            if gc_was_enabled:
                gc.enable()

    def _run_batch(self, elements, times):
        dev = require_cuda()
        _lib.load()
        if "edge" in self.problem:
            raise NotImplementedError("edge problems: the reference path is not runnable (data.py:359, masks.py:294); not built")
        if "graph" in self.problem:
            raise NotImplementedError("run_batch explains node problems; a graph problem reads the whole graph for every "
                                      "element, there is no computational graph to batch: use run")
        if self.node_types is not None or self.edge_types is not None:
            raise NotImplementedError("run_batch does not batch caller-provided node / edge type vectors (the 5-argument "
                                      "forward): use run")
        if isinstance(self.feat, dict) and len(self.feat) >= 2:
            raise NotImplementedError("run_batch does not batch graphs with two or more node types: their zero-edge rule "
                                      "(model.py:213-215) applies per coalition of one query's graph, the engine would "
                                      "apply it over the whole union; use run")
        nvtx = torch.cuda.nvtx
        nvtx.range_push("xpgnn:run_batch:flatten")
        raw = Data(self.feat, self.edge_index)
        if self.pathways is not None:
            raw_pathways = Pathways(self.pathways, self.pathway_names)
        (ntn, etn, self.feat, self.edge_index, node_types, edge_types, nptr, eptr, pads) = raw.preprocess_hetero_graph()
        self.names, _ = raw.hetero2homo_names(self.names)
        if self.pathways is not None:
            self.pathways, self.pathway_names, _ptypes = raw_pathways.hetero2homo(self.problem, nptr, eptr)
        first = _first_index(self.names) if all_str(self.names) else None
        inds = []
        for e in elements:
            if first is not None and type(e) is str:
                assert e in first, "Element name '{}' is not present in the graph".format(e)
                inds.append(first[e])
            else:
                inds.append(self.extract_index(e, self.names))
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:communities")
        cindex = None
        if self.pathways is not None:
            cindex = CommunityIndex(self.pathways, self.pathway_names, self.names, first)
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:engine_build")
        opts = dict(type(self).engine_options)
        opts.update(getattr(self, "options", {}))
        group = max(1, min(int(opts.get("group_size", MAX_QUERIES_PER_KHOP)), MAX_QUERIES_PER_KHOP))
        out_type = self.element_type if isinstance(self.element_type, str) else None
        self.arch.eval()
        plan = None
        self.lowering_status = "not checked"
        if opts.get("verify", True):
            fd = int(self.feat.shape[1]) if ntn is None else {t: int(self.feat.shape[1]) - int(pads[i]) for i, t in enumerate(ntn)}
            plan, self.lowering_status = verify_lowering(self.arch, fd, ntn, etn, out_type)
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:khop")
        feat = self.feat.to(dev)
        edge_index = self.edge_index.to(dev)
        n_hops = Model(self.arch).get_hops(len(etn) if etn is not None else 0) + 1  # data.py:328: one more hop
        del self.feat, self.edge_index  # explainer.py:476: the object is single use
        nvtx.range_pop()
        ctx = dict(feat=feat, node_types=None if node_types is None else node_types.to(dev),
                   edge_types=None if edge_types is None else edge_types.to(dev), ntn=ntn, etn=etn, pads=pads,
                   out_type=out_type, plan=plan, opts=opts, times=times, cindex=cindex)
        self.last_stats = []
        if opts.get("keep_last", False):
            self._last_batch = []
        results = []
        for g0 in range(0, len(inds), group):
            results += self._explain_group(edge_index, inds[g0:g0 + group], n_hops, ctx)
        return results

    def _explain_group(self, edge_index, inds, n_hops, ctx):
        """Cut the computational graphs of ``inds`` together and explain them; halves the group when the union does not
        fit the device."""
        nvtx = torch.cuda.nvtx
        nvtx.range_push("xpgnn:run_batch:khop")
        try:
            mk = khop_subgraph_multi(edge_index, int(ctx["feat"].shape[0]), inds, n_hops)
        except _TOO_LARGE as ex:
            if not _does_not_fit(ex) or len(inds) == 1:
                raise
            mk = None
        nvtx.range_pop()
        if mk is not None:
            try:
                return self._explain_union(mk, ctx)
            except _GroupTooLarge:  # raised before any coalition of the group is drawn: halving keeps the draw order
                pass
        mk = None
        torch.cuda.empty_cache()  # the library's stream-ordered scratch does not come from torch's cache
        h = len(inds) // 2
        return self._explain_group(edge_index, inds[:h], n_hops, ctx) + self._explain_group(edge_index, inds[h:], n_hops, ctx)

    def _explain_union(self, mk, ctx):
        """Explain the queries of one block-diagonal union (``MultiKhop``); splits it when its engine does not fit."""
        nvtx = torch.cuda.nvtx
        opts, times, nq = ctx["opts"], ctx["times"], len(mk)
        nvtx.range_push("xpgnn:run_batch:engine_build")
        queries = [mk.node_off[q] + mk.sub_ind[q] for q in range(nq)]
        try:
            sub_feat = ctx["feat"][mk.subset]
            sub_nt = None if ctx["node_types"] is None else ctx["node_types"][mk.subset]
            sub_et = None
            if ctx["edge_types"] is not None:  # a self loop of the per-query rule (edge_id -1) belongs to no relation
                sub_et = torch.where(mk.edge_id >= 0, ctx["edge_types"][mk.edge_id.clamp(min=0)].to(torch.int64), -1)
            engine = build_engine(sub_feat, mk.edge_index, self.arch, 0, sub_nt, sub_et, ctx["ntn"], ctx["etn"], ctx["pads"],
                                  out_type=ctx["out_type"], hop=mk.level, prune=opts["prune"], precision=opts["precision"],
                                  model=ctx["plan"], queries=queries)
        except _TOO_LARGE as ex:
            nvtx.range_pop()
            if not _does_not_fit(ex) or nq == 1:
                raise
            raise _GroupTooLarge() from None
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:communities")
        subset_host = mk.subset.cpu()
        idx_all = subset_host.tolist()
        names = self.names
        str_names = all_str(names)
        per_q = []
        for q in range(nq):
            n0, n1 = mk.node_off[q], mk.node_off[q + 1]
            idx = idx_all[n0:n1]
            if str_names:  # == Data.comp_graph's names[subset]
                sub_names = list(operator.itemgetter(*idx)(names)) if len(idx) > 1 else [names[i] for i in idx]
            else:
                sub_names = np.array(names, dtype=str)[idx].tolist()
            com_inds = com_names = None
            if ctx["cindex"] is not None:
                com_inds, com_names = ctx["cindex"].resolve(subset_host[n0:n1].numpy())
                if not com_inds:
                    raise IndexError("list index out of range")  # explainer.py:467: no community reaches the graph
            per_q.append(dict(n=n1 - n0, sub_names=sub_names, com_inds=com_inds, com_names=com_names))
        nvtx.range_pop()
        # ---- every query's coalitions, in input order, with the draw sequence of run (masks -> surrogate init -> the
        # DataLoader seed draw, per repeat; set_seed per query when times == 1) ----
        nvtx.range_push("xpgnn:run_batch:masks")
        sync_rng_across_ranks()
        for q, pq in enumerate(per_q):
            if times == 1:
                set_seed(self.params["seed"])
            n0, n1 = mk.node_off[q], mk.node_off[q + 1]
            sub_feat_q = sub_feat[n0:n1]
            sets = []
            for _ in range(times):
                coalitions, _rows = Mask(sub_feat_q, None, pq["com_inds"], self.params, self.problem).mask_generator()
                wlrm = LinearRegression(pq["n"])
                torch.empty((), dtype=torch.int64).random_()
                sets.append((coalitions, wlrm.layer.weight.detach().reshape(-1)))
            pq["sets"] = sets
            if times == 1:
                pq["act"], pq["n_all"] = sets[0][0].act, sets[0][0].n_coalitions
            else:
                pq["act"] = torch.cat([c.act for c, _ in sets], dim=1)
                pq["n_all"] = 32 * int(pq["act"].shape[1])
        w_max = max(int(pq["act"].shape[1]) for pq in per_q)
        act = torch.zeros((int(mk.node_off[-1]), w_max), dtype=torch.int32, device=engine.device)
        for q, pq in enumerate(per_q):  # words >= W_q stay zero: every node of the block is off there
            act[mk.node_off[q]:mk.node_off[q + 1], :pq["act"].shape[1]] = pq["act"]
        n_all = max(pq["n_all"] for pq in per_q)
        check_ranks_agree(act)
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:masked_forward")
        y_all = sharded_eval(engine, act, n_all).contiguous()  # (n_all, nq): column q = query q
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:fit")
        lib = _lib.load()
        lr = optimizer_assertions(self.params)
        descs, kerns, w0s, off = [], [], [], 0
        for q, pq in enumerate(per_q):
            word0 = 0
            pq["w_off"], pq["kern"] = [], []
            for coalitions, w0 in pq["sets"]:
                kern = shap_weights(coalitions.popcount, pq["n"], coalitions.batch_size)
                d = _lib.FitQuery()
                d.act_off, d.y_off = mk.node_off[q] * w_max + word0, 32 * word0 * nq + q
                d.kern_off, d.w_off = sum(int(k.numel()) for k in kerns), off
                d.n, d.s, d.batch, d.losses = pq["n"], coalitions.n_coalitions, coalitions.batch_size, None
                descs.append(d)
                kerns.append(kern.to(torch.float64))
                w0s.append(w0.to(engine.device, torch.float32))
                pq["w_off"].append(off)
                pq["kern"].append(kern)
                off += pq["n"]
                word0 += coalitions.words
        kern_all = torch.cat(kerns).contiguous()
        w_all = torch.cat(w0s).contiguous()
        arr = (_lib.FitQuery * len(descs))(*descs)
        _lib.check(lib.xpgnn_wlm_fit_batch(act.data_ptr(), w_max, y_all.data_ptr(), nq, kern_all.data_ptr(), w_all.data_ptr(),
                                           arr, len(descs), float(lr), float(self.params["l1_lambda"]), 1e-2,
                                           int(bool(engine.broadcast_y)), _lib.stream_ptr()))
        nvtx.range_pop()
        nvtx.range_push("xpgnn:run_batch:aggregate")
        out = []
        for q, pq in enumerate(per_q):
            ws = [w_all[o:o + pq["n"]] for o in pq["w_off"]]
            mean, std = self.weight_stacking(ws)
            config_val_df = Data.config_val_dataframe(mean, std, pq["sub_names"])
            pathway_df = None
            if pq["com_inds"] is not None:
                pathway_df = Pathways(pq["com_inds"], pq["com_names"]).aggregate(mean, pq["com_inds"])
            out.append((config_val_df, pathway_df))
            coalitions, w0 = pq["sets"][-1]
            word0 = sum(c.words for c, _ in pq["sets"][:-1])
            self.last_stats.append(dict(n_sub=pq["n"], e_sub=mk.edge_off[q + 1] - mk.edge_off[q],
                                        coalitions=coalitions.n_coalitions, batch_size=coalitions.batch_size,
                                        tile_coalitions=engine.tile_coalitions, repeats_per_engine_call=times,
                                        queries_per_engine_call=nq, lowering=self.lowering_status))
            if opts.get("keep_last", False):
                subset, sub_ei, sub_ind, _lev, _eid = mk.block(q)
                self._last_batch.append(dict(coalitions=coalitions, y=y_all[32 * word0: 32 * word0 + coalitions.n_coalitions, q],
                                             kernel=pq["kern"][-1], w0=w0, subset_names=pq["sub_names"],
                                             sub_edge_index=sub_ei, sub_ind=sub_ind))
        nvtx.range_pop()
        return out
