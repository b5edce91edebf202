"""Graph data operations behind the reference's ``Data`` interface (``data.py:19-878``).

Only what sits on the perturbation path is provided.  ``comp_graph`` runs the frontier-BFS k-hop
kernel; the hetero <-> homo flattening is tensor plumbing (cat / pad on the device tensors, as in
the reference).  The reference's ``perturbator`` / ``build_edge_mask`` / ``perturb_node`` /
``concat_features`` materialise a block-diagonal batch: the engine never does that, so those
entry points raise ``NotImplementedError`` pointing at ``engine.MaskedForward``.
"""
import itertools
import operator

import numpy as np
import pandas as pd
import torch

from . import _lib
from .engine import require_cuda
from .pathways import all_str


def khop_subgraph(edge_index, n_nodes, query, hops):
    """Device k-hop (``xpgnn_khop_subgraph``).  Returns subset (int64), sub_edge_index (2,E_sub) int64,
    rank of the query, edge_mask (bool, E), hop levels (int8, N; -1 outside), relabel (int32, N)."""
    lib = _lib.load()
    dev = require_cuda()
    ei = edge_index.to(dev, torch.int64).contiguous()
    e = int(ei.shape[1])
    subset = torch.empty(n_nodes, dtype=torch.int64, device=dev)
    relabel = torch.empty(n_nodes, dtype=torch.int32, device=dev)
    hop = torch.empty(n_nodes, dtype=torch.int8, device=dev)
    edge_mask = torch.zeros(max(e, 1), dtype=torch.uint8, device=dev)
    sub_ei = torch.empty((2, max(e, 1)), dtype=torch.int64, device=dev)
    counts = torch.zeros(3, dtype=torch.int64, device=dev)
    _lib.check(lib.xpgnn_khop_subgraph(ei.data_ptr(), e, int(n_nodes), int(query), int(hops), subset.data_ptr(),
                                       relabel.data_ptr(), hop.data_ptr(), edge_mask.data_ptr(), sub_ei.data_ptr(),
                                       counts.data_ptr(), _lib.stream_ptr()))
    n_sub, e_sub, n_bad = (int(v) for v in counts.tolist())
    if n_bad:
        raise IndexError("edge_index holds %d edge(s) with an endpoint outside [0, %d)" % (n_bad, n_nodes))
    subset = subset[:n_sub]
    sub_ei = sub_ei[:, :e_sub].contiguous()
    sub_ind = relabel[int(query)].to(torch.int64).reshape(1)
    return subset, sub_ei, sub_ind, edge_mask[:e].bool(), hop, relabel


MAX_QUERIES_PER_KHOP = 64  # one bit per query in the device reach words


class MultiKhop:
    """Block-diagonal union of the k-hop graphs of several queries (``xpgnn_khop_multi_*``).  Block q holds query q's
    ``subset`` (ascending node ids) in ``subset[node_off[q]:node_off[q+1]]`` with its BFS ``level``s, and its induced
    edges, in input order and relabelled to union positions, in ``edge_index[:, edge_off[q]:edge_off[q+1]]``.
    ``sub_ind[q]`` is the query's rank inside its block; ``edge_id`` the input column of each union edge (-1 for the
    self loop of a query without an induced edge)."""

    def __init__(self, subset, level, sub_ind, edge_index, edge_id, node_off, edge_off):
        self.subset, self.level, self.sub_ind, self.edge_index, self.edge_id = subset, level, sub_ind, edge_index, edge_id
        self.node_off, self.edge_off = node_off, edge_off

    def __len__(self):
        return len(self.node_off) - 1

    def block(self, q):
        """Query q alone: (subset, local sub_edge_index, sub_ind, level, edge_id) -- what ``khop_subgraph`` gives."""
        n0, n1, e0, e1 = self.node_off[q], self.node_off[q + 1], self.edge_off[q], self.edge_off[q + 1]
        return (self.subset[n0:n1], self.edge_index[:, e0:e1] - n0, int(self.sub_ind[q]), self.level[n0:n1],
                self.edge_id[e0:e1])


def khop_subgraph_multi(edge_index, n_nodes, queries, hops):
    """Device k-hop of up to 64 queries at once (one reach word per node and level, one pass over the edges per hop for
    all of them).  Every block of the returned ``MultiKhop`` is bit-identical to ``khop_subgraph`` for that query."""
    lib = _lib.load()
    dev = require_cuda()
    queries = [int(q) for q in queries]
    nq = len(queries)
    if not 1 <= nq <= MAX_QUERIES_PER_KHOP:
        raise ValueError("khop_subgraph_multi takes 1..%d queries, got %d" % (MAX_QUERIES_PER_KHOP, nq))
    if min(queries) < 0 or max(queries) >= n_nodes:
        raise IndexError("query outside [0, %d)" % n_nodes)
    ei = edge_index.to(dev, torch.int64).contiguous()
    e = int(ei.shape[1])
    qt = torch.tensor(queries, dtype=torch.int64, device=dev)
    ws_bytes = int(lib.xpgnn_khop_multi_workspace_bytes(int(n_nodes), int(hops)))
    if ws_bytes < 0:
        raise ValueError("bad n_nodes / hops")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    counts = torch.empty(2 * nq + 1, dtype=torch.int64, device=dev)
    st = _lib.stream_ptr()
    _lib.check(lib.xpgnn_khop_multi_count(ei.data_ptr(), e, int(n_nodes), qt.data_ptr(), nq, int(hops), ws.data_ptr(),
                                          ws_bytes, counts.data_ptr(), st))
    c = counts.tolist()
    if c[2 * nq]:
        raise IndexError("edge_index holds %d edge(s) with an endpoint outside [0, %d)" % (c[2 * nq], n_nodes))
    node_off = np.concatenate([[0], np.cumsum(c[:nq])]).astype(np.int64)
    edge_off = np.concatenate([[0], np.cumsum(np.maximum(c[nq:2 * nq], 1))]).astype(np.int64)
    n_u, e_u = int(node_off[-1]), int(edge_off[-1])
    offs = torch.from_numpy(np.concatenate([node_off, edge_off])).to(dev)
    subset = torch.empty(n_u, dtype=torch.int64, device=dev)
    level = torch.empty(n_u, dtype=torch.int8, device=dev)
    sub_ind = torch.empty(nq, dtype=torch.int64, device=dev)
    sub_ei = torch.empty((2, e_u), dtype=torch.int64, device=dev)
    edge_id = torch.empty(e_u, dtype=torch.int64, device=dev)
    _lib.check(lib.xpgnn_khop_multi_emit(ei.data_ptr(), e, int(n_nodes), qt.data_ptr(), nq, int(hops), ws.data_ptr(), ws_bytes,
                                         counts.data_ptr(), offs.data_ptr(), offs.data_ptr() + 8 * (nq + 1), e_u,
                                         subset.data_ptr(), level.data_ptr(), sub_ind.data_ptr(), sub_ei.data_ptr(),
                                         edge_id.data_ptr(), st))
    return MultiKhop(subset, level, sub_ind.cpu().tolist(), sub_ei, edge_id, node_off.tolist(), edge_off.tolist())


class Data:
    def __init__(self, feat, edge_index):
        self.feat = feat
        self.edge_index = edge_index

    # ------------------------------------------------------------------ hetero -> homo (data.py:39-147, 695-878)
    def preprocess_hetero_graph(self):
        if isinstance(self.edge_index, dict) and isinstance(self.feat, dict):
            ntypes, etypes = list(self.feat.keys()), list(self.edge_index.keys())
            feat_homo, ei_homo, node_types, edge_types, nptr, eptr, pads = self.hetero2homo()
            return ntypes, etypes, feat_homo, ei_homo, node_types, edge_types, nptr, eptr, pads
        return None, None, self.feat, self.edge_index, None, None, None, None, None

    def hetero2homo(self):
        feat_homo, node_types, pads, nptr = self.concatenate_hetero_features()
        ei_homo, edge_types, eptr = self.concatenate_hetero_edge_indices(nptr)
        return feat_homo, ei_homo, node_types, edge_types, nptr, eptr, pads

    def concatenate_hetero_features(self):
        tensors = list(self.feat.values())
        padded, pads, ptrs = pad_feat_tensors(tensors)
        dev = tensors[0].device
        node_types = torch.hstack([torch.zeros(p.shape[0], device=dev) + i for i, p in enumerate(padded)])
        return torch.vstack(padded), node_types, pads, ptrs

    def concatenate_hetero_edge_indices(self, node_pointers):
        names = list(self.feat.keys())
        mapped, types, ptrs, ptr = [], [], [], 0
        for i, (rel, ei) in enumerate(self.edge_index.items()):
            ptrs.append(ptr)
            add = torch.tensor([[node_pointers[names.index(rel[0])]], [node_pointers[names.index(rel[-1])]]],
                               device=ei.device)
            mapped.append(ei + add)
            types.append(torch.zeros(ei.shape[-1], device=ei.device) + i)
            ptr += ei.shape[-1]
        return torch.hstack(mapped), torch.hstack(types), ptrs

    @staticmethod
    def hetero2homo_names(names):
        if isinstance(names, dict):
            lists = list(names.values())
            homo = list(itertools.chain.from_iterable(lists))
            types = torch.cat([torch.zeros(len(l)) + i for i, l in enumerate(lists)])
            return homo, types
        return names, None

    # ------------------------------------------------------------------ k-hop (data.py:281-361)
    def comp_graph(self, ind, n_hops, problem, names, node_types=None, edge_types=None):
        n_hops += 1  # data.py:328: one more hop than the model covers
        n = int(self.feat.shape[0])
        subset, sub_ei, sub_ind, edge_mask, hop, _ = khop_subgraph(self.edge_index, n, ind, n_hops)
        self.last_hop = hop[subset]
        sub_feat = self.feat.to(subset.device)[subset]
        sub_nt = node_types.to(subset.device)[subset] if node_types is not None else None
        sub_et = edge_types.to(subset.device)[edge_mask] if edge_types is not None else None
        if ("node" in problem) or ("graph" in problem):
            idx = subset.cpu().tolist()
            if all_str(names):
                sub_names = list(operator.itemgetter(*idx)(names)) if len(idx) > 1 else [names[i] for i in idx]
                # == np.array(names, dtype=str)[subset].tolist(), without the N-string array
            else:
                sub_names = np.array(names, dtype=str)[idx].tolist()
        else:
            raise NotImplementedError("edge problems: the reference raises here as well (ind_filter is undefined for "
                                      "homogeneous graphs, data.py:359)")
        return sub_feat, sub_ei, sub_names, sub_ind, sub_nt, sub_et

    def element_size(self, problem):
        return self.edge_index.shape[1] if "edge" in problem else self.feat.shape[0]

    # ------------------------------------------------------------------ materialising entry points
    def perturbator(self, *a, **k):
        raise NotImplementedError("the block-diagonal batch of data.py:591-648 is never materialised; "
                                  "use engine.MaskedForward on the packed coalition bits")

    build_edge_mask = perturb_node = perturb_edge = concat_features = perturbator

    @staticmethod
    def config_val_dataframe(config_val_mean, config_val_std, names):
        df = pd.DataFrame({"name": names,
                           "config_value_mean": config_val_mean.cpu().detach().numpy(),
                           "config_value_std": config_val_std.cpu().detach().numpy()}).set_index("name")
        return df.sort_values(by=["config_value_mean"], ascending=False)


def pad_feat_tensors(feat_tensors):
    """data.py:825-878: zero-pad every node type to the widest feature dimension."""
    fmax = max(t.shape[1] for t in feat_tensors)
    padded, pads, ptrs, ptr = [], [], [], 0
    for t in feat_tensors:
        d = fmax - t.shape[1]
        pads.append(d)
        ptrs.append(ptr)
        ptr += t.shape[0]
        padded.append(torch.nn.functional.pad(t, (0, d)) if d > 0 else t)
    return padded, pads, ptrs
