"""Community bookkeeping behind the reference's ``Pathways`` interface (``pathways.py:8-429``).

Name resolution is host work, as in the reference, but not the reference's algorithm: it calls
``np.intersect1d(community, names)`` once per community, i.e. sorts the whole name array C times
(O(C N log N) string compares -- 60 s of a 70 s query at 1 M nodes / 500 communities).  Here one
name -> first-index hash map is built per call and every community is filtered / deduplicated /
sorted on its own (O(N + sum L log L)); the outputs are identical (``tests/test_capi_and_host.py``
checks them against the ``intersect1d`` formulation) -- SURVEY.md 8f-1.  The community-level random
masks live in ``masks.py`` (device), and ``aggregate`` runs the segmented-mean kernel.
"""
import itertools

import numpy as np
import pandas as pd
import torch

from . import _lib
from .engine import require_cuda


def all_str(values):
    """True iff every element is exactly a ``str`` (one C-level pass; a Python generator costs ~1 us per element)."""
    return set(map(type, values)) <= {str}


def _as_str(values):
    """``np.array(values, dtype=str)`` element-wise: strings pass through, everything else via numpy's conversion."""
    if all_str(values):
        return values
    return np.array(values, dtype=str).tolist()


def _first_index(names):
    """name -> index of its first occurrence (``np.unique(..., return_index=True)`` semantics).
    Filled back to front so that the first occurrence is the assignment that survives; runs inside ``dict(zip(...))``."""
    names = _as_str(names)
    n = len(names)
    return dict(zip(reversed(names), range(n - 1, -1, -1)))


class CommunityIndex:
    """Communities resolved once against the global node ids, then per computational graph by id (``Explainer.run_batch``).

    Every id a member name has is kept (names may repeat).  ``resolve(subset)`` gives, for the graph whose ascending
    global node ids are ``subset``, exactly what ``Pathways(...).resolve_indices(names[subset])`` gives: a name's index is
    its first occurrence among the graph's names, i.e. the smallest subgraph rank among its ids; communities without a
    member in the graph are dropped; index lists ascending."""

    def __init__(self, communities, community_names, names, first=None):
        names = _as_str(names)
        if first is None:
            first = _first_index(names)
        extra = {}  # name -> its ids after the first (repeated names)
        if len(first) < len(names):
            firsts = np.fromiter(map(first.__getitem__, names), dtype=np.int64, count=len(names))
            for i in np.nonzero(firsts != np.arange(len(names)))[0].tolist():
                extra.setdefault(names[i], []).append(i)
        com, key, gid = [], [], []
        for c, community in enumerate(communities):
            members = _as_str(community)
            ids = np.fromiter(map(first.get, members, itertools.repeat(-1)), dtype=np.int64, count=len(members))
            ids = ids[ids >= 0]
            com.append(np.full(ids.size, c, dtype=np.int64))
            key.append(ids)
            gid.append(ids)
            if extra:
                for m in set(members) & extra.keys():
                    more = np.asarray(extra[m], dtype=np.int64)
                    com.append(np.full(more.size, c, dtype=np.int64))
                    key.append(np.full(more.size, first[m], dtype=np.int64))
                    gid.append(more)
        cat = lambda parts: np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)  # noqa: E731
        self.com, self.key, self.gid = cat(com), cat(key), cat(gid)
        self.community_names = np.arange(len(communities)).tolist() if community_names is None else list(community_names)

    def resolve(self, subset):
        """``subset``: ascending global node ids of one computational graph.  Returns (index lists, community names)."""
        subset = np.asarray(subset, dtype=np.int64)
        if subset.size == 0 or self.gid.size == 0:
            return [], []
        pos = np.searchsorted(subset, self.gid)
        present = subset[np.minimum(pos, subset.size - 1)] == self.gid
        c, k, r = self.com[present], self.key[present], pos[present]
        o = np.lexsort((r, k, c))  # per (community, name): the smallest rank
        c, k, r = c[o], k[o], r[o]
        head = np.ones(c.size, dtype=bool)
        head[1:] = (c[1:] != c[:-1]) | (k[1:] != k[:-1])
        c, r = c[head], r[head]
        o = np.lexsort((r, c))  # per community: distinct ranks, ascending
        c, r = c[o], r[o]
        head = np.ones(c.size, dtype=bool)
        head[1:] = (c[1:] != c[:-1]) | (r[1:] != r[:-1])
        c, r = c[head], r[head]
        if c.size == 0:
            return [], []
        kept, starts = np.unique(c, return_index=True)
        return [part.tolist() for part in np.split(r, starts[1:])], [self.community_names[i] for i in kept.tolist()]


class Pathways:
    def __init__(self, communities, community_names, community_types=None):
        self.communities = communities
        self.community_names = community_names
        self.community_types = community_types
        self.last_index = None
        if self.community_names is None:
            self.community_names = np.arange(len(self.communities)).tolist()

    def comp_graph(self, names):
        """pathways.py:33-102: keep communities with at least one member in the subgraph.
        Members come back as the sorted unique *names* present in ``names`` (what ``intersect1d`` returns).
        The name -> first-index map is kept in ``last_index`` so that ``names2inds`` on the result need not rebuild it."""
        present = self.last_index = _first_index(names)
        sub, sub_names = [], []
        sub_types = [] if self.community_types is not None else None
        for i, (community, cname) in enumerate(zip(self.communities, self.community_names)):
            common = sorted(present.keys() & set(_as_str(community)))
            if len(common) > 0:
                sub.append(common)
                sub_names.append(cname)
                if sub_types is not None:
                    sub_types.append(self.community_types[i])
        if sub_types is not None:
            sub_types = torch.tensor(sub_types, device=self.community_types.device)
        return sub, sub_names, sub_types

    def names2inds(self, names, index=None, filtered=False):
        """pathways.py:104-136: member names -> subgraph indices, in lexicographic name order.
        ``index``: the name -> first-index map of ``names`` if the caller already has it (``comp_graph(...).last_index``);
        ``filtered``: the communities are what ``comp_graph(names)`` returned (sorted unique names, all present), so the
        per-community intersection is the identity and only the lookup remains.  Same result either way."""
        if isinstance(self.communities[0][0], int):
            return self.communities
        first = _first_index(names) if index is None else index
        if filtered:
            return [[first[m] for m in community] for community in self.communities]
        inds = []
        for community in self.communities:
            common = sorted(first.keys() & set(_as_str(community)))
            inds.append([first[m] for m in common])  # intersect1d(return_indices): first occurrence, name order
        return inds

    def resolve_indices(self, names):
        """``comp_graph`` + ``names2inds`` in one pass, for ``Explainer.run``: the communities with at least one member among
        ``names`` as lists of subgraph indices (first occurrence of each name, duplicates collapsed -- what
        ``np.intersect1d(..., return_indices=True)`` yields, pathways.py:84-96,131-134), plus their names.  The lists are in
        ascending index order instead of lexicographic name order: ``Mask.mask_generator`` sorts them numerically in place
        before anything reads them (masks.py:323), and the community mean does not depend on the order.
        One name -> first-index dict, then per community one pass of C-level dict lookups and a numeric sort (measured
        against a vectorised numpy / pandas join over all members: 0.6 s at 564 k names / 1 M members -- the cost is hashing
        scattered Python strings either way)."""
        first = _first_index(names)
        lookup = first.get
        inds, kept = [], []
        for community, cname in zip(self.communities, self.community_names):
            # one C-level pass of dict lookups over the members (absent names give None), duplicates collapse in the set of
            # indices.  (Same 0.42 s as "set(members) & keys, then look the survivors up" at 564 k names / 1 M members: the time
            # is the 1 M probes into a hash table that does not fit the caches.)
            found = set(map(lookup, _as_str(community)))
            found.discard(None)
            if found:
                inds.append(sorted(found))
                kept.append(cname)
        return inds, kept

    def shift_hetero_pathways(self, pointers):
        for key, pointer in zip(list(self.communities.keys()), pointers):
            for i in range(len(self.communities[key])):
                self.communities[key][i] = (np.array(self.communities[key][i]) + pointer).tolist()

    def hetero2homo(self, problem, node_pointers=None, edge_pointers=None):
        """pathways.py:162-232 (note the exact ``problem == "node"`` match of :210-213)."""
        if not isinstance(self.communities, dict):
            return self.communities, self.community_names, None
        keys = list(self.communities.keys())
        first = self.communities[keys[0]][0][0]
        if isinstance(first, (int, float)):
            if problem == "node":
                self.shift_hetero_pathways(node_pointers)
            elif problem == "edge":
                self.shift_hetero_pathways(edge_pointers)
        types, homo, homo_names = [], [], []
        for i, key in enumerate(keys):
            types.append(torch.zeros(len(self.communities[key])) + i)
            homo.extend(self.communities[key])
            homo_names.append(self.community_names[key])
        return homo, list(itertools.chain.from_iterable(homo_names)), torch.hstack(types)

    def aggregate(self, config_val, community_inds):
        """pathways.py:387-429: mean importance per community (device), sorted DataFrame."""
        lib = _lib.load()
        dev = require_cuda()
        w = config_val.detach().to(dev, torch.float32).contiguous()
        lens = [len(c) for c in community_inds]
        ptr = torch.tensor(np.concatenate([[0], np.cumsum(lens)]), dtype=torch.int32, device=dev)
        idx = torch.tensor(list(itertools.chain.from_iterable(community_inds)) or [0], dtype=torch.int32, device=dev)
        score = torch.empty(max(len(lens), 1), dtype=torch.float32, device=dev)
        _lib.check(lib.xpgnn_community_mean(w.data_ptr(), ptr.data_ptr(), idx.data_ptr(), len(lens), score.data_ptr(),
                                            _lib.stream_ptr()))
        df = pd.DataFrame({"name": self.community_names, "score": score[:len(lens)].cpu().tolist()}).set_index("name")
        return df.sort_values(by=["score"], ascending=False).dropna()
