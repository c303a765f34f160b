"""The ACL clause for the test references, kept beside them rather than inside oracle/ and the existing test double:

  * ``AclOracleVectorStore``: oracle.OracleVectorStore whose ``search`` takes ``visible_to`` and applies the clause as
    this project defines it (not a Qdrant construct): a row passes if its payload has no ``allowed_users`` (or it is
    None) or if that list shares an entry with ``visible_to``.  An empty list passes for nobody; Qdrant's IsEmpty
    would treat it as public, so that condition is not borrowed.
  * ``ScopedFakeIndex``: the C-oracle test double with ``set_scope`` (vb_set_scope: a write to the scope column).
"""
from __future__ import annotations

import numpy as np

import _acl_data as A
from _fake_index import FakeIndex
from oracle import oracle as O


class _VisibleFilter:
    """A payload filter (or None) plus the ACL clause for ``principals``."""

    def __init__(self, inner, principals):
        self.inner, self.principals = inner, list(principals)


class _AclCollection(O.LocalCollection):
    def _mask(self, flt):
        if not isinstance(flt, _VisibleFilter):
            return super()._mask(flt)
        m = super()._mask(flt.inner)
        return m & np.array([A.visible(p.get("allowed_users"), flt.principals) for p in self.payload], dtype=bool)


class AclOracleVectorStore(O.OracleVectorStore):
    def __init__(self, dim: int, has_sparse: bool = True, fusion: str = "weighted"):
        super().__init__(dim, has_sparse=has_sparse, fusion=fusion)
        self.coll = _AclCollection(dim, has_sparse=has_sparse)

    def search(self, query_embedding, limit=10, folder_filter=None, include_folders=None, exclude_folders=None,
               exclude_index_folders=None, sparse_query=None, sparse_weight=0.1, date_start=None, date_end=None,
               date_field=None, visible_to=None):
        """OracleVectorStore.search with the ACL clause ANDed into the payload filter of both branches."""
        flt = O.build_filter(folder_filter, include_folders, exclude_folders, exclude_index_folders,
                             date_start=date_start, date_end=date_end, date_field=date_field)
        if visible_to is not None:
            flt = _VisibleFilter(flt, visible_to)
        if sparse_query and self._has_sparse:
            indices, values = sparse_query
            if indices:
                dense, sparse = self.search_branches(query_embedding, limit, flt, (indices, values))
                if self.fusion == "rrf":
                    fused = O.reciprocal_rank_fusion([dense, sparse], limit)
                else:
                    fused = O.weighted_fusion(dense, sparse, limit, sparse_weight)
                return [O.payload_to_chunk(pid, r.payload, sc) for pid, sc, r in fused]
        res = self.coll.query_dense(query_embedding, limit, flt)
        return [O.payload_to_chunk(r.id, r.payload, r.score) for r in res]


class ScopedFakeIndex(FakeIndex):
    def set_scope(self, rows, scope_id):
        self.scope[np.asarray(rows, np.int64)] = np.asarray(scope_id, np.uint32)
        self._cc = None
