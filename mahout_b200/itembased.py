"""Item-based recommendation over the item top-k lists: the aggregate-and-recommend phase of upstream RecommenderJob
(UserVectorSplitterMapper, PartialMultiplyMapper, AggregateAndRecommendReducer) as one kernel call, K_RECOMMEND's
`k_itembased` in csrc/recommend.cu.  Independent of SketchBank: any top-k lists in cosine_topk's layout will do.

    lists = item_similarity(row, user, pref, num_items, k, device=True)      # (idx, sim, cnt) on the GPU
    uv = user_vectors(prep.row, prep.user, prep.pref)                        # CSR over user rows, on the GPU
    items, values, counts = recommend(lists, uv, prep.item_id, how_many=10)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from . import sketch as sk

DEFAULT_NUM_RECOMMENDATIONS = 10   # RecommenderJob.DEFAULT_NUM_RECOMMENDATIONS
DEFAULT_MAX_PREFS_PER_USER = 10    # UserVectorSplitterMapper.DEFAULT_MAX_PREFS_PER_USER_CONSIDERED
MAX_HOW_MANY = 1024


class UserVectors:
    """The user vectors as CSR over user rows: user_ids [U] ascending, user_ptr [U+1], pref_row [nnz] int32 item rows
    ascending within a user, pref_val [nnz] float32."""

    def __init__(self, user_ids, user_ptr, pref_row, pref_val):
        self.user_ids, self.user_ptr, self.pref_row, self.pref_val = user_ids, user_ptr, pref_row, pref_val

    @property
    def num_users(self) -> int:
        return int(self.user_ptr.shape[0]) - 1


def user_vectors(row, user, pref) -> UserVectors:
    """CSR of the prepared columns (one pref per (user, item row): Events.prepare), sorted by (userID, row) on the
    device.  Torch does the sorting; these are plumbing, not the hot path."""
    import torch
    row = torch.as_tensor(row)
    dev = row.device if row.is_cuda else torch.device(f"cuda:{sk.default_context().device}")
    row = row.to(dev)
    user = torch.as_tensor(user).to(dev)
    pref = torch.as_tensor(pref).to(dev)
    o1 = torch.sort(row, stable=True).indices
    o2 = torch.sort(user[o1], stable=True).indices
    order = o1[o2]
    u = user[order]
    ids, counts = torch.unique_consecutive(u, return_counts=True)
    ptr = torch.zeros(ids.numel() + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=ptr[1:])
    return UserVectors(ids, ptr, row[order].to(torch.int32).contiguous(), pref[order].to(torch.float32).contiguous())


def allowed_mask(item_id, allowed_ids) -> np.ndarray:
    """bit mask over item rows of the items whose itemID is in allowed_ids (--itemsFile)"""
    item_id = np.asarray(item_id, np.int64)
    hit = np.isin(item_id, np.asarray(list(allowed_ids), np.int64))
    words = np.zeros((item_id.shape[0] + 31) // 32, np.uint32)
    r = np.nonzero(hit)[0]
    np.bitwise_or.at(words, r >> 5, (np.uint32(1) << (r & 31).astype(np.uint32)))
    return words


def recommend(lists, uv: UserVectors, item_id, users=None, how_many: int = DEFAULT_NUM_RECOMMENDATIONS,
              max_prefs_per_user: int = DEFAULT_MAX_PREFS_PER_USER, boolean_data: bool = False, allowed=None,
              ctx: sk.Context | None = None):
    """Recommendations for the user rows `users` (None: every user row) from the item top-k lists (idx [I, k],
    sim [I, k], cnt [I] as cosine_topk returns them).  item_id [I]: row -> itemID.  allowed: optional bit mask over
    item rows (allowed_mask).  Every array host (numpy) or every array device (torch.cuda).  Returns (items [m,
    how_many] int64 itemIDs, values [m, how_many] float32, counts [m] int32); unused slots are -1 / 0."""
    ctx = ctx or sk.default_context()
    idx, sim, cnt = lists
    if users is None:
        users = np.arange(uv.num_users, dtype=np.int64)
        if sk._is_torch(uv.user_ptr) and uv.user_ptr.is_cuda:
            import torch
            users = torch.arange(uv.num_users, dtype=torch.int64, device=uv.user_ptr.device)
    si = sk._Arg(idx, np.int64, "int64")
    sv = sk._Arg(sim, np.float64, "float64")
    sc = sk._Arg(cnt, np.int32, "int32")
    up = sk._Arg(uv.user_ptr, np.int64, "int64")
    pr = sk._Arg(uv.pref_row, np.int32, "int32")
    pv = sk._Arg(uv.pref_val, np.float32, "float32")
    ii = sk._Arg(item_id, np.int64, "int64")
    us = sk._Arg(users, np.int64, "int64")
    al = sk._Arg(allowed, np.uint32, "int32", allow_none=True)
    n_items = sc.n
    ld = si.n // n_items if n_items else 1
    if si.n != n_items * ld or sv.n != si.n or ii.n != n_items or pr.n != pv.n or up.n < 1:
        raise ValueError("lists must be idx / sim [I, k] and cnt [I], item_id [I]; pref_row and pref_val the same "
                         "length")
    if al.ptr is not None and al.n != (n_items + 31) // 32:
        raise ValueError(f"allowed must hold {(n_items + 31) // 32} words for {n_items} items")
    mem = sk._same_mem(si, sv, sc, up, pr, pv, ii, us, al)
    m, n = us.n, int(how_many)
    items, pi = sk._out((m, max(n, 0)), np.int64, "int64", mem, ctx.device)
    vals, pv_ = sk._out((m, max(n, 0)), np.float32, "float32", mem, ctx.device)
    counts, pc = sk._out((m,), np.int32, "int32", mem, ctx.device)
    a = N.ItemBasedArgs(si.ptr, sv.ptr, sc.ptr, n_items, max(ld, 1), up.ptr, pr.ptr, pv.ptr, up.n - 1, pr.n, ii.ptr,
                        al.ptr, us.ptr, m, n, int(max_prefs_per_user), int(bool(boolean_data)), pi, pv_, pc, mem)
    N.check(N.lib().mb200_recommend_item_based(ctx.handle, C.byref(a)), ctx.handle)
    return items, vals, counts


def itembased_plan(ctx: sk.Context | None = None) -> dict:
    """what the last recommend on the context did (mb200_itembased_last_plan)"""
    ctx = ctx or sk.default_context()
    pl = N.ItemBasedPlan()
    N.check(N.lib().mb200_itembased_last_plan(ctx.handle, C.byref(pl)), ctx.handle)
    return {f: getattr(pl, f) for f, _ in pl._fields_}
