"""oracle/itembased.py (the numpy restatement the GPU's item-based recommender is compared with) against a second,
literal restatement of upstream RecommenderJob's chain in pure Python, and both against two hand-checked answers
through the job's text format.  Also the job's argument errors and Float.toString.  No GPU needed."""
import math

import numpy as np
import pytest

from oracle import itembased as oib

NAN = float("nan")
MIN_VALUE = float(np.float32(1.4e-45))


def literal(prefs, lists, item_ids, max_prefs, boolean_data, how_many, allowed=None):
    """RecommenderJob step by step.  prefs: {userID: {row: pref}}; lists: {row: [(row, sim), ...]} (the similarity
    matrix rows); returns {userID: [(itemID, value), ...]}."""
    out = {}
    for uid in sorted(prefs):
        # ToUserVectorsReducer: RandomAccessSparseVector.set(i, 0) stores nothing
        vec = {r: float(np.float32(p)) for r, p in prefs[uid].items() if p != 0}
        # UserVectorSplitterMapper.maybePruneUserVector: prefs below the P-th largest |pref| become NaN
        if len(vec) > max_prefs:
            smallest = sorted((abs(p) for p in vec.values()), reverse=True)[max_prefs - 1]
            vec = {r: (p if abs(p) >= smallest else NAN) for r, p in vec.items()}
        # SimilarityMatrixRowWrapperMapper puts NaN on the diagonal; PartialMultiplyMapper skips NaN prefs
        partials = []
        for r in sorted(vec):
            if math.isnan(vec[r]):
                continue
            column = dict(lists.get(r, []))
            column[r] = NAN
            partials.append((vec[r], column))
        if not partials:
            continue
        # AggregateAndRecommendReducer
        if boolean_data:
            predictions = dict(partials[0][1])
            for _, column in partials[1:]:
                for i, s in column.items():
                    predictions[i] = predictions.get(i, 0.0) + s
        else:
            num, den, used = {}, {}, {}
            for p, column in partials:
                for i, s in column.items():
                    used[i] = used.get(i, 0) + 1
                    num[i] = num.get(i, 0.0) + s * p
                    den[i] = den.get(i, 0.0) + abs(s)
            predictions = {i: num[i] / den[i] for i in num if used[i] > 1}
        # writeRecommendedItems: (float) value, NaN skipped; TopItemsQueue's sentinel is Float.MIN_VALUE and the
        # comparison is strict; ties go lower itemID first (the project's rule)
        items = []
        for i, v in predictions.items():
            if allowed is not None and int(item_ids[i]) not in allowed:
                continue
            f = float(np.float32(v))
            if not math.isnan(f) and f > MIN_VALUE:
                items.append((int(item_ids[i]), f))
        items.sort(key=lambda t: (-t[1], t[0]))
        if items:
            out[uid] = items[:how_many]
    return out


def lists_from_columns(idx, sim, cnt):
    return {j: [(int(idx[j, e]), float(sim[j, e])) for e in range(int(cnt[j]))] for j in range(idx.shape[0])}


def random_case(seed, n_items=60, n_users=40, k=12, max_prefs_per_user=30, shift=0.0):
    """top-k lists in cosine_topk's layout (distinct entries, sim > 0, (sim desc, row asc)) and de-duplicated prefs
    with ties, zeros and (with shift) negative values"""
    rng = np.random.Generator(np.random.PCG64(seed))
    idx = np.full((n_items, k), -1, np.int64)
    sim = np.zeros((n_items, k))
    cnt = np.zeros(n_items, np.int32)
    for j in range(n_items):
        c = int(rng.integers(0, k + 1))
        others = rng.choice(np.setdiff1d(np.arange(n_items), [j]), c, replace=False)
        s = rng.integers(1, 9, c) / 8.0 * rng.random(c).round(1).clip(0.1)     # ties among similarities
        order = np.lexsort((others, -s))
        idx[j, :c], sim[j, :c], cnt[j] = others[order], s[order], c
    item_ids = rng.permutation(n_items).astype(np.int64) * 7 + 3                # not ascending in row order
    rows, users, prefs = [], [], []
    for u in range(n_users):
        n = int(rng.integers(0, max_prefs_per_user + 1))
        r = np.sort(rng.choice(n_items, n, replace=False))
        p = (rng.integers(0, 11, n) * 0.5 + shift).astype(np.float32)
        rows.append(r)
        users.append(np.full(n, 1000 - 3 * u, np.int64))
        prefs.append(p)
    return (idx, sim, cnt), item_ids, np.concatenate(rows), np.concatenate(users), np.concatenate(prefs)


def run_both(lists, item_ids, row, user, pref, how_many, max_prefs, boolean_data, allowed_ids=None):
    ids, ptr, prow, pval = oib.user_csr(row, user, pref)
    allowed = None if allowed_ids is None else np.isin(item_ids, list(allowed_ids))
    gi, gv, gc = oib.recommend(*lists, ptr, prow, pval, item_ids, np.arange(ids.shape[0]), how_many, max_prefs,
                               boolean_data, allowed)
    got = {int(ids[t]): list(zip(gi[t, :gc[t]].tolist(), gv[t, :gc[t]].tolist())) for t in range(ids.shape[0])
           if gc[t]}
    prefs = {}
    for r, u, p in zip(row, user, pref):
        prefs.setdefault(int(u), {})[int(r)] = p
    want = literal(prefs, lists_from_columns(*lists), item_ids, max_prefs, boolean_data, how_many, allowed_ids)
    return got, want


@pytest.mark.parametrize("seed,max_prefs,boolean_data,shift,how_many", [
    (1, 10, False, 0.0, 10), (2, 3, False, 0.0, 5), (3, 1000, False, 0.0, 1000), (4, 5, False, -2.5, 7),
    (5, 10, True, 0.0, 10), (6, 1, False, 0.0, 1), (7, 4, True, -1.0, 3)])
def test_oracle_equals_literal_restatement(seed, max_prefs, boolean_data, shift, how_many):
    lists, item_ids, row, user, pref = random_case(seed, shift=shift)
    got, want = run_both(lists, item_ids, row, user, pref, how_many, max_prefs, boolean_data)
    assert got == want
    assert got, "the case recommends nothing"


def test_oracle_equals_literal_with_allowed_items():
    lists, item_ids, row, user, pref = random_case(11)
    allowed = set(item_ids[::3].tolist())
    got, want = run_both(lists, item_ids, row, user, pref, 10, 10, False, allowed)
    assert got == want and got
    assert all(i in allowed for recs in got.values() for i, _ in recs)


def test_pruning_keeps_ties_at_the_threshold():
    vals = np.array([5, 4, 4, 4, 1, 0, -4], np.float32)
    assert oib.considered(vals, 2).tolist() == [True, True, True, True, False, False, True]
    assert oib.considered(vals, 10).tolist() == [True] * 5 + [False, True]
    assert oib.considered(np.ones(20, np.float32), 3).all()                  # boolean data is never pruned


# ---- hand-checked answers through the job's text format ---------------------------------------------------------
def exact_lists(text, boolean_data=False, k=100):
    """cosine_topk of the exact measure on a tiny input: item rows = ascending itemIDs"""
    ev = [tuple(float(x) for x in line.split(",")) for line in text.strip().split("\n")]
    users = sorted({int(u) for u, _, _ in ev})
    items = sorted({int(i) for _, i, _ in ev})
    M = np.zeros((len(items), len(users)))
    for u, i, p in ev:
        M[items.index(int(i)), users.index(int(u))] = 1.0 if boolean_data else p
    n = len(items)
    idx = np.full((n, k), -1, np.int64)
    sim = np.zeros((n, k))
    cnt = np.zeros(n, np.int32)
    for a in range(n):
        cand = []
        for b in range(n):
            if b != a:
                s = float(M[a] @ M[b]) / (math.sqrt(M[a] @ M[a]) * math.sqrt(M[b] @ M[b]))
                if s > 0:
                    cand.append((-s, b))
        cand.sort()
        for e, (s, b) in enumerate(cand[:k]):
            idx[a, e], sim[a, e] = b, -s
        cnt[a] = min(len(cand), k)
    row = np.array([items.index(int(i)) for _, i, _ in ev])
    user = np.array([int(u) for u, _, _ in ev])
    pref = np.array([1.0 if boolean_data else p for _, _, p in ev], np.float32)
    return (idx, sim, cnt), np.array(items, np.int64), row, user, pref


def job_text(case, boolean_data):
    from mahout_b200.recommenditembased import format_line
    lists, item_ids, row, user, pref = case
    got, want = run_both(lists, item_ids, row, user, pref, 10, 10, boolean_data)
    assert got == want
    return "".join(format_line(u, [i for i, _ in recs], [v for _, v in recs]) for u, recs in sorted(got.items()))


HAND_1 = "1,1,5\n1,2,3\n2,1,4\n2,2,2\n2,3,5\n3,2,1\n3,3,4\n4,1,2\n4,3,1\n"
HAND_2 = "2,1,1\n1,2,1\n3,4,1\n1,3,2\n2,3,1\n"     # ItemSimilarityJobTest.testCompleteJob


def test_hand_checked_answer_exact_measure():
    assert job_text(exact_lists(HAND_1), False) == "1\t[3:3.9341865]\n3\t[1:2.0673192]\n4\t[2:1.6134744]\n"
    s13, s23 = 22 / math.sqrt(1890), 14 / math.sqrt(588)
    assert float(np.float32((5 * s13 + 3 * s23) / (s13 + s23))) == float(np.float32(3.9341865))


def test_hand_checked_answer_boolean_data():
    assert job_text(exact_lists(HAND_2, True), True) == "1\t[1:0.70710677]\n2\t[2:0.70710677]\n"
    assert job_text(exact_lists(HAND_2, False), False) == ""        # no item reaches 2 datapoints


# ---- the job's argument errors and Float.toString ------------------------------------------------------------
def test_cli_argument_errors_return_minus_one(tmp_path):
    from mahout_b200.recommenditembased import RecommenderJob
    p = tmp_path / "in.csv"
    p.write_text(HAND_1)
    base = ["--input", str(p), "--output", str(tmp_path / "out")]
    assert RecommenderJob().run([]) == -1                                             # required options
    assert RecommenderJob().run(base) == -1                                           # no similarityClassname
    assert RecommenderJob().run(base + ["-s", "SIMILARITY_TANIMOTO_COEFFICIENT"]) == -1
    assert RecommenderJob().run(base + ["-s", "SIMILARITY_COSINE", "--bogus", "1"]) == -1
    for flag in ("--filterFile", "--userItemFile", "--sequencefileOutput"):
        assert RecommenderJob().run(base + ["-s", "SIMILARITY_COSINE", flag, "x"]) == -1
    for bad in (["--numRecommendations", "0"], ["--numRecommendations", "1025"], ["--maxPrefsPerUser", "0"],
                ["--maxSimilaritiesPerItem", "0"]):
        assert RecommenderJob().run(base + ["-s", "SIMILARITY_COSINE"] + bad) == -1
    assert not (tmp_path / "out").exists()


@pytest.mark.parametrize("v,s", [(1.0, "1.0"), (0.001, "0.001"), (1e-4, "1.0E-4"), (1e7, "1.0E7"),
                                 (9999999.0, "9999999.0"), (0.70710677, "0.70710677"), (float("nan"), "NaN"),
                                 (-2.5, "-2.5"), (1.4e-45, "1.4E-45"), (3.9341865, "3.9341865")])
def test_java_float_to_string(v, s):
    from mahout_b200.similarity import java_float_to_string
    assert java_float_to_string(v) == s
