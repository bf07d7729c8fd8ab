"""Item-based recommendation on all GPUs of the process (mb200_itembased_multi_*, csrc/itembased_multi.cu): one
replica of the item lists and user vectors per GPU, users split t mod G.  Every call is checked byte for byte --
itemIDs, float bits, counts and unused slots -- against itembased.recommend on one context, at G = 1, 2, all visible
GPUs and two contexts on GPU 0; and the --numGpus jobs against the single-GPU jobs' files."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from test_itembased_gpu import Case

pytestmark = pytest.mark.gpu

UNLIMITED = 2 ** 31 - 1


def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(scope="module")
def ctx():
    import mahout_b200 as mb
    c = mb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", params=[1, 2, 0, "0,0"], ids=["G1", "G2", "Gall", "G2-one-device"])
def multi(request):
    """a MultiGpu over 1, 2 or all visible GPUs (the last only when that is more than 2), and two contexts on GPU 0:
    the split, the scatter and a failure on the second worker at G = 2 on a one-GPU machine"""
    from mahout_b200.multi import MultiGpu
    have = _gpus()
    g = request.param
    if g == 2 and have < 2:
        pytest.skip("needs 2 GPUs")
    if g == 0 and have <= 2:
        pytest.skip("all visible GPUs is already covered")
    m = MultiGpu(devices=[0, 0]) if g == "0,0" else MultiGpu(g)
    yield m
    m.close()


def _many(multi, c, device=False):
    from mahout_b200 import itembased as ib
    lists, uv, ids = c.lists, ib.UserVectors(c.uids, c.ptr, c.prow, c.pval), c.item_ids
    if device:
        import torch
        t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()   # noqa: E731
        lists = tuple(t(x) for x in lists)
        uv = ib.UserVectors(*(t(x) for x in (c.uids, c.ptr, c.prow, c.pval)))
        ids = t(ids)
    return multi.item_based(lists, uv, ids)


def _same(got, want):
    for g, w in zip(got, want):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape and g.dtype == w.dtype
        assert g.tobytes() == w.tobytes()


def _check(many, c, users=None, how_many=10, max_prefs=10, boolean_data=False, allowed_ids=None):
    """one MultiItemBased call against the same call on one context"""
    from mahout_b200 import itembased as ib
    mask = None if allowed_ids is None else ib.allowed_mask(c.item_ids, allowed_ids)
    want = c.run(users=users, how_many=how_many, max_prefs=max_prefs, boolean_data=boolean_data,
                 allowed_ids=allowed_ids)
    got = many.recommend(users, how_many, max_prefs, boolean_data, mask)
    _same(got, want)
    return got


def _plans(multi):
    from mahout_b200 import _native as N
    out = []
    for h in multi.contexts():
        pl = N.ItemBasedPlan()
        N.check(N.lib().mb200_itembased_last_plan(h, C.byref(pl)))
        out.append({f: getattr(pl, f) for f, _ in pl._fields_})
    return out


def _launches(multi):
    from mahout_b200 import _native as N
    out = []
    for h in multi.contexts():
        n = C.c_int64()
        N.check(N.lib().mb200_launch_count(h, C.byref(n)))
        out.append(n.value)
    return out


@pytest.mark.parametrize("exact", [False, True])
def test_table_path_all_users(ctx, multi, exact):
    """every user in the shared-memory table; how_many 1, 10 and 1024; an allowed mask; rating shift"""
    for shift in (0.0, -2.5):
        c = Case(ctx, 3 + int(exact), shift=shift, exact=exact)
        many = _many(multi, c)
        for how_many in (1, 10, 1024):
            got = _check(many, c, how_many=how_many)
            assert (got[2] > 0).any()
        _check(many, c, how_many=15, allowed_ids=set(c.item_ids[::4].tolist()))
        assert sum(p["dense_users"] for p in _plans(multi)) == 0
        many.close()


@pytest.mark.parametrize("exact", [False, True])
def test_dense_path(ctx, multi, exact):
    """maxPrefsPerUser unlimited: users above 1024 entries take the dense slices, the others the table"""
    c = Case(ctx, 8 + int(exact), n_items=3000, n_users=400, max_n=200, k=100, exact=exact)
    many = _many(multi, c)
    for max_prefs in (UNLIMITED, 50):
        _check(many, c, how_many=50, max_prefs=max_prefs)
        plans = _plans(multi)
        assert sum(p["dense_users"] for p in plans) > 0 and sum(p["smem_users"] for p in plans) > 0, plans
    _check(many, c, how_many=1024, max_prefs=UNLIMITED, allowed_ids=set(c.item_ids[::3].tolist()))
    many.close()


@pytest.mark.parametrize("exact", [False, True])
def test_boolean_data(ctx, multi, exact):
    c = Case(ctx, 12, boolean_data=True, exact=exact)
    many = _many(multi, c)
    for max_prefs in (10, UNLIMITED):
        got = _check(many, c, how_many=20, max_prefs=max_prefs, boolean_data=True)
        assert (got[2] > 0).any()
    many.close()


def test_device_inputs(ctx, multi):
    """lists, user vectors and itemIDs from device memory replicate the same data"""
    c = Case(ctx, 16)
    many = _many(multi, c, device=True)
    _check(many, c, how_many=12, allowed_ids=set(c.item_ids[::3].tolist()))
    many.close()


def test_shuffled_subset_fewer_users_than_gpus_and_none(ctx, multi):
    c = Case(ctx, 15)
    U = c.uids.shape[0]
    many = _many(multi, c)
    rng = np.random.Generator(np.random.PCG64(5))
    users = rng.permutation(np.concatenate([rng.choice(U, 200, replace=False), rng.choice(U, 40)]))
    users[7] = users[3] = users[100]
    _check(many, c, users=users, how_many=17)
    G = multi.n_gpus
    few = np.array([U - 1, 0, 17][: max(G - 1, 1)], np.int64)            # fewer users than GPUs when G > 1
    _check(many, c, users=few)
    assert many.stats()["work"] == [len(range(g, few.shape[0], G)) for g in range(G)]
    items, vals, cnt = many.recommend(np.zeros(0, np.int64), how_many=10)
    assert items.shape == (0, 10) and vals.shape == (0, 10) and cnt.shape == (0,)
    assert many.stats()["work"] == [0] * G
    many.close()


def test_stats_follow_the_split(ctx, multi):
    c = Case(ctx, 17, n_users=120)
    U = c.uids.shape[0]
    many = _many(multi, c)
    G = multi.n_gpus
    assert many.stats()["work"] == [U] * G                               # create: every GPU holds every user
    rng = np.random.Generator(np.random.PCG64(7))
    for q in (1, G + 1, 59, U):
        many.recommend(rng.integers(0, U, q), how_many=5)
        st = many.stats()
        assert st["work"] == [len(range(g, q, G)) for g in range(G)]
        assert len(st["seconds"]) == G and all(s >= 0 for s in st["seconds"])
        assert st["wall_s"] >= max(st["seconds"]) * 0.5
    many.close()


def test_bad_arguments_then_a_good_call(ctx, multi):
    from mahout_b200 import _native as N
    c = Case(ctx, 18, n_users=80)
    U = c.uids.shape[0]
    many = _many(multi, c)
    users = np.arange(U)

    def good():
        _check(many, c, how_many=10)

    good()
    before = _launches(multi)
    for kw in ({"how_many": 0}, {"how_many": 1025}, {"max_prefs_per_user": 0},
               {"allowed": np.zeros(3, np.uint32)}):
        with pytest.raises(ValueError):
            many.recommend(users, **kw)
    L = N.lib()
    h = C.c_void_p()
    raw = [  # m < 0 and NULL arrays through the C ABI itself
        lambda: L.mb200_itembased_multi_recommend(many.handle, None, -1, 10, 10, 0, None, None, None, None),
        lambda: L.mb200_itembased_multi_recommend(many.handle, None, 5, 10, 10, 0, None, None, None, None),
        lambda: L.mb200_itembased_multi_create(multi._h, None, None, None, 10, 5, None, None, None, 3, 0, None,
                                               C.byref(h)),
        lambda: L.mb200_itembased_multi_create(multi._h, None, None, None, 0, 0, None, None, None, 0, 0, None,
                                               C.byref(h)),
    ]
    for call in raw:
        assert call() == N.ERR_BAD_ARG
    assert _launches(multi) == before                                   # nothing reached a GPU
    good()
    # a user row out of range at position 1: the second worker's share (the first's with one GPU)
    bad = users.copy()
    bad[1] = U
    name = f"GPU {multi.devices[1 % multi.n_gpus]}:"
    with pytest.raises(ValueError, match=name):
        many.recommend(bad)
    good()
    bad[1] = -1
    with pytest.raises(ValueError, match=name):
        many.recommend(bad, how_many=3, max_prefs_per_user=UNLIMITED)
    good()
    # a malformed user CSR, found on the device by the first GPU's worker
    from mahout_b200 import itembased as ib
    ptr = c.ptr.copy()
    ptr[5] = ptr[6] + 1
    broken = multi.item_based(c.lists, ib.UserVectors(c.uids, ptr, c.prow, c.pval), c.item_ids)
    with pytest.raises(ValueError, match=f"GPU {multi.devices[0]}:"):
        broken.recommend(np.array([5, 0, 1]))
    broken.close()
    good()
    many.close()


# ---- the jobs with --numGpus ----------------------------------------------------------------------------------------

def _write_input(path, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    n = 8000
    u = rng.integers(1, 301, n) * 3
    i = rng.integers(1, 400, n) * 11
    p = rng.integers(1, 11, n) * 0.5
    path.write_text("".join(f"{a},{b},{c}\n" for a, b, c in zip(u, i, p)))


def _gpu_counts():
    have = _gpus()
    return sorted({1, min(2, have)}) + [0]                              # 0 = every visible GPU


@pytest.mark.parametrize("measure", ["SIMILARITY_COSINE", "SIMILARITY_SKETCH_COSINE"])
def test_recommenditembased_num_gpus_writes_the_same_file(tmp_path, measure):
    """--numGpus 1 / 2 / all: the job's file (and the similarity matrix) byte-identical to the single-GPU job's, at
    --precision rescored, where the multi-GPU similarity lists equal the single-GPU ones bit for bit"""
    from mahout_b200.recommenditembased import RecommenderJob
    from mahout_b200.seqfile import read_sequence_file
    inp = tmp_path / "in.csv"
    _write_input(inp, 31)
    users_file, items_file = tmp_path / "users.txt", tmp_path / "items.txt"
    users_file.write_text("".join(f"{3 * u}\n" for u in range(1, 301, 2)))
    items_file.write_text("".join(f"{11 * i}\n" for i in range(1, 400, 3)))
    base = ["--input", str(inp), "-s", measure, "-m", "30", "--sketchWidth", "1024", "--sketchDepth", "3",
            "--precision", "rescored"]
    variants = [[], ["--numRecommendations", "25", "--maxPrefsPerUser", "5", "--usersFile", str(users_file),
                     "--itemsFile", str(items_file), "--booleanData", "true"]]
    for v, extra in enumerate(variants):
        single, smat = tmp_path / f"single{v}.txt", tmp_path / f"single{v}.mat"
        assert RecommenderJob().run(base + extra + ["--output", str(single),
                                                    "--outputPathForSimilarityMatrix", str(smat)]) == 0
        assert len(single.read_text().splitlines()) > 50
        for g in _gpu_counts():
            out, mat = tmp_path / f"g{g}_{v}.txt", tmp_path / f"g{g}_{v}.mat"
            job = RecommenderJob()
            assert job.run(base + extra + ["--output", str(out), "--outputPathForSimilarityMatrix", str(mat),
                                           "--numGpus", str(g)]) == 0
            assert out.read_bytes() == single.read_bytes(), (g, extra)
            # the records (the sync marker is derived from the path)
            assert read_sequence_file(str(mat)) == read_sequence_file(str(smat)), g
            assert {"prepare", "similarity", "replicate", "recommend", "write"} <= set(job.phase_s)


def test_recommenditembased_bad_num_gpus_and_unsupported_flags(tmp_path, capsys):
    from mahout_b200.recommenditembased import RecommenderJob
    inp, out = tmp_path / "in.csv", tmp_path / "out.txt"
    _write_input(inp, 32)
    base = ["--input", str(inp), "--output", str(out), "-s", "SIMILARITY_COSINE"]
    for n in ("-1", str(_gpus() + 1)):
        assert RecommenderJob().run(base + ["--numGpus", n]) == -1
        assert "GPUs asked for" in capsys.readouterr().err
    assert not out.exists()
    for flag in ("--filterFile", "--userItemFile", "--sequencefileOutput"):
        assert RecommenderJob().run(base + ["--numGpus", "1", flag, "x"]) == -1
    assert RecommenderJob().run(base + ["--numGpus", "1", "--numRecommendations", "0"]) == -1


@pytest.mark.parametrize("measure", ["SIMILARITY_COSINE", "SIMILARITY_SKETCH_COSINE"])
def test_python_itemsimilarity_num_gpus_equals_native(tmp_path, measure):
    """the Python mirror with --numGpus N writes the native driver's file with --numGpus N, byte for byte"""
    from mahout_b200 import build
    from mahout_b200.itemsimilarity import ItemSimilarityJob
    rng = np.random.Generator(np.random.PCG64(33))
    n = 20000
    inp = tmp_path / "prefs.csv"
    inp.write_text("".join(f"{u},{i * 5},{p}\n" for u, i, p in zip(rng.integers(1, 500, n), rng.integers(1, 300, n),
                                                                   rng.integers(1, 11, n) * 0.5)))
    flags = ["-s", measure, "-m", "9", "-mp", "2", "--sketchWidth", "1024", "--sketchDepth", "4", "--threshold", "0.05"]
    for g in _gpu_counts():
        py_out, cc_out = tmp_path / f"py{g}.tsv", tmp_path / f"cc{g}.tsv"
        assert ItemSimilarityJob().run(["-i", str(inp), "-o", str(py_out), *flags, "--numGpus", str(g)]) == 0
        r = subprocess.run([build.CLI_BIN, "-i", str(inp), "-o", str(cc_out), *flags, "--numGpus", str(g)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert py_out.read_text() == cc_out.read_text(), g
        assert len(py_out.read_text().splitlines()) > 100
