"""Single-sketch K1 through the key table (k_update_single_v2's table path + k_keytab_flush) against the oracle, bit
for bit.  The path is forced with MB200_K1_KEYTABLE_MIN_EVENTS and witnessed through the MB200_TRACE line."""
import re

import numpy as np
import pytest

import oracle as orc

pytestmark = pytest.mark.gpu

R = 1 << 24  # rows of the key table
ENV = "MB200_K1_KEYTABLE_MIN_EVENTS"


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


@pytest.fixture(scope="module")
def ctx(mb):
    c = mb.Context(0)
    yield c
    c.close()


def _k1_lines(capfd):
    err = capfd.readouterr().err
    return [dict(re.findall(r"(\w+)=(\S+)", ln)) for ln in err.splitlines() if "k1: path=" in ln]


def _keys(rng, n, narrow):
    key = np.minimum(rng.zipf(1.1, n), 10 ** 7).astype(np.int64)
    special = [0, R - 1, R, 2 ** 32 - 1] + ([] if narrow else [-1, -(2 ** 40), 2 ** 62, 2 ** 63 - 1])
    for i, k in enumerate(special):
        key[i::997] = k
    if not narrow:
        key[5::53] = rng.integers(-2 ** 62, 2 ** 62, key[5::53].shape[0])
    return key


@pytest.mark.parametrize("d", [4, 3])
@pytest.mark.parametrize("kind", ["f32", "f64", "u8"])
def test_table_path_bit_exact(mb, ctx, capfd, monkeypatch, kind, d):
    """float, double and narrow inputs; host and device memory; keys 0, R-1, R, 2^32-1, negative and >= 2^62 mixed
    in; negative increments; n % 4 == 3"""
    import torch
    monkeypatch.setenv(ENV, "0")
    monkeypatch.setenv("MB200_TRACE", "1")
    rng = np.random.Generator(np.random.PCG64(900 + d + len(kind)))
    n, w = 400003, 1 << 16
    narrow = kind == "u8"
    key = _keys(rng, n, narrow)
    if narrow:
        quanta = rng.integers(0, 256, n).astype(np.uint8)
        inc = (quanta * 0.5).astype(np.float32)
    else:
        inc = (rng.integers(-6, 11, n) * 0.5).astype(np.float32)
    a, b = orc.hash_params(42, d)
    want = np.zeros((1, d, w))
    orc.bank_update(want, d, w, a, b, None, key, inc)
    for where in ("host", "device"):
        bank = mb.SketchBank(1, w, d, 42, 1, ctx)
        capfd.readouterr()
        if narrow:
            k32 = key.astype(np.uint32)
            if where == "host":
                bank.update_u8(None, k32, quanta)
            else:
                bank.update_u8(None, torch.from_numpy(k32.view(np.int32)).cuda(), torch.from_numpy(quanta).cuda())
        else:
            v = inc.astype(np.float64) if kind == "f64" else inc
            if where == "host":
                bank.update(None, key, v)
            else:
                bank.update(None, torch.from_numpy(key).cuda(), torch.from_numpy(v).cuda())
        bank.check()
        lines = _k1_lines(capfd)
        assert lines and all(ln["path"] == "table" for ln in lines), (where, lines)
        assert sum(int(ln["misses_table"]) for ln in lines) > 0 and sum(int(ln["flushed_keys"]) for ln in lines) > 0
        assert bank.read().tobytes() == want.tobytes(), (kind, d, where)
        bank.close()


def test_table_comes_back_zeroed(mb, ctx, capfd, monkeypatch):
    """two calls in a row on one bank, one call each on two banks of one context with different hash families, and a
    call after mb200_release_workspace: every call starts from an all-zero table"""
    import torch
    from mahout_b200 import _native as N
    monkeypatch.setenv(ENV, "0")
    monkeypatch.setenv("MB200_TRACE", "1")
    rng = np.random.Generator(np.random.PCG64(77))
    n, d, w = 300001, 4, 1 << 18
    k1, k2 = _keys(rng, n, False), _keys(rng, n, False)
    i1 = (rng.integers(-4, 9, n) * 0.5).astype(np.float32)
    i2 = (rng.integers(-4, 9, n) * 0.5).astype(np.float32)
    a, b = orc.hash_params(42, d)
    both = np.zeros((1, d, w))
    orc.bank_update(both, d, w, a, b, None, k1, i1)
    orc.bank_update(both, d, w, a, b, None, k2, i2)
    a7, b7 = orc.hash_params(7, d)
    other = np.zeros((1, d, w))
    orc.bank_update(other, d, w, a7, b7, None, k2, i2)
    capfd.readouterr()
    bank = mb.SketchBank(1, w, d, 42, 1, ctx)
    bank.update(None, torch.from_numpy(k1).cuda(), torch.from_numpy(i1).cuda())
    bank.update(None, torch.from_numpy(k2).cuda(), torch.from_numpy(i2).cuda())
    assert bank.read().tobytes() == both.tobytes()
    bank7 = mb.SketchBank(1, w, d, 7, 1, ctx)
    bank7.update(None, torch.from_numpy(k2).cuda(), torch.from_numpy(i2).cuda())
    assert bank7.read().tobytes() == other.tobytes()
    N.check(N.lib().mb200_release_workspace(ctx.handle), ctx.handle)
    bank7.clear()
    bank7.update(None, torch.from_numpy(k2).cuda(), torch.from_numpy(i2).cuda())
    assert bank7.read().tobytes() == other.tobytes()
    lines = _k1_lines(capfd)
    assert [ln["path"] for ln in lines] == ["table"] * 4
    for bk in (bank, bank7):
        bk.close()


def test_default_threshold_paths(mb, ctx, capfd, monkeypatch):
    """no override: a call of 2^26 events takes the table and one of 2^20 the direct path; both equal the oracle"""
    import torch
    from mahout_b200 import synth
    monkeypatch.delenv(ENV, raising=False)
    monkeypatch.setenv("MB200_TRACE", "1")
    n, d, w = 1 << 26, 4, 1 << 20
    cdf = torch.from_numpy(synth.zipf_cdf(10_000_000, 1.1)).cuda()
    _, item, pref = synth.events_device(ctx, 20240002, 0, n, 1_000_000, cdf, None, want_user=False)
    a, b = orc.hash_params(42, d)
    for m, path in ((n, "table"), (1 << 20, "direct")):
        want = np.zeros((1, d, w))
        orc.bank_update(want, d, w, a, b, None, item[:m].cpu().numpy(), pref[:m].cpu().numpy(),
                        nthreads=orc.max_threads())
        bank = mb.SketchBank(1, w, d, 42, 1, ctx)
        capfd.readouterr()
        bank.update(None, item[:m], pref[:m])
        bank.check()
        lines = _k1_lines(capfd)
        assert [ln["path"] for ln in lines] == [path] and int(lines[0]["n"]) == m
        assert bank.read().tobytes() == want.tobytes(), m
        bank.close()
