"""Host-side checks of the exact-input oracle of tests/test_gpu_headtail_configs.py (no GPU needed): on its grid the fp32
convolution sum is the same number in every summation order, the planted ties are exact half midpoints that
round-to-nearest-even resolves the same way in fp64 -> half and fp32 -> half, and its cases cover the launch space of
the fused head-tail kernel."""
import numpy as np
import pytest
import torch

from test_gpu_headtail_configs import CASES, derive, exact_case, half_midpoint

# the widest head any of those tests runs (test_shared_memory_sizing): c3 = 448 at nc = 192
WIDE = dict(B=2, tasks=[(80, 448, 192)], levels=[(8, 16)], seed=448 + 192)


def _pairwise(p):
    """fp32 tree sum over axis 1."""
    while p.shape[1] > 1:
        if p.shape[1] % 2:
            p = np.concatenate([p, np.zeros_like(p[:, :1])], axis=1)
        p = (p[:, 0::2] + p[:, 1::2]).astype(np.float32)
    return p[:, 0]


def _orders(p32, rng):
    """The fp32 sums of p32 [rows, K] over K in several orders."""
    yield "sequential", np.cumsum(p32, axis=1, dtype=np.float32)[:, -1]
    yield "reversed", np.cumsum(p32[:, ::-1], axis=1, dtype=np.float32)[:, -1]
    yield "pairwise", _pairwise(p32)
    yield "numpy", p32.sum(axis=1, dtype=np.float32)
    k = p32.shape[1]
    blocks = np.pad(p32, ((0, 0), (0, -k % 16))).reshape(p32.shape[0], -1, 16).sum(axis=2, dtype=np.float32)
    yield "K=16 blocks", np.cumsum(blocks, axis=1, dtype=np.float32)[:, -1]
    for i in range(3):
        yield f"permutation {i}", np.cumsum(p32[:, rng.permutation(k)], axis=1, dtype=np.float32)[:, -1]


def test_fp32_sum_is_exact_in_every_order():
    host, _ = exact_case(**WIDE)
    rng = np.random.default_rng(0)
    for tower, wk, bk in (("box", "bw", "bb"), ("cls", "cw", "cb")):
        x = host[tower][0][0].numpy().reshape(WIDE["B"], -1, 128)        # [B, c, hw]
        w = host[wk][0][0].numpy().reshape(host[wk][0][0].shape[0], -1)  # [n, c]
        b = host[bk][0][0].numpy()
        prods = (w[None, :, :, None] * x[:, None, :, :]).transpose(0, 1, 3, 2).reshape(-1, x.shape[1])  # [B*n*hw, c]
        s64 = prods.sum(axis=1) + np.repeat(np.tile(b, x.shape[0]), 128)
        p32 = prods.astype(np.float32)
        assert np.array_equal(p32.astype(np.float64), prods), "a product is not an fp32 number"
        b32 = np.repeat(np.tile(b, x.shape[0]), 128).astype(np.float32)
        for name, s in _orders(p32, rng):
            got = (s + b32).astype(np.float64)
            assert np.array_equal(got, s64), f"{tower}: the fp32 sum in {name} order differs from the fp64 sum"
        # the sums need more bits than a half has, so the one rounding left (fp32 -> half) is exercised
        assert np.abs(s64).max() >= 16 and (s64.astype(np.float16).astype(np.float64) != s64).mean() > 0.5


def test_planted_ties_are_half_midpoints():
    host, plants = exact_case(**WIDE)
    assert len(plants) >= 24 and {p[2] for p in plants} == {"box", "cls"}
    for t, l, tower, n, p, v in plants:
        x, w, b = (host["box"], host["bw"], host["bb"]) if tower == "box" else (host["cls"], host["cw"], host["cb"])
        xs = x[t][l][0].reshape(x[t][l].shape[1], -1)
        assert float(w[t][l].reshape(w[t][l].shape[0], -1)[n] @ xs[:, p] + b[t][l][n]) == v
        assert half_midpoint(v), (tower, n, p, v)
        assert float(np.float32(v)) == v  # so the kernel's fp32 sum holds the midpoint itself
        for src in (torch.float64, torch.float32):  # the reference's and the kernel's conversions
            h = torch.tensor(v, dtype=src).half()
            assert h.view(torch.int16).item() % 2 == 0 and float(h) == float(np.float16(v))
    # the example of a planted value: 33 + 2^-6 lies halfway between the halves 33 and 33 + 2^-5 and rounds to 33
    v = 33 + 2.0**-6
    assert half_midpoint(v) and not half_midpoint(33.0) and v * 2**10 == int(v * 2**10)
    assert float(torch.tensor(v, dtype=torch.float64).half()) == 33.0 == float(torch.tensor(v).half())


def test_cerb_library_error_carries_the_return_code():
    from cerberusdet_b200 import _lib

    with pytest.raises(_lib.CerbLibraryError) as err:
        _lib.check(_lib.CERB_ENOSPC)
    assert err.value.code == _lib.CERB_ENOSPC
    assert _lib.CerbLibraryError("python side").code is None


def test_cases_cover_the_launch_space():
    """The derived configurations of CASES hit every value the kernel's launch space distinguishes."""
    ncs = {nc for c in CASES for _, _, nc in c.tasks}
    assert {1, 8, 9, 17, 64, 65, 96, 97, 176, 177, 192} <= ncs
    widths = {w for c in CASES for c2, c3, _ in c.tasks for w in (c2, c3)}
    assert {16, 48, 80, 112, 144, 176, 320} <= widths
    assert {368, 384, 400} <= {c2 + c3 for c in CASES for c2, c3, _ in c.tasks}
    launches = {c.name: derive(c.tasks, len(c.levels)) for c in CASES}
    assert {c.name: len(launches[c.name]) for c in CASES if c.name.startswith("T")} == {"T5": 2, "T8L3": 2, "T4L4": 2, "T8L4": 3}
    nbs = {lc["NB"] for ls in launches.values() for lc in ls}
    assert nbs == {2, 3, 4}
    assert {lc["groups"] for ls in launches.values() for lc in ls} == {1, 2}
    rbs = {r for ls in launches.values() for lc in ls for pair in lc["rb"] for r in pair}
    assert {16, 48, 80, 112, 128} <= rbs
    assert [lc["NB"] for lc in launches["nc64"]] == [4] and [lc["NB"] for lc in launches["nc65"]] == [3]
    assert [lc["NB"] for lc in launches["L1-nc96"]] == [3] and [lc["NB"] for lc in launches["L2-nc97"]] == [2]
    assert [lc["groups"] for lc in launches["sum368"]] == [2] and [lc["groups"] for lc in launches["sum384"]] == [1]
    assert [lc["S"] for lc in launches["nc176"]] == [2] and [lc["S"] for lc in launches["nc192"]] == [4]
    # at 232448 bytes of opt-in shared memory: one ring stage short of fitting from nc = 177 at c2 = 80, c3 = 384
    assert [derive([(80, 384, nc)], 3)[0]["S"] for nc in (176, 177, 192)] == [2, 1, 1]
    assert derive([(80, 448, 192)], 3)[0]["S"] == 1 and derive([(80, 320, 192)], 3)[0]["S"] == 4
    hws = {h * w for c in CASES for h, w in c.levels}
    assert 128 in hws and any(n <= 64 for n in hws) and any(n % 128 not in (0, 64) for n in hws)
    assert any(w == 1 for c in CASES for _, w in c.levels) and any(h != w for c in CASES for h, w in c.levels)
    tiles = {c.name: c.B * sum((h * w + 127) // 128 for h, w in c.levels) for c in CASES}
    assert tiles["persist640"] > 148 * 4 and tiles["nc64"] < 148
