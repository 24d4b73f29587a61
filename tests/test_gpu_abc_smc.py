"""ABC-SMC on the GPU (ecdna_b200_abc_smc_propose / _weights / ecdna_b200_abc_smc, DESIGN.md section 9): the two
population kernels against float64 numpy, generation 0 against rejection ABC, every particle against the oracle,
determinism across chunk sizes and GPU counts, the posterior against rejection ABC, and the CLI's files.

Toy problem: birth-death runs to 2 000 cells, the target the oracle's run at (b1 = 1.4, d0 = d1 = 0.2)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import special, stats

import oracle_binding as ob
from test_gpu_parity import oracle_opts

pytestmark = pytest.mark.gpu
BINS = 128
THR = (0.2, 0.5, 0.5, 0.5)
BOX = dict(b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.0, 0.5))
DOMAIN = 0x5A1C5A1C  # the proposals' Philox domain (abc_smc.cu)
UINT64_MAX = 2**64 - 1


@pytest.fixture(scope="module")
def problem(pkg):
    o = pkg.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=2000, runs=1, save_snapshots=False)
    target = ob.run(oracle_opts(o, 260), hist_cap=BINS).hist
    return o, target


@pytest.fixture(scope="module")
def mc(pkg):
    m = pkg.MultiContext([0])
    yield m
    m.close()


def _u53(a, b):
    return ((a >> 5).astype(np.float64) * 67108864.0 + (b >> 6).astype(np.float64)) / 9007199254740992.0


def _uniforms(seed, idx):
    """The eight Philox words of draw idx's proposal, as four 53-bit uniforms: parent, b1, d0, d1."""
    w = np.zeros((len(idx), 8), dtype=np.uint64)
    for n, i in enumerate(idx):
        i = int(i)
        for blk in (0, 1):
            w[n, 4 * blk:4 * blk + 4] = ob.philox([DOMAIN, blk, i & 0xFFFFFFFF, i >> 32], [seed & 0xFFFFFFFF, seed >> 32])
    return np.stack([_u53(w[:, 2 * q], w[:, 2 * q + 1]) for q in range(4)], axis=1)


def _rho(dist, stop, thr):
    """The scalar distance of every draw (inf: invalid or not comparable)."""
    rho = np.zeros(len(dist), dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        for j, t in enumerate(np.float32(thr)):
            if not t >= 0:
                continue
            d = dist[:, j]
            r = np.where(d == 0, np.float32(0), np.float32(np.inf)) if t == 0 else (d / t).astype(np.float32)
            rho = np.maximum(rho, np.where(np.isnan(d), np.float32(np.inf), r))
    code = stop & 0xFF
    bad = (code == 5) | (code == 6) | ((stop & 0x100) != 0)
    return np.where(bad, np.float32(np.inf), rho)


def _rejection(pkg, ctx, o, target, seed, idx_begin, n, thr):
    rates = ctx.abc_draw_priors(seed, idx_begin, n, **BOX)
    res = ctx.run(o, n_runs=n, idx_begin=idx_begin, want=("stop_reason", "nminus", "nplus", "abc_distance", "abc_accept"),
                  rates_per_run=rates, abc_target=target.astype(np.uint64), abc_thresholds=thr, snapshots=False)
    ok = (res.abc_accept != 0) & np.isfinite(_rho(res.abc_distance, res.stop_reason, thr))
    return rates, res, ok


@pytest.mark.parametrize("case", ["wide", "narrow"])
def test_proposal_kernel_against_numpy(pkg, ctx, case):
    rng = np.random.default_rng(11)
    M, n, seed, idx0 = 1000, 100_000, 26, 12_345
    if case == "wide":  # truncation negligible: the perturbation is N(0, 1) in sigma units
        box = dict(b1_range=(0.0, 100.0), d0_range=(0.0, 100.0), d1_range=(0.0, 100.0))
        prev = np.column_stack([np.ones(M), rng.uniform(45, 55, (M, 3))]).astype(np.float32)
        sigma = (0.5, 0.25, 0.75)
    else:  # the default box, parents on its edges, d1 fixed
        box = dict(b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.2, 0.2))
        prev = np.column_stack([np.full(M, 1.25), rng.uniform(1, 2, M), rng.uniform(0, 0.5, M), np.full(M, 0.2)]).astype(
            np.float32)
        prev[::4, 1], prev[1::4, 1], prev[::3, 2], prev[1::3, 2] = 1.0, 2.0, 0.0, 0.5
        sigma = (0.4, 0.3, 0.1)
    w = rng.uniform(0.1, 1.0, M)
    cum = np.cumsum(w / w.sum())
    rates, parent = ctx.abc_smc_propose(seed, idx0, n, prev, cum, sigma, **box)
    u = _uniforms(seed, np.arange(idx0, idx0 + n, dtype=np.uint64))
    np.testing.assert_array_equal(parent, np.searchsorted(cum, u[:, 0] * cum[-1], side="right"))
    np.testing.assert_array_equal(rates[:, 0], prev[parent, 0])
    ranges = [box["b1_range"], box["d0_range"], box["d1_range"]]
    for k in range(3):
        lo, hi = np.float32(ranges[k][0]), np.float32(ranges[k][1])
        x = rates[:, k + 1]
        assert np.all((x >= lo) & (x <= hi))
        if lo == hi:
            np.testing.assert_array_equal(x, prev[parent, k + 1])  # a fixed parameter is never perturbed
            continue
        p = prev[parent, k + 1].astype(np.float64)
        a, b = (np.float64(lo) - p) / sigma[k], (np.float64(hi) - p) / sigma[k]
        fa, fb = special.ndtr(a), special.ndtr(b)
        ref = np.clip(p + sigma[k] * special.ndtri(fa + u[:, k + 1] * (fb - fa)), lo, hi)
        err = np.abs(x.astype(np.float64) - ref)
        assert np.all(err <= 1e-5 * sigma[k] + np.spacing(np.float32(ref)).astype(np.float64)), float(err.max())
        if case == "wide":
            z = (x.astype(np.float64) - p) / sigma[k]
            assert stats.kstest(z, "norm").pvalue > 1e-3
    if case == "narrow":
        assert np.mean(rates[:, 2] < 0.05) > 0.05  # the parents on d0 = 0 keep their mass inside the box


def _weights_ref(new, prev, w, sigma, ranges, with_z=True):
    s = np.asarray(sigma, dtype=np.float64)
    p = prev[:, 1:].astype(np.float64)
    lo, hi = np.array([r[0] for r in ranges], dtype=np.float64), np.array([r[1] for r in ranges], dtype=np.float64)
    z = np.prod(special.ndtr((hi - p) / s) - special.ndtr((lo - p) / s), axis=1) if with_z else np.ones(len(p))
    wz = w / z
    out = np.zeros(len(new))
    x = new[:, 1:].astype(np.float64)
    for b in range(0, len(new), 512):
        q = (((x[b:b + 512, None, :] - p[None, :, :]) / s) ** 2).sum(axis=2)
        out[b:b + 512] = np.exp(-0.5 * q) @ wz
    out = 1.0 / out
    return out / out.sum()


def test_weights_kernel_against_float64(pkg, ctx):
    rng = np.random.default_rng(3)
    N = M = 4096
    ranges = [BOX["b1_range"], BOX["d0_range"], BOX["d1_range"]]

    def particles(n):
        x = np.column_stack([np.ones(n), rng.uniform(1, 2, n), rng.uniform(0, 0.5, (n, 2))]).astype(np.float32)
        x[::5, 2] = 0.0            # on the edge d0 = 0
        x[1::5, 3] = 0.5           # on the edge d1 = 0.5
        x[2::5, 1] = 1.0 + rng.uniform(0, 0.01, len(x[2::5]))  # near b1 = 1
        x[3::5, 2] = rng.uniform(0, 0.005, len(x[3::5]))       # near d0 = 0
        return x
    prev, new = particles(M), particles(N)
    w = rng.uniform(0.2, 1.0, M)
    w /= w.sum()
    sigma = (0.3, 0.1, 0.12)
    got = ctx.abc_smc_weights(new, prev, w, sigma, **BOX)
    ref = _weights_ref(new, prev, w, sigma, ranges)
    np.testing.assert_allclose(got, ref, rtol=1e-5)
    assert abs(got.sum() - 1.0) < 1e-12
    # the truncation normaliser matters at these edges: without it the weights are off by far more than the tolerance
    assert np.max(np.abs(_weights_ref(new, prev, w, sigma, ranges, with_z=False) / ref - 1)) > 1e-2
    again = ctx.abc_smc_weights(new, prev, w, sigma, **BOX)
    np.testing.assert_array_equal(again.view(np.uint64), got.view(np.uint64))
    # a fixed parameter has no factor: the same weights as without the parameter's differences
    prev2, new2 = prev.copy(), new.copy()
    prev2[:, 3] = new2[:, 3] = 0.25
    fixed = ctx.abc_smc_weights(new2, prev2, w, sigma, b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.25, 0.25))
    np.testing.assert_allclose(fixed, _weights_fixed_ref(new2, prev2, w, sigma, ranges), rtol=1e-5)


def _weights_fixed_ref(new, prev, w, sigma, ranges):
    """Reference with d1 fixed: only b1 and d0 have a factor."""
    s = np.asarray(sigma[:2], dtype=np.float64)
    p = prev[:, 1:3].astype(np.float64)
    lo, hi = np.array([ranges[0][0], ranges[1][0]]), np.array([ranges[0][1], ranges[1][1]])
    z = np.prod(special.ndtr((hi - p) / s) - special.ndtr((lo - p) / s), axis=1)
    x = new[:, 1:3].astype(np.float64)
    out = np.zeros(len(new))
    for b in range(0, len(new), 512):
        q = (((x[b:b + 512, None, :] - p[None, :, :]) / s) ** 2).sum(axis=2)
        out[b:b + 512] = np.exp(-0.5 * q) @ (w / z)
    out = 1.0 / out
    return out / out.sum()


def test_generation0_is_rejection_abc(pkg, ctx, mc, problem):
    o, target = problem
    M = 200
    r = mc.abc_smc(o, target, THR, M, max_generations=1, chunk=700, **BOX)
    assert r["generations"] == 1 and r["status"] == "max_generations"
    assert r["epsilon"][0] == np.inf and np.all(r["parent_idx"][0] == UINT64_MAX)
    np.testing.assert_array_equal(r["weight"][0], np.full(M, 1.0 / M))
    n = int(r["consumed"][0])
    rates, res, _ = _rejection(pkg, ctx, o, target, o.seed, o.idx_begin, n, (np.inf,) * 4)
    valid = np.nonzero(np.isfinite(_rho(res.abc_distance, res.stop_reason, THR)))[0]
    assert len(valid) == M and valid[-1] == n - 1
    np.testing.assert_array_equal(r["idx"][0], o.idx_begin + valid)
    np.testing.assert_array_equal(r["rates"][0], rates[valid])
    np.testing.assert_array_equal(r["distance"][0].view(np.uint32), res.abc_distance[valid].view(np.uint32))
    np.testing.assert_array_equal(r["cells"][0], (res.nminus + res.nplus)[valid])
    assert r["simulated"][0] >= n and r["simulated"][0] % 700 == 0


@pytest.fixture(scope="module")
def run4(mc, problem):
    o, target = problem
    return mc.abc_smc(o, target, THR, 300, max_generations=6, chunk=4096, **BOX)


def test_every_particle_is_an_accepted_simulation(pkg, problem, run4):
    o, target = problem
    r = run4
    G = r["generations"]
    assert G >= 3, r["epsilon"]
    eps = r["epsilon"]
    assert np.all(np.diff(eps) <= 0) and eps[0] == np.inf and np.all(eps[1:] >= 1)
    thr = np.float32(THR)
    for t in range(G):
        w = r["weight"][t]
        assert np.all(w > 0) and abs(w.sum() - 1.0) < 1e-6
        assert 0 < r["ess"][t] <= 300 + 1e-9 and r["consumed"][t] >= 300 and r["simulated"][t] >= r["consumed"][t]
        assert np.all(np.diff(r["idx"][t].astype(np.int64)) > 0)
        if t:
            assert r["idx"][t][0] > r["idx"][t - 1][-1]
            assert np.all(np.isin(r["parent_idx"][t], r["idx"][t - 1]))
            lim = thr * np.float32(eps[t])
            assert np.all(r["distance"][t] <= lim[None, :])
        rates = r["rates"][t]
        for lo, hi, k in ((1.0, 2.0, 1), (0.0, 0.5, 2), (0.0, 0.5, 3)):
            assert np.all((rates[:, k] >= np.float32(lo)) & (rates[:, k] <= np.float32(hi)))
        for i in range(t % 7, 300, 37):  # a strided sample against the oracle, on the particle's own rates and index
            ref = ob.abc_batch(oracle_opts(o, 0), int(r["idx"][t][i]), 1, rates[i:i + 1], target, tuple(thr * eps[t]), 0,
                               hist_cap=512)
            np.testing.assert_array_equal(r["distance"][t][i].view(np.uint32), ref.distance[0].view(np.uint32))
            assert ref.accept[0] == 1


def _same(a, b):
    assert a["generations"] == b["generations"] and a["status"] == b["status"]
    for k in ("idx", "parent_idx", "cells", "consumed", "epsilon", "rates", "distance", "weight", "ess"):
        x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
        np.testing.assert_array_equal(x.view(np.uint8), y.view(np.uint8), err_msg=k)


def test_result_does_not_depend_on_chunk_size(mc, problem, run4):
    o, target = problem
    _same(mc.abc_smc(o, target, THR, 300, max_generations=6, chunk=512, **BOX), run4)


def test_result_does_not_depend_on_gpu_count(pkg, problem, run4):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible: the multi-GPU run needs two or more")
    o, target = problem
    m = pkg.MultiContext()
    try:
        _same(m.abc_smc(o, target, THR, 300, max_generations=6, chunk=4096, **BOX), run4)
    finally:
        m.close()


def test_budget_returns_the_complete_generations(mc, problem, run4):
    o, target = problem
    budget = int(run4["consumed"][:3].sum()) - 1  # generation 2 cannot complete
    r = mc.abc_smc(o, target, THR, 300, max_generations=6, chunk=1000, max_simulations=budget, **BOX)
    assert r["status"] == "budget" and r["generations"] == 2
    for k in ("idx", "weight", "epsilon", "consumed"):
        np.testing.assert_array_equal(r[k], run4[k][:2], err_msg=k)


def test_driver_rejects_bad_options(pkg, mc, problem):
    o, target = problem
    for kw in (dict(population=0), dict(quantile=0.0), dict(quantile=1.0), dict(max_generations=0),
               dict(b1_range=(2.0, 1.0)), dict(d0_range=(0.3, 0.1))):
        args = dict(dict(population=10, quantile=0.5, max_generations=2), **kw)
        p = args.pop("population")
        box = dict(BOX, **{k: v for k, v in args.items() if k.endswith("_range")})
        rest = {k: v for k, v in args.items() if not k.endswith("_range")}
        with pytest.raises(pkg.EcdnaB200Error, match="status 1"):
            mc.abc_smc(o, target, THR, p, **rest, **box)
    with pytest.raises(pkg.EcdnaB200Error, match="status 1"):
        mc.abc_smc(o, target, (-1.0, -1.0, -1.0, -1.0), 10, **BOX)
    with pytest.raises(pkg.EcdnaB200Error, match="status 1"):
        mc.abc_smc(o, target, THR, 10, rates_per_run=np.ones((1, 4), dtype=np.float32), **BOX)
    # abc_enabled unset
    p = mc.make_params(o, 1)
    opt = pkg.SmcOptionsT()
    opt.population, opt.quantile, opt.max_generations = 10, 0.5, 2
    opt.b1_range[:], opt.d0_range[:], opt.d1_range[:] = BOX["b1_range"], BOX["d0_range"], BOX["d1_range"]
    res = pkg.SmcResultT()
    assert pkg.lib().ecdna_b200_abc_smc(mc._h, C.byref(p), C.byref(opt), C.byref(res)) == 1


def test_posterior_matches_rejection_abc(pkg, ctx, mc, problem):
    """The SMC population at eps = 1 and rejection ABC at the same thresholds sample the same posterior."""
    o, target = problem
    n_rej, thr = 1_000_000, (0.05, 0.1, 0.1, 0.1)  # (C4's thresholds: a small fraction of the prior is accepted)
    rates, res, ok = _rejection(pkg, ctx, o, target, 1234, 10_000_000, n_rej, thr)
    acc = rates[ok][:, 1:].astype(np.float64)
    assert len(acc) >= 2000, len(acc)
    r = mc.abc_smc(o, target, thr, 2000, max_generations=25, max_simulations=20_000_000, **BOX)
    assert r["status"] == "reached", (r["status"], r["epsilon"])
    th, w, ess = r["rates"][-1][:, 1:].astype(np.float64), r["weight"][-1], float(r["ess"][-1])
    assert ess > 200
    for k in range(3):
        m_rej, var = acc[:, k].mean(), acc[:, k].var()
        m_smc = float(np.sum(w * th[:, k]))
        bound = 4 * np.sqrt(var / len(acc) + var / ess)
        assert abs(m_smc - m_rej) <= bound, (k, m_smc, m_rej, bound)
    print(f"SMC: {int(r['simulated'].sum())} draws simulated, {int(r['consumed'].sum())} consumed over "
          f"{r['generations']} generations (eps {r['epsilon'].tolist()}); rejection: {len(acc)} of {n_rej} accepted")


def test_cli_writes_what_write_abc_smc_writes(pkg, mc, tmp_path):
    import json
    pkg.build()
    exe = os.path.join(os.path.dirname(pkg.LIB_PATH), "host", "ecdna")
    o = pkg.SimulationOptions(cells=2000, seed=7, save_snapshots=False)
    target = ob.run(oracle_opts(pkg.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=2000, seed=7), 999),
                    hist_cap=256).hist
    tfile = tmp_path / "target.json"
    tfile.write_text(json.dumps({str(k): int(c) for k, c in enumerate(target) if c}))
    out = tmp_path / "cli"
    r = subprocess.run([exe, "abc", "--target", str(tfile), "--generations", "4", "--population", "150", "--quantile",
                        "0.4", "--max-simulations", "3000000", "--cells", "2000", "--seed", "7", "--thresholds",
                        ",".join(map(str, THR)), "--d1-range", "0.05,0.45", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    res = mc.abc_smc(o, target, THR, 150, quantile=0.4, max_generations=4, max_simulations=3_000_000,
                     b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.05, 0.45))
    py = tmp_path / "py"
    assert pkg.write_abc_smc(str(py), o, res) == res["generations"] >= 2
    names = sorted(os.listdir(py))
    assert sorted(os.listdir(out)) == names and "abc_smc.json" in names
    for f in names:
        assert (out / f).read_bytes() == (py / f).read_bytes(), f
