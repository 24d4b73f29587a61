"""ABC-SMC on the host side, no GPU needed: the files write_abc_smc produces, the ctypes mirrors of the two new
structs, and the command line of `ecdna abc --generations`."""
import csv
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_result(pkg, G=2, M=3):
    rng = np.random.default_rng(5)
    return {
        "idx": np.arange(G * M, dtype=np.uint64).reshape(G, M) + 260,
        "parent_idx": np.vstack([np.full(M, 2**64 - 1, dtype=np.uint64)] + [np.arange(M, dtype=np.uint64) + 260] * (G - 1)),
        "rates": np.column_stack([np.ones(G * M), rng.uniform(1, 2, G * M), rng.uniform(0, 0.5, (G * M, 2))]).astype(
            np.float32).reshape(G, M, 4),
        "distance": rng.uniform(0, 0.3, (G, M, 4)).astype(np.float32),
        "weight": np.full((G, M), 1.0 / M),
        "cells": np.full((G, M), 2000, dtype=np.uint64),
        "epsilon": np.array([np.inf] + [1.5] * (G - 1), dtype=np.float32),
        "consumed": np.array([10, 40][:G], dtype=np.uint64),
        "simulated": np.array([16, 48][:G], dtype=np.uint64),
        "ess": np.full(G, float(M)),
        "generations": G, "status": "reached",
        "options": {"seed": 26, "idx_begin": 260, "population": M, "quantile": 0.5, "max_generations": 4,
                    "max_simulations": 1000, "b1_range": [1.0, 2.0], "d0_range": [0.0, 0.5], "d1_range": [0.0, 0.5],
                    "thresholds": [0.05, 0.1, -1.0, 0.1]},
    }


def test_write_abc_smc_schema(pkg, tmp_path):
    o = pkg.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=2000, initial={2: 3, 0: 1})
    res = _fake_result(pkg)
    assert pkg.write_abc_smc(str(tmp_path), o, res) == 2
    assert sorted(os.listdir(tmp_path)) == ["abc_gen0.csv", "abc_gen1.csv", "abc_smc.json"]
    assert pkg.SMC_FIELDS == pkg.ABC_FIELDS + ["generation", "epsilon", "weight"]
    raw = open(tmp_path / "abc_gen0.csv", "rb").read()
    assert b"\r" not in raw and raw.startswith((",".join(pkg.SMC_FIELDS) + "\n").encode())
    for t in (0, 1):
        rows = list(csv.DictReader(open(tmp_path / f"abc_gen{t}.csv")))
        assert list(rows[0].keys()) == pkg.SMC_FIELDS and len(rows) == 3
        assert [int(r["idx"]) for r in rows] == [int(x) for x in res["idx"][t]]
        assert [r["parental_idx"] for r in rows] == (["", "", ""] if t == 0 else ["260", "261", "262"])
        assert all(int(r["generation"]) == t for r in rows)
        assert float(rows[0]["epsilon"]) == float(res["epsilon"][t])
        assert abs(sum(float(r["weight"]) for r in rows) - 1.0) < 1e-12
        r, x, d = rows[1], res["rates"][t][1], res["distance"][t][1]
        # the first 16 columns are abc_rows': f1/d1 = cells with ecDNA, f2/d2 = without; f32 values round-trip
        assert np.float32(r["f1"]) == x[1] and np.float32(r["f2"]) == x[0] and np.float32(r["d1"]) == x[3]
        assert np.float32(r["d2"]) == x[2] and np.float32(r["ecdna"]) == d[0] and np.float32(r["entropy"]) == d[2]
        assert r["cells"] == r["tumour_cells"] == "2000" and r["seed"] == "26" and r["timepoint"] == "0"
        assert float(r["init_mean"]) == 1.5 and r["init_cells"] == "4" and r["init_copies"] == "6"
    js = json.load(open(tmp_path / "abc_smc.json"))
    assert list(js) == ["status", "generations", "epsilon", "consumed", "simulated", "ess", "options"]
    assert js["status"] == "reached" and js["generations"] == 2
    assert js["epsilon"] == [float("inf"), 1.5] and js["consumed"] == [10, 40] and js["simulated"] == [16, 48]
    assert js["ess"] == [3.0, 3.0]
    assert js["options"] == res["options"]


def test_smc_structs_match_the_header(pkg, tmp_path):
    c = tmp_path / "layout.c"
    c.write_text('''
#include <stdio.h>
#include <stddef.h>
#include "ecdna_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu ", sizeof(ecdna_b200_smc_options_t), offsetof(ecdna_b200_smc_options_t, quantile),
         offsetof(ecdna_b200_smc_options_t, max_simulations), offsetof(ecdna_b200_smc_options_t, chunk),
         offsetof(ecdna_b200_smc_options_t, d1_range));
  printf("%zu %zu %zu %zu\\n", sizeof(ecdna_b200_smc_result_t), offsetof(ecdna_b200_smc_result_t, time_ms),
         offsetof(ecdna_b200_smc_result_t, generations), offsetof(ecdna_b200_smc_result_t, status));
  return 0;
}''')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)],
                   check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    O, R = pkg.SmcOptionsT, pkg.SmcResultT
    assert got == [C.sizeof(O), O.quantile.offset, O.max_simulations.offset, O.chunk.offset, O.d1_range.offset,
                   C.sizeof(R), R.time_ms.offset, R.generations.offset, R.status.offset]


@pytest.fixture(scope="module")
def cli(pkg):
    pkg.build()
    return os.path.join(os.path.dirname(pkg.LIB_PATH), "host", "ecdna")


@pytest.mark.parametrize("args, msg", [
    (["abc", "--target", "t.json", "--generations", "0"], "--generations"),
    (["abc", "--target", "t.json", "--generations", "3", "--quantile", "0"], "--quantile"),
    (["abc", "--target", "t.json", "--generations", "3", "--quantile", "1"], "--quantile"),
    (["abc", "--target", "t.json", "--generations", "3", "--quantile", "1.5"], "--quantile"),
    (["abc", "--target", "t.json", "--generations", "3", "--population", "0"], "--population"),
    (["--generations", "3"], "'abc' subcommand"),
    (["abc", "--target", "t.json", "--generations", "3", "--runs", "100"], "cannot be used with '--runs"),
    (["abc", "--target", "t.json", "--population", "100"], "require '--generations"),
])
def test_cli_smc_argument_errors(cli, tmp_path, args, msg):
    """Caught before any device is touched: exit 2 with a clap-style message, nothing written."""
    out = tmp_path / "out"
    r = subprocess.run([cli] + args + [str(out)], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 2 and "error:" in r.stderr and msg in r.stderr, r.stderr
    assert not out.exists()


def test_cli_smc_without_a_gpu_fails_loudly(cli, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the ABC-SMC CLI is covered by the gpu tests")
    (tmp_path / "t.json").write_text('{"0": 5, "1": 3}')
    out = tmp_path / "out"
    r = subprocess.run([cli, "abc", "--generations", "3", "--target", str(tmp_path / "t.json"), str(out)],
                       capture_output=True, text=True)
    assert r.returncode == 101 and "no CPU path" in r.stderr + r.stdout
    assert not out.exists()
