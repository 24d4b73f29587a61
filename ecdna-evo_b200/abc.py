"""ABC record writer: the CSV of the reference's removed `abc` binary (abc.md:38-55), one row per
prior draw, ALL draws saved so the thresholds can be tuned afterwards (abc.md:57-71); and the files of an
ABC-SMC run, one CSV per generation's population plus abc_smc.json.

Input is what the kernel's fused epilogue returns per draw (distances, accept flag, final counts) and
the prior draws; nothing is simulated here."""
import csv
import os

import numpy as np

REC_HEADER = 16  # ECDNA_B200_ABC_REC_HEADER: 32-bit words in front of a record's distribution


def record_words(rec_bins):
    return REC_HEADER + rec_bins


def decode_records(words, rec_bins):
    """Records of ecdna_b200_abc_pack ([n][16 + rec_bins] u32) as a dict of arrays (layout: include/ecdna_b200.h)."""
    w = np.ascontiguousarray(words, dtype=np.uint32).reshape(-1, record_words(rec_bins))
    f = w.view(np.float32)
    return {"idx": w[:, 0].astype(np.uint64) | (w[:, 1].astype(np.uint64) << np.uint64(32)), "rates": f[:, 2:6].copy(),
            "distance": f[:, 6:10].copy(), "mean": f[:, 10].copy(), "frequency": f[:, 11].copy(),
            "entropy": f[:, 12].copy(), "cells": w[:, 13].copy(), "kmax": w[:, 14].copy(), "stop": w[:, 15] & 0xFF,
            "hist": w[:, REC_HEADER:].copy()}


def merge_gathered(all_records, all_counts, capacity, rec_bins):
    """What ecdna_b200_abc_allgather leaves on every rank - [world][capacity] record blocks and [world] counts -
    as one [n_accepted_total][words] array in rank order (= index order, ranks own contiguous index blocks)."""
    all_counts = np.asarray(all_counts, dtype=np.int64)
    if np.any(all_counts > capacity):
        raise OverflowError(f"a rank accepted {int(all_counts.max())} draws but the record blocks hold {capacity}: "
                            "raise the capacity and run the exchange again")
    blocks = np.asarray(all_records, dtype=np.uint32).reshape(len(all_counts), capacity, record_words(rec_bins))
    return np.concatenate([blocks[r, : all_counts[r]] for r in range(len(all_counts))], axis=0)


ABC_FIELDS = ["parental_idx", "idx", "timepoint", "seed", "ecdna", "mean", "entropy", "f1", "f2", "d1", "d2", "cells",
              "tumour_cells", "init_mean", "init_cells", "init_copies"]


def abc_rows(opts, idx_begin, rates, abc_distance, nminus, nplus, timepoint=0, sample_cells=None, parental_idx=None):
    """Yield one dict per draw with the columns of abc.md:38-55.

    rates[i] = (b0, b1, d0, d1).  abc.md's naming: f1/d1 belong to the cells WITH ecDNA, f2/d2 to the
    cells WITHOUT.  abc_distance[i] = (ks, rel.mean, rel.entropy, rel.frequency)."""
    init_cells = sum(opts.distribution.values())
    init_copies = sum(k * c for k, c in opts.distribution.items())
    init_mean = init_copies / init_cells if init_cells else 0.0
    for i in range(len(rates)):
        tumour = int(nminus[i]) + int(nplus[i])
        yield {
            "parental_idx": "" if parental_idx is None else parental_idx, "idx": idx_begin + i, "timepoint": timepoint,
            "seed": opts.seed, "ecdna": float(abc_distance[i][0]), "mean": float(abc_distance[i][1]),
            "entropy": float(abc_distance[i][2]), "f1": float(rates[i][1]), "f2": float(rates[i][0]),
            "d1": float(rates[i][3]), "d2": float(rates[i][2]),
            "cells": tumour if sample_cells is None else int(sample_cells), "tumour_cells": tumour,
            "init_mean": init_mean, "init_cells": init_cells, "init_copies": init_copies,
        }


def write_abc_csv(path, opts, idx_begin, rates, abc_distance, nminus, nplus, **kw):
    with open(path, "w", newline="") as f:
        w = csv.DictWriter(f, fieldnames=ABC_FIELDS)
        w.writeheader()
        n = 0
        for row in abc_rows(opts, idx_begin, rates, abc_distance, nminus, nplus, **kw):
            w.writerow(row)
            n += 1
    return n


SMC_FIELDS = ABC_FIELDS + ["generation", "epsilon", "weight"]


def _g9(x):
    """printf("%.9g") of an f32 value: what `ecdna abc` writes (it round-trips f32)."""
    return "%.9g" % float(x)


def _g17(x):
    """printf("%.17g") of an f64 value (round-trips f64)."""
    return "%.17g" % float(x)


def _cell(v):
    return _g9(v) if isinstance(v, float) else str(v)


def _json_float(s):
    return {"inf": "Infinity", "-inf": "-Infinity"}.get(s, s)


def _kernel_json(result, G):
    """'"kernel":...,"kernel_used":[...],' for the correlated kernels; nothing for the component kernel, whose files
    stay those of a run without the choice."""
    kernel = result.get("kernel", "component")
    if kernel == "component":
        return ""
    used = ",".join("null" if k is None else f'"{k}"' for k in result["kernel_used"][:G])
    return f'"kernel":"{kernel}","kernel_used":[{used}],'


def write_abc_smc(path, opts, result):
    """The files of an ABC-SMC run (MultiContext.abc_smc): <path>/abc_gen<t>.csv with generation t's population
    (the columns of abc.md:38-55, parental_idx = the idx of the perturbed particle, then generation, epsilon,
    weight) and <path>/abc_smc.json (per generation: epsilon, consumed and simulated draws, ESS; the status; the
    options; with the mvn or olcm kernel also the kernel and the one each generation used).  `ecdna abc
    --generations` writes the same bytes: f32 values as %.9g, f64 values as %.17g, "\n" line ends.  Returns the
    number of generations written."""
    os.makedirs(path, exist_ok=True)
    G = int(result["generations"])
    for t in range(G):
        rates, dist, cells = result["rates"][t], result["distance"][t], result["cells"][t]
        zeros = np.zeros(len(cells), dtype=np.uint64)
        eps = _g9(result["epsilon"][t])
        with open(os.path.join(path, f"abc_gen{t}.csv"), "w", newline="") as f:
            f.write(",".join(SMC_FIELDS) + "\n")
            for i, row in enumerate(abc_rows(opts, 0, rates, dist, cells, zeros)):
                row["idx"] = int(result["idx"][t][i])
                if t > 0:
                    row["parental_idx"] = int(result["parent_idx"][t][i])
                f.write(",".join(_cell(row[k]) for k in ABC_FIELDS) + f",{t},{eps},{_g17(result['weight'][t][i])}\n")
    o = result["options"]

    def arr(xs, fmt):
        return "[" + ",".join(_json_float(fmt(x)) for x in xs) + "]"

    opts_json = (f'{{"seed":{o["seed"]},"idx_begin":{o["idx_begin"]},"population":{o["population"]},'
                 f'"quantile":{_g17(o["quantile"])},"max_generations":{o["max_generations"]},'
                 f'"max_simulations":{o["max_simulations"]},"b1_range":{arr(o["b1_range"], _g9)},'
                 f'"d0_range":{arr(o["d0_range"], _g9)},"d1_range":{arr(o["d1_range"], _g9)},'
                 f'"thresholds":{arr(o["thresholds"], _g9)}}}')
    text = (f'{{"status":"{result["status"]}","generations":{G},'
            f'"epsilon":{arr(result["epsilon"][:G], _g9)},'
            f'"consumed":[{",".join(str(int(x)) for x in result["consumed"][:G])}],'
            f'"simulated":[{",".join(str(int(x)) for x in result["simulated"][:G])}],'
            f'"ess":{arr(result["ess"][:G], _g17)},{_kernel_json(result, G)}"options":{opts_json}}}\n')
    with open(os.path.join(path, "abc_smc.json"), "w", newline="") as f:
        f.write(text)
    return G
