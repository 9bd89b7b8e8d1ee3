"""Two modification types in one call (score_typed) against one call per type, by the wall clock around the public calls.

    python tools/typed_rates.py [--psms 1000000] [--reps 5] [--parent DIR] [--bench-reps 2] [--out FILE]

Workload: config 2 (lowres_phospho, bench.py's seed), `--psms` phospho PSMs plus, for every PSM whose peptide has a K, an
acetyl-K row (mass 42.010565) on the same spectrum, as one float64 host batch in pinned memory.
  typed:    score_typed([phospho, acetyl], batch, psm_type) -- the spectra cross the host link and are binned once;
  separate: phospho.score_batch(phospho rows) + acetyl.score_batch(acetyl rows), each batch carrying the full spectra.
Both forms use the same two scorers, are warmed up (which also settles the library's m/z narrowing decision), then
alternate `--reps` times; the results of the two forms are checked bit-identical.  With --parent (a checkout of the
parent commit with its library built), `python bench.py` -- the default line -- of the parent tree and of this tree
alternate `--bench-reps` times in the same run, to show that the single-type numbers stay within their spread.  The
GPU's name and power limit are read in the same run.  Writes one JSON file (--out).  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RESULTS = ("best_sig", "best_score", "n_iso", "n_sites", "ascores", "alt_sites", "psm_status")
COUNTERS = ("n_chunks", "bytes_h2d", "bytes_d2h", "n_peaks", "launches_bin", "launches_count", "n_spec_exact",
            "ms_bin", "ms_count", "ms_total", "ms_narrow_wait")


def gpu_info(index=0):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().split(",")]
        return dict(name=name, power_limit_w=float(power), sm_max_mhz=float(clock))
    except Exception as e:                                    # noqa: BLE001 -- reported, not hidden
        return dict(name=None, power_limit_w=None, error="nvidia-smi: %s" % e)


def bench_line(tree):
    r = subprocess.run([sys.executable, "bench.py"], cwd=tree, capture_output=True, text=True, timeout=1800)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        return dict(error="bench.py exited %d: %s" % (r.returncode, (r.stderr or r.stdout)[-2000:]))
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--psms", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--parent", default="", help="tree of the parent commit (library built) for the bench.py A/B")
    ap.add_argument("--bench-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "typed_rates.json"))
    args = ap.parse_args()

    from pyascore_b200 import Scorer, pin_batch, score_typed, synth
    gpu = gpu_info(0)
    base = synth.make_batch("lowres_phospho", args.psms, seed=20261017)
    batch, psm_type = synth.typed_batch(base, ["K"])
    rows = [np.flatnonzero(psm_type == t) for t in range(2)]
    batch = pin_batch(batch)
    spectra = ("spec_off", "mz", "inten")                     # one pinned copy of the spectra, shared by all batches
    per_type = []
    for r in rows:
        sub = synth.select_rows(batch, r)
        per_type.append(dict(pin_batch({k: v for k, v in sub.items() if k not in spectra}), **{k: batch[k] for k in spectra}))
    ph = Scorer(100., 10, "STY", 79.966331, 0.5, "by")
    ac = Scorer(100., 10, "K", 42.010565, 0.5, "by")

    def typed():
        t0 = time.perf_counter()
        r = score_typed([ph, ac], batch, psm_type)
        return time.perf_counter() - t0, r, ph.counters()

    def separate():
        t0 = time.perf_counter()
        r0 = ph.score_batch(per_type[0])
        c0 = ph.counters()
        r1 = ac.score_batch(per_type[1])
        return time.perf_counter() - t0, (r0, r1), (c0, ac.counters())

    for _ in range(args.warmup):
        typed()
        separate()
    t_typed, t_sep, c_typed, c_sep = [], [], None, None
    for _ in range(args.reps):
        dt, r_typed, c_typed = typed()
        t_typed.append(dt)
        dt, r_sep, c_sep = separate()
        t_sep.append(dt)
    mo = np.zeros(psm_type.size + 1, np.int64)
    np.cumsum(batch["n_mod"], out=mo[1:])
    same = True
    for t in range(2):
        idx, _ = synth._ragged(mo, rows[t])
        for k in RESULTS:
            got = r_typed[k][idx] if k in ("ascores", "alt_sites") else r_typed[k][rows[t]]
            same &= got.tobytes() == np.ascontiguousarray(r_sep[t][k]).tobytes()
    n = int(psm_type.size)
    out = dict(
        gpu=gpu, workload="lowres_phospho + acetyl-K rows (config 2 spectra), float64 host batch, pinned",
        psms_phospho=int(rows[0].size), psms_acetyl=int(rows[1].size), spectra=int(batch["spec_off"].size - 1),
        peaks=int(batch["spec_off"][-1]), results_identical=bool(same),
        typed_s=t_typed, separate_s=t_sep,
        typed_median_s=float(np.median(t_typed)), separate_median_s=float(np.median(t_sep)),
        typed_mpsm_s=n / float(np.median(t_typed)) / 1e6, separate_mpsm_s=n / float(np.median(t_sep)) / 1e6,
        speedup=float(np.median(t_sep) / np.median(t_typed)),
        counters_typed={k: c_typed[k] for k in COUNTERS},
        counters_separate=[{k: c[k] for k in COUNTERS} for c in c_sep])
    ph.close()
    ac.close()
    print(json.dumps({k: v for k, v in out.items() if not k.startswith("counters")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def save():                                              # after every step: a cut-short run keeps what it measured
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    save()
    if args.parent:
        out["bench"] = []
        for i in range(args.bench_reps):
            for which, tree in (("parent", args.parent), ("this", ROOT)):
                t0 = time.perf_counter()
                line = bench_line(tree)
                out["bench"].append(dict(tree=which, rep=i, wall_s=time.perf_counter() - t0, line=line))
                print(which, "%.0f s" % (time.perf_counter() - t0), json.dumps(line)[:400], flush=True)
                save()


if __name__ == "__main__":
    main()
