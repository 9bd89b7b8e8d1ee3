"""Generate the committed golden vectors from the UNMODIFIED reference (oracle/_ref).

Run in the build container (needs /root/reference for the pickled fixtures and oracle/_ref built
by `make -C oracle ref`):

    python tests/golden/make_golden.py

Writes tests/golden/*.npz.  Each file holds the inputs (CSR batch + scorer settings) and what the
reference returned for every PSM: best_sequence, best_score, ascores, alt_sites and the full
pep_scores table in the reference's own order.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle.cscorer import RefPyAscore  # noqa: E402
from pyascore_b200 import shard, synth  # noqa: E402
import _fixtures  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def batch_from_psms(psms):
    """psms: list of dict(mz, inten, peptide, n_mod, max_charge, aux_pos, aux_mass) -> CSR batch"""
    spec_off = [0]; pep_off = [0]; aux_off = [0]
    mz = []; inten = []; pep = []; ap = []; am = []
    for p in psms:
        mz.append(p["mz"]); inten.append(p["inten"]); spec_off.append(spec_off[-1] + p["mz"].size)
        b = np.frombuffer(p["peptide"].encode(), np.uint8); pep.append(b); pep_off.append(pep_off[-1] + b.size)
        a = p.get("aux_pos"); m = p.get("aux_mass")
        if a is None:
            a = np.zeros(0, np.uint32); m = np.zeros(0, np.float32)
        ap.append(np.asarray(a, np.uint32)); am.append(np.asarray(m, np.float32)); aux_off.append(aux_off[-1] + len(a))
    return dict(spec_off=np.array(spec_off, np.int64), mz=np.concatenate(mz), inten=np.concatenate(inten),
                psm_spec=np.arange(len(psms), dtype=np.int32), pep_off=np.array(pep_off, np.int32),
                pep=np.concatenate(pep), n_mod=np.array([p["n_mod"] for p in psms], np.int32),
                max_charge=np.array([p["max_charge"] for p in psms], np.int32), aux_off=np.array(aux_off, np.int32),
                aux_pos=np.concatenate(ap) if ap else np.zeros(0, np.uint32),
                aux_mass=np.concatenate(am) if am else np.zeros(0, np.float32))


def run_reference(scorer_kw, neutral_losses, batch, scorer_cls=RefPyAscore):
    """score every PSM of `batch` with the compiled reference (or another class with its surface, such as
    oracle.cscorer.OraclePyAscore) -> per-PSM results and the whole pep_scores table in golden layout"""
    R = scorer_cls(**scorer_kw)
    for g, m in neutral_losses:
        R.add_neutral_loss(g, m)
    n = batch["n_mod"].size
    seqs = []; best = np.zeros(n, np.float32); n_iso = np.zeros(n, np.int64); S = np.zeros(n, np.int32)
    asc = []; alt_off = [0]; alt = []
    iso_sig = []; iso_cnt = []; iso_sc = []; iso_w = []; iso_tot = []
    for i in range(n):
        a = synth.psm_view(batch, i)
        R.score(*a)
        seqs.append(R.best_sequence); best[i] = R.best_score
        sig, cnt, sc, w, tot = R.pep_score_tables()
        n_iso[i] = w.size; S[i] = sig.shape[1] if w.size else 0
        bits = np.zeros(w.size, np.uint64)
        for j in range(sig.shape[1]):
            bits |= (sig[:, j].astype(np.uint64) << np.uint64(j))
        iso_sig.append(bits); iso_cnt.append(cnt); iso_sc.append(sc); iso_w.append(w); iso_tot.append(tot)
        asc.append(R.ascores)
        for s in R.alt_sites:
            alt.append(np.asarray(s, np.uint32)); alt_off.append(alt_off[-1] + len(s))
    D = scorer_kw["n_top"]
    return dict(best_sequence=np.frombuffer("\n".join(seqs).encode(), np.uint8), best_score=best, n_iso=n_iso,
                n_sites=S, ascores=np.concatenate(asc) if asc else np.zeros(0, np.float32),
                alt_off=np.array(alt_off, np.int64), alt=np.concatenate(alt) if alt else np.zeros(0, np.uint32),
                iso_sig=np.concatenate(iso_sig), iso_counts=np.concatenate(iso_cnt).reshape(-1, D),
                iso_scores=np.concatenate(iso_sc).reshape(-1, D), iso_weighted=np.concatenate(iso_w),
                iso_total=np.concatenate(iso_tot))


def save(name, scorer_kw, neutral_losses, batch):
    ref = run_reference(scorer_kw, neutral_losses, batch)
    meta = dict(scorer=scorer_kw, neutral_losses=neutral_losses)
    arrays = {"in_" + k: v for k, v in batch.items()}
    arrays.update({"ref_" + k: v for k, v in ref.items()})
    arrays["meta"] = np.frombuffer(json.dumps(meta).encode(), np.uint8)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("%-28s psms %5d isoforms %7d  %.0f KB" % (name, batch["n_mod"].size, ref["iso_weighted"].size,
                                                     os.path.getsize(path) / 1e3))


def edge_cases():
    rng = np.random.default_rng(7)
    def spec(n=120, lo=150., hi=1400.):
        mz = np.sort(rng.uniform(lo, hi, n)); return mz, np.exp(rng.normal(5., 1., n))
    P = []
    def add(pep, k, z=1, aux_pos=None, aux_mass=None, mzint=None):
        mz, it = mzint if mzint is not None else spec()
        P.append(dict(mz=mz, inten=it, peptide=pep, n_mod=k, max_charge=z, aux_pos=aux_pos, aux_mass=aux_mass))
    add("ASAK", 1)                      # k == #sites: unambiguous
    add("ASAK", 2)                      # k > #sites: no isoform
    add("AAAK", 1)                      # no site at all
    add("ASTK", 1, 1, np.array([0, 2], np.uint32), np.array([42.010565, 10.0], np.float32),
        (np.array([5000., 5001.]), np.array([1., 2.])))   # aux on a site + N-term aux, all ties
    add("ASSSSSSK", 2, 1, None, None, (np.array([5000., 5001.]), np.array([1., 2.])))   # all ties, 15 isoforms
    add("A" + "S" * 8 + "K", 3, 2, None, None, (np.array([5000., 5001.]), np.array([1., 2.])))  # 56 tied isoforms
    add("ASTYSTYSTYK", 4, 2)            # 126 isoforms
    add("STYSTYK", 0, 1)                # zero mods
    # ("MSTK", k=1, charge 0) makes the reference dereference an empty vector (segfault): not a golden case
    add("SK", 1, 1)                     # shortest useful peptide
    add("S", 1, 1)                      # single residue
    add("KSTMC", 1, 2, np.array([5], np.uint32), np.array([57.021464], np.float32))
    add("PEPSTIDEK", 1, 3, None, None, (np.array([400.25]), np.array([10.])))   # single peak
    add("PEPSTIDEK", 2, 2, None, None, spec(900, 100., 2100.))                  # dense spectrum, > 10 per bin
    return batch_from_psms(P)


def main():
    phos = dict(bin_size=100., n_top=10, mod_group="STY", mod_mass=79.966331, mz_error=0.5, fragment_types="by")
    fx = _fixtures.load_pairs()
    def fx_batch(charge_fn):
        return batch_from_psms([dict(mz=p["mz"], inten=p["inten"], peptide=p["peptide"], n_mod=p["n_mod"],
                                     max_charge=charge_fn(p)) for p in fx])
    save("fixtures_by_05", phos, [], fx_batch(lambda p: p["charge"] - 1))
    save("fixtures_by_05_z1", phos, [], fx_batch(lambda p: 1))
    save("fixtures_by_05_nlST", phos, [("ST", 18.01528)], fx_batch(lambda p: p["charge"] - 1))
    save("fixtures_by_002_nlst", dict(phos, mz_error=0.02), [("st", 97.9769)], fx_batch(lambda p: min(2, p["charge"] - 1)))
    save("fixtures_yb_05", dict(phos, fragment_types="yb"), [], fx_batch(lambda p: p["charge"] - 1))
    save("fixtures_cZ_002_nl2", dict(phos, mz_error=0.02, fragment_types="cZ"), [("ST", 18.01528), ("st", 97.9769)],
         fx_batch(lambda p: min(2, p["charge"] - 1)))
    save("fixtures_nKc_05", dict(phos, mod_group="nKc", mod_mass=42.010565), [], fx_batch(lambda p: 1))
    save("edge_cases", phos, [], edge_cases())
    save("edge_cases_nl", dict(phos, mz_error=0.05), [("ST", 18.01528), ("st", 97.9769), ("K", 17.026549)], edge_cases())
    # (workload, PSMs generated, PSMs kept): the first `kept` PSMs keep every golden file under 1 MB
    for wl, n, kept in (("lowres_phospho", 400, 190), ("hires_phospho_nl", 300, 170), ("acetyl_k", 300, 300),
                        ("stress", 2, 2)):
        w = synth.WORKLOADS[wl]
        b = shard.take_shard(synth.make_batch(wl, n, seed=20261017, chunk_index=0), 0, kept)
        if w["hits"] > 1:   # golden files are per-PSM: expand the shared spectra
            pass
        save("synth_" + wl, w["scorer"], [list(x) for x in w["neutral_losses"]], b)


if __name__ == "__main__":
    main()
