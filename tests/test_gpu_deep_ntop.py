"""Scoring at peak depths n_top = 11 .. 64 (include/pyascore_b200.h, PA_N_TOP / PA_MAX_N_TOP).

In the reference, n_top > 10 keeps n_top peaks per bin, adds count / score columns for the depths 10 .. n_top-1 to
pep_scores and lets calculateAmbiguity pick the depth with the largest score difference among all n_top depths
(cpp/Ascore.cpp:165-175), so an Ascore can be computed at a depth >= 10.  The weights still have ten entries: PepScores,
isoform order, best_sequence and the alternative sites are those of n_top = 10.

GPU tests (marker gpu) compare the library with the C oracle run live at the same n_top, bit for bit: statuses, n_iso,
best_sequence, best_score, Ascores, alternative sites and the whole n_top-wide pep_scores tables.  Each case also proves
from the oracle's own tables that it reached an Ascore taken at a depth >= 10 (one that differs from the n_top = 10
oracle's).  The CPU tests check the argument envelope and the oracle's n_top > 10 tables against its n_top = 10 ones.
"""
import ctypes as C

import numpy as np
import pytest

import _golden
import _limits
from pyascore_b200 import synth

gpu = pytest.mark.gpu

SWEEP = (11, 12, 20, 31, 32, 40, 64)     # 31 / 32 straddle k_bin_rows' n_top <= 31; from 20 on spectra pass PA_RCAP peaks
SWEEP_PSMS = 1200


def _meta(workload, n_top, **kw):
    w = synth.WORKLOADS[workload]
    return dict(scorer=dict(w["scorer"], n_top=n_top, **kw), neutral_losses=w["neutral_losses"])


def _at(meta, n_top):
    return dict(meta, scorer=dict(meta["scorer"], n_top=n_top))


def _argmax_depth(sa, sb):
    """calculateAmbiguity's depth (cpp/Ascore.cpp:165-175): the first strict maximum of sa - sb, starting from 0"""
    best, depth = np.float32(0), 0
    for d in range(sa.size):
        diff = np.float32(sa[d]) - np.float32(sb[d])
        if diff > best:
            best, depth = diff, d
    return depth


def deep_reach(meta, batch, ref):
    """Ascore entries of `ref` (the oracle at meta's n_top) that differ from the n_top = 10 oracle's and belong to a
    PSM in which the best isoform and some other isoform have their largest score difference at a depth >= 10.  An
    Ascore can only change with n_top through that depth, so a non-empty list shows the case scored at depth >= 10."""
    ref10 = _golden.oracle_ref(_at(meta, 10), batch)
    a, b = ref["ascores"], ref10["ascores"]
    moved = np.flatnonzero((a.view(np.uint32) != b.view(np.uint32)) & ~(np.isnan(a) & np.isnan(b)))
    out = []
    for q in moved:
        i = int(np.searchsorted(ref["mod_off"], q, "right") - 1)
        lo, hi = int(ref["iso_off"][i]), int(ref["iso_off"][i + 1])
        sc = ref["iso_scores"][lo:hi]
        depths = [_argmax_depth(sc[0], sc[r]) for r in range(1, hi - lo)]
        if depths and max(depths) >= 10:
            out.append((int(q), i, max(depths)))
    return out


def _check(meta, batch, ref=None, nan_cells=False):
    """the library at meta's scorer against the oracle, then the depth >= 10 proof"""
    from test_gpu_parity import check_against_ref, make_scorer
    if ref is None:
        ref = _golden.oracle_ref(meta, batch)
    s = make_scorer(meta)
    assert s.n_top == meta["scorer"]["n_top"]
    if nan_cells:
        check_nan_tables(s, batch, ref)
    else:
        check_against_ref(s, batch, ref)
        assert ref["iso_counts"].shape[1] == meta["scorer"]["n_top"]
    c = s.counters()
    assert c["launches_deep"] == c["n_chunks"] and c["ms_deep"] > 0
    s.close()
    reach = deep_reach(meta, batch, ref)
    assert reach, "no Ascore of this case was taken at a depth >= 10"
    return ref, reach


def check_nan_tables(s, batch, ref):
    """check_against_ref where deep score cells may be NaN (p_d >= 1): NaN exactly where the oracle has NaN (its bit
    pattern is not compared), every other cell and every other field bit for bit"""
    from pyascore_b200 import format_results
    res = s.score_batch(batch, keep_isoforms=True)
    assert np.all(res["psm_status"] == 0) and np.array_equal(res["n_iso"], ref["n_iso"])
    n_nan = 0
    for i in range(batch["n_mod"].size):
        seq, best, asc, alts = format_results(s, batch, res, i)
        k, mo = int(batch["n_mod"][i]), int(ref["mod_off"][i])
        assert seq == ref["best_sequence"][i]
        assert _golden.same_bits(np.float32(best), np.float32(ref["best_score"][i]))
        assert _golden.same_bits(asc, ref["ascores"][mo:mo + k])
        for j in range(k):
            assert _golden.same_bits(alts[j], _golden.ref_alt(ref, i, j))
        a, b = int(ref["iso_off"][i]), int(ref["iso_off"][i + 1])
        sig, cnt, sc, w, tot = s.fetch_pep_scores(i)
        assert _golden.same_bits(sig, ref["iso_sig"][a:b]) and _golden.same_bits(cnt, ref["iso_counts"][a:b])
        assert _golden.same_bits(w, ref["iso_weighted"][a:b]) and np.array_equal(tot, ref["iso_total"][a:b])
        rs = ref["iso_scores"][a:b]
        nan = np.isnan(rs)
        assert np.array_equal(np.isnan(sc), nan)
        assert _golden.same_bits(np.where(nan, 0, sc).astype(np.float32), np.where(nan, 0, rs).astype(np.float32))
        n_nan += int(nan.sum())
    return n_nan


# ------------------------------------------------------------------------------------------------------ CPU: envelope
def test_n_top_envelope_without_gpu():
    """n_top 10 .. 64 passes the argument check (without a GPU the CUDA error follows); 9 and 65 are refused first"""
    import torch
    from pyascore_b200 import PyAscore, _lib
    assert (_lib.PA_N_TOP, _lib.PA_MAX_N_TOP) == (10, 64)
    for bad in (9, 65):
        with pytest.raises(ValueError, match="n_top"):
            PyAscore(100., bad, "STY", 79.966331)
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present: test_n_top_envelope covers it")
    for ok in (12, 64):
        with pytest.raises(RuntimeError, match="no CPU path|CUDA"):
            PyAscore(100., ok, "STY", 79.966331)


@pytest.mark.parametrize("n_top", SWEEP)
def test_oracle_deep_tables_extend_n_top_10(n_top):
    """the oracle at n_top = N against itself at 10: same isoforms, order, first ten count / score columns, PepScores,
    best sequences and alternative sites; cumulative counts non-decreasing in depth and at most total_fragments"""
    meta = _meta("lowres_phospho", n_top)
    batch = synth.make_batch("lowres_phospho", 150, seed=31, chunk_index=n_top)
    ref, ref10 = _golden.oracle_ref(meta, batch), _golden.oracle_ref(_at(meta, 10), batch)
    assert ref["iso_counts"].shape[1] == n_top and ref["iso_scores"].shape[1] == n_top
    for k in ("iso_sig", "iso_weighted", "iso_total", "n_iso", "best_score", "alt_off", "alt"):
        assert _golden.same_bits(ref[k], ref10[k]), k
    assert ref["best_sequence"] == ref10["best_sequence"]
    assert _golden.same_bits(np.ascontiguousarray(ref["iso_counts"][:, :10]), ref10["iso_counts"])
    assert _golden.same_bits(np.ascontiguousarray(ref["iso_scores"][:, :10]), ref10["iso_scores"])
    cnt = ref["iso_counts"]
    assert np.all(np.diff(cnt, axis=1) >= 0)
    assert np.all(cnt[:, -1] <= ref["iso_total"])


# ------------------------------------------------------------------------------------------------------ GPU
@gpu
def test_n_top_envelope():
    from pyascore_b200 import PyAscore, Scorer
    for bad in (9, 65):
        with pytest.raises(ValueError, match="n_top"):
            PyAscore(100., bad, "STY", 79.966331)
    s = Scorer(100., 64, "STY", 79.966331)
    assert s.n_top == 64
    s.close()


@gpu
@pytest.mark.parametrize("n_top", SWEEP)
def test_n_top_sweep(n_top):
    """lowres_phospho at every n_top of the sweep"""
    batch = synth.make_batch("lowres_phospho", SWEEP_PSMS, seed=1010, chunk_index=n_top)
    _check(_meta("lowres_phospho", n_top), batch)


@gpu
@pytest.mark.parametrize("workload", ["hires_phospho_nl", "acetyl_k"])
@pytest.mark.parametrize("n_top", [12, 40])
def test_other_workloads(workload, n_top):
    """neutral losses (the stream form of K3b) and acetyl-K with a fixed mod and three hits per spectrum"""
    batch = synth.make_batch(workload, 2000, seed=2020, chunk_index=n_top)
    _check(_meta(workload, n_top), batch)


@gpu
def test_large_and_multi_charge():
    """n_top = 20: stress-shaped PSMs (C(20, 5) isoforms: several K2 / K2d units per PSM), PSMs of charges up to 39
    (K3b's stream classes and K3c), and ordinary low-res PSMs"""
    meta = _meta("lowres_phospho", 20)
    stress = synth.make_batch(dict(synth.WORKLOADS["stress"], scorer=meta["scorer"]), 4, seed=44, chunk_index=0)
    g = _limits.charge_group()
    filler = synth.make_batch("lowres_phospho", 400, seed=45, chunk_index=0)
    batch = synth.concat_batches([stress, g.batch(), filler])
    ref, _ = _check(meta, batch)
    assert ref["n_iso"][:4].min() > 1024
    assert int(batch["max_charge"].max()) >= 13


@gpu
def test_batch_layouts():
    """a host batch of 48 000 PSMs at n_top = 20 runs in several chunks, and its last PSMs need a larger score table
    (T and T_deep grow between chunks); the same batch device-resident gives the same results everywhere, and the
    first and last PSMs equal the oracle"""
    import torch
    from pyascore_b200 import Scorer
    from test_gpu_parity import check_against_ref
    meta = _meta("lowres_phospho", 20)
    rng = np.random.default_rng(4000)
    extra = _limits.Group("limits", meta["scorer"])
    for L, Z in ((100, 20), (126, 16)):             # 3960 and 4000 fragments per isoform
        sites = [5, 40, 80, L - 4]
        pep = _limits.peptide(rng, L, sites)
        mz, it = _limits.spectrum(rng, _limits.ions(pep, [40, 80], "by", Z))
        extra.add(pep, 2, Z, mz, it)
    base = synth.make_batch("lowres_phospho", 48000, seed=4848, chunk_index=0)
    full = synth.concat_batches([base, extra.batch()])
    n = full["n_mod"].size
    s = Scorer(**meta["scorer"])
    res = s.score_batch(full)
    c = s.counters()
    assert c["n_chunks"] >= 3 and c["launches_deep"] == c["n_chunks"], c
    dev = {k: torch.from_numpy(v.view(np.int32) if v.dtype == np.uint32 else v).cuda() for k, v in full.items()}
    rd = Scorer(**meta["scorer"]).score_batch(dev)
    torch.cuda.synchronize()
    for k in ("best_sig", "best_score", "n_iso", "n_sites", "psm_status", "ascores", "alt_sites"):
        assert rd[k].cpu().numpy().tobytes() == res[k].tobytes(), k
    from pyascore_b200.shard import take_shard
    mo = full["mod_off"]
    for p0, p1 in ((0, 600), (n - 600, n)):
        part = take_shard(full, p0, p1)
        alone = Scorer(**meta["scorer"])
        r = check_against_ref(alone, part, _golden.oracle_ref(meta, part))
        for k in ("best_sig", "best_score", "n_iso", "psm_status"):
            assert _golden.same_bits(res[k][p0:p1], r[k]), k
        for k in ("ascores", "alt_sites"):
            assert _golden.same_bits(res[k][mo[p0]:mo[p1]], r[k]), k
        alone.close()
    s.close()


def _oracle_table(n_top, err=0.5):
    from oracle.cscorer import lib
    L = lib("orc_")._dll
    L.orc_new.restype = C.c_void_p
    L.orc_new.argtypes = [C.c_float, C.c_size_t, C.c_char_p, C.c_float, C.c_float, C.c_char_p]
    L.orc_depth_score.restype = C.c_float
    L.orc_depth_score.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t]
    L.orc_free.argtypes = [C.c_void_p]
    return L, L.orc_new(100., n_top, b"STY", 79.966331, err, b"by")


def _table_rows_differ(L, h, T, rows, n_top):
    bad = []
    for n in rows:
        for d in range(n_top):
            ref = np.array([L.orc_depth_score(h, d, k, n) for k in range(n + 1)], np.float32)
            got = T[n * (n + 1) // 2:n * (n + 1) // 2 + n + 1, d]
            if ref.tobytes() != got.tobytes():
                bad.append((n, d, int(np.argmax(ref.view(np.uint32) != got.view(np.uint32)))))
    return bad


@gpu
def test_tail_table_deep():
    """K0 at n_top = 64: every depth of rows up to n = 700 against orc_depth_score, then up to n = 4095 on a sample of
    rows, on a scorer that grows 700 -> 1500 -> 4095 and on one built at 4095 at once"""
    from pyascore_b200 import Scorer
    L, h = _oracle_table(64)
    grown = Scorer(100., 64, "STY", 79.966331, 0.5, "by")
    t700 = grown.tail_table(700)
    assert t700.shape == (701 * 702 // 2, 64)
    rng = np.random.default_rng(64)
    rows = sorted(set([0, 1, 2, 3, 10, 34, 68, 136, 312, 511, 512, 513, 700] + rng.integers(1, 700, 30).tolist()))
    bad = _table_rows_differ(L, h, t700, rows, 64)
    assert not bad, "%d (row, depth) differ, first: %r" % (len(bad), bad[:5])
    t1500 = grown.tail_table(1500)
    assert _golden.same_bits(t1500[:t700.shape[0]], t700)
    del t700
    T = grown.tail_table(4095)
    assert _golden.same_bits(T[:t1500.shape[0]], t1500)
    del t1500
    grown.close()
    rows = sorted(set([1023, 1024, 1025, 2047, 2048, 2049, 4094, 4095] + rng.integers(701, 4095, 4).tolist()))
    bad = _table_rows_differ(L, h, T, rows, 64)
    assert not bad, "%d (row, depth) differ, first: %r" % (len(bad), bad[:5])
    fresh = Scorer(100., 64, "STY", 79.966331, 0.5, "by")
    assert _golden.same_bits(fresh.tail_table(4095), T)
    fresh.close()
    L.orc_free(h)


@gpu
def test_calculate_ambiguity_at_deep_depths():
    """pa_calculate_ambiguity with n_top-wide score rows equals the oracle's calculate_ambiguity on isoform pairs
    whose largest score difference is at a depth >= 10"""
    from oracle.cscorer import OraclePyAscore
    from pyascore_b200 import Scorer
    from pyascore_b200.shard import take_shard
    meta = _meta("lowres_phospho", 40)
    batch = synth.make_batch("lowres_phospho", 400, seed=4040, chunk_index=0)
    ref = _golden.oracle_ref(meta, batch)
    s = Scorer(**meta["scorer"])
    O = OraclePyAscore(**meta["scorer"])
    n_pairs = 0
    for i in range(batch["n_mod"].size):
        lo, hi = int(ref["iso_off"][i]), int(ref["iso_off"][i + 1])
        sc = ref["iso_scores"][lo:hi]
        pairs = [r for r in range(1, hi - lo) if _argmax_depth(sc[0], sc[r]) >= 10][:3]
        if not pairs:
            continue
        s.score_batch(take_shard(batch, i, i + 1), keep_isoforms=True)
        sig, cnt, gsc, w, tot = s.fetch_pep_scores(0)
        O.score(*synth.psm_view(batch, i))
        ops = O.pep_scores
        for r in pairs:
            got = s.calculate_ambiguity(0, int(sig[0]), gsc[0], w[0], int(sig[r]), gsc[r], w[r])
            want = O.calculate_ambiguity(ops[0], ops[r])
            assert np.float32(got).tobytes() == np.float32(want).tobytes(), (i, r, got, want)
            n_pairs += 1
    assert n_pairs >= 20, n_pairs
    with pytest.raises(ValueError, match="n_top"):
        s.calculate_ambiguity(0, int(sig[0]), gsc[0][:10], w[0], int(sig[1]), gsc[1][:10], w[1])
    s.close()


@gpu
def test_pyascore_drop_in_n_top_12():
    """PyAscore(n_top=12) on the reference's 31 fixture PSMs: pep_scores rows carry 12 counts and scores, the
    invariants of the reference's test/test_ascore.py hold, and everything equals the oracle at n_top = 12"""
    import math
    import re
    from oracle.cscorer import OraclePyAscore
    from pyascore_b200 import PyAscore
    meta, batch, _ = _golden.load("fixtures_by_05")
    kw = dict(meta["scorer"], n_top=12)
    for i in range(batch["n_mod"].size):
        mz, inten, pep, n_mod, z, aux_pos, aux_mass = synth.psm_view(batch, i)
        a = PyAscore(**kw)
        a.score(np.ascontiguousarray(mz), np.ascontiguousarray(inten), pep, n_mod, z,
                np.ascontiguousarray(aux_pos, np.uint32), np.ascontiguousarray(aux_mass, np.float32))
        O = OraclePyAscore(**kw)
        O.score(mz, inten, pep, n_mod, z, aux_pos, aux_mass)
        ps, ops = a.pep_scores, O.pep_scores
        assert len(ps) == math.comb(len(ps[0]["signature"]), n_mod) == len(ops)
        assert np.all(np.diff([p["weighted_score"] for p in ps]) <= 0)
        for p, q in zip(ps, ops):
            assert p["counts"].shape == (12,) and p["scores"].shape == (12,)
            assert np.array_equal(p["counts"], q["counts"]) and p["scores"].tobytes() == q["scores"].tobytes()
            assert np.array_equal(p["signature"], q["signature"]) and p["sequence"] == q["sequence"]
        assert a.best_sequence == O.best_sequence
        assert np.float32(a.best_score).tobytes() == np.float32(O.best_score).tobytes()
        assert np.asarray(a.ascores, np.float32).tobytes() == O.ascores.tobytes()
        for alt in a.alt_sites:
            assert alt.shape[0] == np.unique(alt).shape[0]
        modified = [ind + 1 for ind, m in enumerate(re.finditer("[A-Z][^A-Z]*", a.best_sequence)) if "[80]" in m.group()]
        alts = np.concatenate(a.alt_sites) if len(a.alt_sites) else np.zeros(0, np.uint32)
        assert np.intersect1d(modified, alts).shape[0] == 0
        assert a.calculate_ambiguity(ps[0], ps[0]) == 0.
        if len(ps) > 1:
            got = a.calculate_ambiguity(ps[0], ps[1])
            assert np.float32(got).tobytes() == np.float32(O.calculate_ambiguity(ops[0], ops[1])).tobytes()


@gpu
def test_nan_region():
    """mz_error = 1.5 at n_top = 40: p_d = 2 * 1.5 * d / 100 >= 1 from d = 34 on, where log(1 - p_d) is NaN or -inf and
    the reference's deep scores are NaN.  Those cells are NaN here too, and the depth argmax never picks them"""
    meta = _meta("lowres_phospho", 40, mz_error=1.5)
    batch = synth.make_batch(dict(synth.WORKLOADS["lowres_phospho"], scorer=meta["scorer"]), 600, seed=1515, chunk_index=0)
    ref = _golden.oracle_ref(meta, batch)
    nan = np.isnan(ref["iso_scores"])
    assert nan[:, 33:].any() and not nan[:, :33].any()
    _check(meta, batch, ref, nan_cells=True)
