"""GPU: every instantiation of the scoring kernels and every shape limit the header promises, against the C oracle
run live, bit for bit (n_iso, the whole pep_scores table in the reference's order, best_sequence, best_score,
ascores, alt_sites -- test_gpu_parity.check_against_ref).

The parity suite scores two-ion-type scorers at mz_error <= 0.5 on synthetic peptides of 7..40 residues.  The
library switches code paths on things those inputs never cross: the number of ion types and mz_error > 0.5 select
the k_count_score instantiation, the peptide length and the number of retained peaks select its walk, the charge
and the neutral-loss variants the Ascore kernel class, the isoform count the selection kernel, the fragment count
the size of the score table.  The library has no counter that says which path ran, so every case below proves from
its inputs (and from the tables fetched back) that it reached both sides of the limit it is about.
"""
import numpy as np
import pytest

import _golden
import _limits
from pyascore_b200 import synth
from test_gpu_parity import check_against_ref, make_scorer

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------------------------------------- (a) variant matrix
# (the host-side check that VARIANTS covers all eight instantiations is tests/test_oracle_limits.py::
# test_variant_matrix_covers_every_instantiation, which runs without a GPU)
VARIANTS, NLS = _limits.VARIANTS, _limits.NLS


@pytest.mark.parametrize("q", range(len(VARIANTS)), ids=["%s-%g-nl%d" % (f, e, len(nl)) for f, e, nl in VARIANTS])
def test_variant_matrix(q):
    """a few hundred synthetic PSMs (7..20 residues, charges 1..2) per scorer set-up"""
    ftypes, err, nl = VARIANTS[q]
    w = dict(synth.WORKLOADS["lowres_phospho"], L=(7, 20), neutral_losses=nl,
             scorer=dict(_limits.PHOS, fragment_types=ftypes, mz_error=err))
    batch = synth.make_batch(w, 160, seed=2026, chunk_index=q)
    meta = dict(scorer=w["scorer"], neutral_losses=nl)
    s = make_scorer(meta)
    check_against_ref(s, batch, _golden.oracle_ref(meta, batch))
    s.close()


def test_fifth_loss_mass_is_refused():
    """PA_MAX_NL_MASSES = 4 distinct masses: a fifth is refused and leaves the scorer as it was"""
    from pyascore_b200 import Scorer
    s = Scorer(**_limits.PHOS)
    for g, m in NLS[2]:
        s.add_neutral_loss(g, m)
    s.add_neutral_loss("N", 17.026549)                 # a mass already configured is no new one
    with pytest.raises(ValueError):
        s.add_neutral_loss("R", 17.03)
    meta = dict(scorer=_limits.PHOS, neutral_losses=NLS[2] + [("N", 17.026549)])
    w = dict(synth.WORKLOADS["lowres_phospho"], L=(7, 20))
    batch = synth.make_batch(w, 100, seed=5, chunk_index=0)
    check_against_ref(s, batch, _golden.oracle_ref(meta, batch))
    s.close()


# ---------------------------------------------------------------------------------------------- (b) shape limits
GROUPS = {"length": _limits.length_group, "length_nl": lambda: _limits.length_group([("st", 97.9769)]),
          "sites": _limits.sites_group, "peaks_50": lambda: _limits.peaks_group(50.),
          "peaks_10": lambda: _limits.peaks_group(10.), "peaks_7.3": lambda: _limits.peaks_group(7.3),
          "charge": _limits.charge_group, "charge_nl": lambda: _limits.charge_group([("ST", 18.01528)]),
          "fragments": _limits.frag_group, "fragments_nl": _limits.frag_group_nl,
          "isoforms": _limits.isoform_group, "dense": _limits.dense_group}


def both_sides(values, limit):
    """some value <= limit and some value > limit"""
    values = list(values)
    return min(values) <= limit < max(values)


def prove_reached(name, g, ref, retained, n_bins):
    """host-side proof that group `name` scored both sides of its limits (from the inputs and the oracle's tables,
    which the GPU results were just found equal to)"""
    info = g.info
    L = [x["L"] for x in info]
    S = [x["S"] for x in info]
    Z = [x["Z"] for x in info]
    amb = [x["k"] < x["S"] for x in info]
    off = ref["iso_off"]
    tot = [ref["iso_total"][off[i]:off[i + 1]] for i in range(len(info))]
    best = [int(ref["iso_sig"][off[i]]) if off[i + 1] > off[i] else 0 for i in range(len(info))]
    sc = g.meta["scorer"]
    if name.startswith("length"):
        # pa_walk_fast takes 2 <= L <= 64 when the peaks are staged (<= PA_RCAP): every spectrum here is staged, so
        # the length alone decides; 1, 2..64 and 65..126 all occur, and past residue 64 the best isoform carries a mod
        assert max(retained) <= _limits.RCAP
        assert 1 in L and both_sides([x for x in L if x >= 2], _limits.LMAX_FAST) and max(L) == _limits.MAX_PEPTIDE
        for i, x in enumerate(info):
            if x["L"] > _limits.LMAX_FAST and amb[i]:
                pos = [j for j, c in enumerate(g.psms[i]["peptide"]) if c in sc["mod_group"]]
                assert any(pos[j] >= 64 for j in range(len(pos)) if (best[i] >> j) & 1), (i, bin(best[i]))
    elif name == "sites":
        # site indices >= 32 in the best signature and among the alternative sites
        assert both_sides(S, 32) and max(S) == _limits.MAX_SITES
        assert all(best[i] >> 32 for i in range(len(info)) if S[i] >= 33)
        alt_idx = []
        for i, x in enumerate(info):
            pos = [j for j, c in enumerate(g.psms[i]["peptide"]) if c in sc["mod_group"]]
            for j in range(x["k"]):
                alt_idx += [pos.index(int(r) - 1) for r in _golden.ref_alt(ref, i, j)]    # 1-based residues -> sites
        assert max(alt_idx) >= 32
    elif name.startswith("peaks"):
        # staged (<= 255 retained) and global peaks (> 255) in K2.  K1's row form runs on calls of at least 256
        # spectra (the batch is padded to that) and takes spectra of at most 128 bins; 7.3-Th bins over 1500 Th are
        # more and go to k_bin_topn
        assert list(retained) == [x["retained"] for x in info]
        assert both_sides(retained, _limits.RCAP)
        if sc["bin_size"] == 7.3:
            assert min(n_bins) > _limits.ROW_MAX_BINS
        else:
            assert max(n_bins) <= _limits.ROW_MAX_BINS
    elif name.startswith("charge"):
        # K3b classes by streams (V neutral-loss variants x Z charges): 1, 2, <= 4, <= 12; more goes to K3c, and so
        # do lists longer than PA_LCAP.  One-residue PSMs are scored too (they have one site, so no Ascore work)
        zs = [Z[i] for i in range(len(info)) if amb[i]]
        if not g.meta["neutral_losses"]:
            assert {1, 2} <= set(zs) and {3, 4} & set(zs) and {5, 12} <= set(zs) and max(zs) > _limits.MAXSTREAM
        else:
            assert both_sides(zs, _limits.MAXSTREAM // 3)
        n_types = len(sc["fragment_types"])
        assert max(int(t.max()) // n_types for t, a in zip(tot, amb) if a) > _limits.LCAP
        assert 1 in L
    elif name.startswith("fragments") or name == "dense":
        for i, x in enumerate(info):
            assert np.all(tot[i] == x["n_frag"]), (i, tot[i], x["n_frag"])
        n = sorted(x["n_frag"] for x in info)
        if name == "fragments":
            assert n == [511, 512, 513, 1024, 1025, 2048, _limits.MAX_FRAGMENTS]
        elif name == "fragments_nl":
            assert n == [2048, 2049]
        else:
            # counts near the 12-bit fields K2 packs them in
            assert ref["iso_counts"][:, -1].max() > 3000 and max(retained) > 2000
    elif name == "isoforms":
        I = [int(x) for x in ref["n_iso"][:len(info)]]
        for lim in (_limits.SORTCAP, _limits.SEL_THREAD_MAX, _limits.UNIT):
            assert both_sides(I, lim) and any(lim // 2 < i <= lim for i in I), (lim, I)
        assert max(I) > 2 * _limits.UNIT - 100 and min(Z) >= 3
        # the std::sort replay runs only when the top weighted score is shared (and I > 16): tied PSMs on both sides
        # of PA_SORTCAP (shared against global sort arena) and of PA_SEL_THREAD_MAX
        w = ref["iso_weighted"]
        tied = [I[i] for i in range(len(info)) if np.sum(w[off[i]:off[i + 1]] == w[off[i]]) > 1]
        assert both_sides(tied, _limits.SORTCAP) and both_sides(tied, _limits.SEL_THREAD_MAX) and min(tied) > 16, tied


@pytest.mark.parametrize("name", list(GROUPS))
def test_shape_limits(name):
    from oracle.cscorer import OraclePyAscore
    g = GROUPS[name]()
    batch = g.batch()
    if name.startswith("peaks"):
        # K1's row form only runs on calls of at least 256 spectra (PA_ROWS_MIN_SPECTRA): ordinary synthetic PSMs of
        # the same scorer fill the call up, behind the limit PSMs
        w = dict(synth.WORKLOADS["lowres_phospho"], L=(7, 20), scorer=g.meta["scorer"])
        batch = synth.concat_batches([batch, synth.make_batch(w, 300, seed=256, chunk_index=0)])
        assert batch["spec_off"].size - 1 >= 256
    s = make_scorer(g.meta)
    ref = _golden.oracle_ref(g.meta, batch)
    check_against_ref(s, batch, ref)
    if name.startswith("peaks"):
        assert s.counters()["launches_bin"] == 2          # k_bin_rows + k_bin_topn over the spectra it declined
    # retained peaks per spectrum: K1's count, equal to the oracle's binning
    _, _, retained = s.bin_spectra(batch["spec_off"], batch["mz"], batch["inten"])
    O = OraclePyAscore(**g.meta["scorer"])
    n_bins = []
    for q in range(len(g.info)):
        a, b = batch["spec_off"][q], batch["spec_off"][q + 1]
        bo = O.binned(batch["mz"][a:b], batch["inten"][a:b])
        assert bo["bin"].size == retained[q]
        n_bins.append(bo["n_bins"])
    prove_reached(name, g, ref, list(retained[:len(g.info)]), n_bins)
    s.close()


def test_refused_shapes():
    """one past every per-PSM limit gets its status, next to the largest accepted shape (scored and checked)"""
    g = _limits.status_group()
    batch = g.batch()
    s = make_scorer(g.meta)
    res = s.score_batch(batch)
    want = [x["status"] for x in g.info]
    assert list(res["psm_status"]) == want
    assert set(want) == {0, 2, 3, 4, 8}
    ok = [i for i, st in enumerate(want) if st == 0]
    acc = _limits.Group("accepted", g.meta["scorer"])
    for i in ok:
        p = g.psms[i]
        acc.add(p["peptide"], p["n_mod"], p["max_charge"], p["mz"], p["inten"])
    b2 = acc.batch()
    check_against_ref(s, b2, _golden.oracle_ref(g.meta, b2))
    assert max(x["L"] for x in acc.info) == _limits.MAX_PEPTIDE and max(x["S"] for x in acc.info) == _limits.MAX_SITES
    s.close()


# ---------------------------------------------------------------------------------------------- (c) growth in a batch
RESULT_KEYS = ("best_sig", "best_score", "n_iso", "n_sites", "psm_status")


def _same_results(a, b, ia, ib, ma, mb):
    for k in RESULT_KEYS:
        assert _golden.same_bits(np.asarray(a[k])[ia], np.asarray(b[k])[ib]), k
    for k in ("ascores", "alt_sites"):
        assert _golden.same_bits(np.asarray(a[k])[ma], np.asarray(b[k])[mb]), k


def test_growth_within_one_batch():
    """60 000 low-res PSMs with the limit shapes of the default scorer only at the end: the call runs in several
    chunks on two streams, and in the last one the score table grows 512 -> 4095 and the tie-order lists of (S, k)
    combinations no earlier chunk had are uploaded while the other slot's chunk is in flight.  Every PSM gets what a
    fresh scorer gives it alone, and the limit PSMs what the oracle gives.  Then the same batch device-resident
    (torch CUDA tensors; such a batch runs as one chunk), on a fresh scorer that grows its table inside that call."""
    import torch
    from pyascore_b200 import Scorer
    extra = _limits.Group("limits", _limits.PHOS)
    for g in (_limits.length_group(), _limits.sites_group()):
        extra.psms += g.psms
        extra.info += g.info
    rng = np.random.default_rng(4000)
    for L, Z in ((100, 20), (126, 16)):              # 3960 and 4000 fragments per isoform
        sites = [5, 40, 80, L - 4]
        pep = _limits.peptide(rng, L, sites)
        mz, it = _limits.spectrum(rng, _limits.ions(pep, [40, 80], "by", Z))
        extra.add(pep, 2, Z, mz, it)
    xb = extra.batch()
    base = synth.make_batch("lowres_phospho", 60000, seed=606, chunk_index=0)
    full = synth.concat_batches([base, xb])
    n0, n = base["n_mod"].size, full["n_mod"].size
    s = Scorer(**_limits.PHOS)
    res = s.score_batch(full)
    chunks = s.counters()["n_chunks"]
    assert chunks >= 3, chunks
    # what the score table needs: the synthetic PSMs stay within its first size (512 trials), the limit PSMs need
    # nearly all of it ((L - 1) x Z x 2 ion types fragments per isoform)
    frag = np.diff(full["pep_off"]).clip(min=2) - 1
    frag = frag * full["max_charge"] * 2
    assert frag[:n0].max() <= 512 and frag[n0:].max() > 2048
    # host chunks hold max(16 384, n / 8) PSMs (PA_CHUNK_MIN, pa_lib.cu): the last one starts well before the
    # limit PSMs, so every earlier chunk ran with the small table
    assert n - n0 < n - (chunks - 1) * 16384
    mo = full["mod_off"]
    alone = Scorer(**_limits.PHOS)
    r_x = check_against_ref(alone, xb, _golden.oracle_ref(dict(scorer=_limits.PHOS, neutral_losses=[]), xb))
    _same_results(res, r_x, slice(n0, n), slice(0, n - n0), slice(mo[n0], mo[n]), slice(0, None))
    r_b = Scorer(**_limits.PHOS).score_batch(base)
    _same_results(res, r_b, slice(0, n0), slice(0, n0), slice(0, mo[n0]), slice(0, None))
    dev = {k: torch.from_numpy(v.view(np.int32) if v.dtype == np.uint32 else v).cuda() for k, v in full.items()}
    s2 = Scorer(**_limits.PHOS)
    rd = s2.score_batch(dev)
    torch.cuda.synchronize()
    rd = {k: v.cpu().numpy() for k, v in rd.items()}
    for k in RESULT_KEYS + ("ascores", "alt_sites"):
        assert rd[k].tobytes() == res[k].tobytes(), k
    for x in (s, s2, alone):
        x.close()


# ---------------------------------------------------------------------------------------------- (d) K0 to its limit
def test_tail_table_to_the_limit():
    """K0: score-table rows up to n = 4095 (PA_MAX_FRAGMENTS), bit for bit against the oracle, on a scorer that grows
    600 -> 1500 -> 4095 (rows built before a growth must survive it) and on a fresh one built at 4095 at once"""
    import ctypes as C
    from oracle.cscorer import lib
    from pyascore_b200 import Scorer
    grown = Scorer(**_limits.PHOS)
    t600 = grown.tail_table(600)
    t1500 = grown.tail_table(1500)
    T = grown.tail_table(4095)
    assert _golden.same_bits(T[:t600.shape[0]], t600) and _golden.same_bits(T[:t1500.shape[0]], t1500)
    del t600, t1500
    fresh = Scorer(**_limits.PHOS)
    assert _golden.same_bits(fresh.tail_table(4095), T)
    fresh.close()
    L = lib("orc_")._dll
    L.orc_new.restype = C.c_void_p
    L.orc_new.argtypes = [C.c_float, C.c_size_t, C.c_char_p, C.c_float, C.c_float, C.c_char_p]
    L.orc_depth_score.restype = C.c_float
    L.orc_depth_score.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t]
    L.orc_free.argtypes = [C.c_void_p]
    h = L.orc_new(100., 10, b"STY", 79.966331, 0.5, b"by")
    rng = np.random.default_rng(4095)
    rows = sorted(set([0, 1, 511, 512, 513, 600, 1023, 1024, 1025, 1500, 2047, 2048, 2049, 4094, 4095]
                      + rng.integers(601, 4095, 8).tolist()))
    bad = []
    for n in rows:
        for d in range(10):
            ref = np.array([L.orc_depth_score(h, d, k, n) for k in range(n + 1)], np.float32)
            got = T[n * (n + 1) // 2:n * (n + 1) // 2 + n + 1, d]
            if ref.tobytes() != got.tobytes():
                bad.append((n, d, int(np.argmax(ref != got))))
    L.orc_free(h)
    grown.close()
    assert not bad, "%d rows differ from the oracle, first: %r" % (len(bad), bad[:5])
