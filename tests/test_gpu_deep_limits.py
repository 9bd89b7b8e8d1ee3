"""GPU: the n_top > 10 path (K2d k_count_deep, T_deep, the DEEP forms of K3b / K3c, K1 at deep n_top) at every
scoring-kernel variant and shape limit of tests/test_gpu_limits.py, against the C oracle run live at the same n_top, bit
for bit: statuses, n_iso, the whole n_top-wide pep_scores tables, best sequence and score, Ascores and alternative sites
(NaN deep score cells, p_d >= 1, NaN exactly where the oracle's are).

The shape groups of tests/_limits.py hold at most ten peaks per bin, which gives no rank >= 10; every case here runs on
spectra densified to 11 .. n_top peaks per bin (_limits.densify) and proves from the oracle's tables that it reached
ranks >= 10 (tests/test_oracle_deep_limits.py checks the same without a GPU)."""
import numpy as np
import pytest

import _golden
import _limits
from pyascore_b200 import synth
from test_gpu_deep_ntop import _argmax_depth, check_nan_tables, deep_reach
from test_gpu_limits import prove_reached
from test_gpu_parity import check_against_ref, make_scorer
from test_gpu_shard import _same
from test_oracle_deep_limits import deep_rank_psms, prove_deep

pytestmark = pytest.mark.gpu


def _compare(meta, batch, ref):
    """the library against `ref`; the scorer stays open for the caller"""
    s = make_scorer(meta)
    assert s.n_top == meta["scorer"]["n_top"]
    if np.isnan(ref["iso_scores"]).any():
        check_nan_tables(s, batch, ref)
    else:
        check_against_ref(s, batch, ref)
    c = s.counters()
    assert c["launches_deep"] == c["n_chunks"]
    return s


# ---------------------------------------------------------------------------------------------- (a) variant matrix
@pytest.mark.parametrize("q,n_top", _limits.DEEP_MATRIX,
                         ids=["%s-%g-nl%d-top%d" % (_limits.VARIANTS[q][0], _limits.VARIANTS[q][1],
                                                    len(_limits.VARIANTS[q][2]), t) for q, t in _limits.DEEP_MATRIX])
def test_deep_variant_matrix(q, n_top):
    """every k_count_score set-up at n_top 20 (both k_count_deep instantiations), one per instantiation at 64"""
    meta, batch = _limits.deep_variant_case(q, n_top)
    ref = _golden.oracle_ref(meta, batch)
    _compare(meta, batch, ref).close()
    assert np.mean(deep_rank_psms(ref, batch["n_mod"].size)) > 0.25


# ---------------------------------------------------------------------------------------------- (b) shape limits
@pytest.mark.parametrize("name,n_top", _limits.DEEP_SHAPES, ids=["%s-%d" % c for c in _limits.DEEP_SHAPES])
def test_deep_shape_limits(name, n_top):
    from oracle.cscorer import OraclePyAscore
    g = _limits.deep_group(name, n_top)
    batch = g.batch()
    if name == "peaks_deep":
        # K1's row form only runs on calls of at least 256 spectra (PA_ROWS_MIN_SPECTRA) and n_top <= 31
        w = dict(synth.WORKLOADS["lowres_phospho"], L=(7, 20), scorer=g.meta["scorer"])
        batch = synth.concat_batches([batch, synth.make_batch(w, 300, seed=256, chunk_index=n_top)])
    ref = _golden.oracle_ref(g.meta, batch)
    s = _compare(g.meta, batch, ref)
    if name == "peaks_deep":
        assert s.counters()["launches_bin"] == (2 if n_top <= 31 else 1)
    _, _, retained = s.bin_spectra(batch["spec_off"], batch["mz"], batch["inten"])
    s.close()
    O = OraclePyAscore(**g.meta["scorer"])
    n_bins = []
    for q in range(len(g.info)):
        a, b = batch["spec_off"][q], batch["spec_off"][q + 1]
        bo = O.binned(batch["mz"][a:b], batch["inten"][a:b])
        assert bo["bin"].size == retained[q]
        n_bins.append(bo["n_bins"])
    prove_reached(name, g, ref, list(retained[:len(g.info)]), n_bins)
    prove_deep(name, g, ref)
    if (name, n_top) not in _limits.DEEP_SHALLOW_ASCORES:
        assert deep_reach(g.meta, batch, ref)


# ---------------------------------------------------------------------------------------------- (c) ambiguity probe
def test_deep_ambiguity_probe_long_lists():
    """pa_calculate_ambiguity (k_ambiguity) at n_top 40 on the kept charge-39 PSMs with a neutral loss (K3c's shape: lists
    of 13 x 2 x 39 fragments per ion type, longer than PA_LCAP), on isoform pairs whose argmax depth is >= 10"""
    from oracle.cscorer import OraclePyAscore
    from pyascore_b200.shard import take_shard
    g = _limits.deep_group("charge_nl", 40)
    batch = g.batch()
    s = make_scorer(g.meta)
    O = OraclePyAscore(**g.meta["scorer"])
    for grp, m in g.meta["neutral_losses"]:
        O.add_neutral_loss(grp, m)
    n_pairs = 0
    for i, x in enumerate(g.info):
        if x["Z"] != 39 or x["k"] >= x["S"]:
            continue
        assert (x["L"] - 1) * 2 * x["Z"] > _limits.LCAP
        s.score_batch(take_shard(batch, i, i + 1), keep_isoforms=True)
        sig, cnt, sc, w, tot = s.fetch_pep_scores(0)
        O.score(*synth.psm_view(batch, i))
        ops = O.pep_scores
        for a in range(sig.size):
            for r in range(sig.size):
                if a == r or _argmax_depth(ops[a]["scores"], ops[r]["scores"]) < 10:
                    continue
                got = s.calculate_ambiguity(0, int(sig[a]), sc[a], w[a], int(sig[r]), sc[r], w[r])
                want = O.calculate_ambiguity(ops[a], ops[r])
                assert np.float32(got).tobytes() == np.float32(want).tobytes(), (i, a, r, got, want)
                n_pairs += 1
    assert n_pairs >= 5, n_pairs
    s.close()


# ---------------------------------------------------------------------------------------------- (d) refused shapes
def test_deep_refused_shapes():
    """at n_top 64: one past every per-PSM limit gets its status, the largest accepted shapes equal the oracle"""
    g = _limits.densify(_limits.status_group(), 64, _limits.DEEP_SEED)
    s = make_scorer(g.meta)
    res = s.score_batch(g.batch())
    want = [x["status"] for x in g.info]
    assert list(res["psm_status"]) == want and set(want) == {0, 2, 3, 4, 8}
    acc = _limits.Group("accepted", g.meta["scorer"])
    for i in [i for i, st in enumerate(want) if st == 0]:
        p = g.psms[i]
        acc.add(p["peptide"], p["n_mod"], p["max_charge"], p["mz"], p["inten"])
    b2 = acc.batch()
    ref = _golden.oracle_ref(g.meta, b2)
    check_against_ref(s, b2, ref)
    assert max(x["L"] for x in acc.info) == _limits.MAX_PEPTIDE and max(x["S"] for x in acc.info) == _limits.MAX_SITES
    assert any(deep_rank_psms(ref, len(acc.info)))
    s.close()


# ---------------------------------------------------------------------------------------------- (e) K1 at deep n_top
def _awkward(batch):
    """the spectra of test_gpu_shard.test_row_form_binning_equals_topn_kernel: ties, unsorted, NaN / negative / huge m/z,
    peaks on bin boundaries, pairs of equal m/z"""
    off, mz, inten = batch["spec_off"], batch["mz"], batch["inten"]
    rng = np.random.default_rng(5)
    seg = lambda q: slice(int(off[q]), int(off[q + 1]))
    for q in (1, 4, 11):
        sl = seg(q)
        inten[sl] = np.round(inten[sl], -1) + 10.
    v = inten[seg(2)]
    v[1::2] = v[0]
    sl = seg(6)
    perm = rng.permutation(sl.stop - sl.start)
    mz[sl], inten[sl] = mz[sl][perm], inten[sl][perm]
    mz[int(off[8]) + 3] = np.nan
    mz[int(off[9])] = -5.
    mz[int(off[14]) - 1] = 3.0e6
    sl = seg(15)
    mz[sl] = np.sort(np.where(rng.random(sl.stop - sl.start) < 0.2, np.round(mz[sl], -2), mz[sl]))
    v = mz[seg(16)]
    v[1::2] = v[::2][: v[1::2].size]
    return batch


@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("n_top", [20, 31])
def test_deep_row_form_binning_equals_topn_kernel(n_top, f32, monkeypatch):
    """k_bin_rows against k_bin_topn (PA_K1=topn) at the deep n_top the row form takes, bit for bit, float64 and float32
    intensities; the spectra hold more than n_top peaks in some bins"""
    from pyascore_b200 import Scorer
    sc = dict(synth.WORKLOADS["lowres_phospho"]["scorer"], n_top=n_top)
    batch = _awkward(synth.make_batch("lowres_phospho", 4000, seed=77, chunk_index=n_top))
    if f32:
        batch["inten32"] = batch.pop("inten").astype(np.float32)
    res = {}
    for mode in ("topn", "rows"):
        monkeypatch.setenv("PA_K1", mode)
        s = Scorer(**sc)
        res[mode] = s.score_batch(dict(batch), keep_isoforms=True)
        res[mode + "_launches"] = s.counters()["launches_bin"]
        res[mode + "_tables"] = [s.fetch_pep_scores(i)[1:3] for i in range(0, batch["n_mod"].size, 97)]
        s.close()
    assert _same(res["topn"], res["rows"])
    for (ca, sa), (cb, sb) in zip(res["topn_tables"], res["rows_tables"]):
        assert _golden.same_bits(ca, cb) and _golden.same_bits(sa, sb)
    assert res["rows_launches"] == 2 * res["topn_launches"]
    assert any(np.any(c[:, -1] > c[:, 9]) for c, _ in res["rows_tables"])          # ranks >= 10 were binned and matched


# ---------------------------------------------------------------------------------------------- (f) float32, narrowing
def test_deep_float32_and_narrowing(monkeypatch):
    """n_top 40 (k_bin_topn bins every spectrum): float32 intensities give what float64 gives, and host narrowing of m/z
    (PA_NARROW=1) what the float64 path gives, bit for bit, with peaks on and next to bin boundaries"""
    from pyascore_b200 import Scorer
    sc = dict(synth.WORKLOADS["lowres_phospho"]["scorer"], n_top=40)
    batch = synth.make_batch("lowres_phospho", 4000, seed=55, chunk_index=40)
    off, mz = batch["spec_off"], batch["mz"]
    for q, val in ((2, 700.), (5, np.nextafter(900., 0.)), (7, np.nextafter(500., 1000.))):
        a, b = int(off[q]), int(off[q + 1])
        seg = mz[a:b]
        seg[np.argmin(np.abs(seg - val))] = val
        mz[a:b] = np.sort(seg)
    b32 = {k: v for k, v in batch.items() if k != "inten"}
    b32["inten32"] = batch["inten"].astype(np.float32)
    b64 = dict(batch, inten=b32["inten32"].astype(np.float64))
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("PA_NARROW", mode)
        s = Scorer(**sc)
        res[mode] = s.score_batch(dict(batch), keep_isoforms=True)
        res[mode + "_exact"] = s.counters()["n_spec_exact"]
        res[mode + "_tables"] = [s.fetch_pep_scores(i)[1:3] for i in range(0, batch["n_mod"].size, 97)]
        res[mode + "_32"] = s.score_batch(b32)
        res[mode + "_64"] = s.score_batch(b64)
        s.close()
    assert _same(res["0"], res["1"]) and _same(res["0_32"], res["1_32"]) and _same(res["0_64"], res["0_32"])
    for (ca, sa), (cb, sb) in zip(res["0_tables"], res["1_tables"]):
        assert _golden.same_bits(ca, cb) and _golden.same_bits(sa, sb)
    assert res["0_exact"] == 0 and res["1_exact"] >= 1
    assert any(np.any(c[:, -1] > c[:, 9]) for c, _ in res["1_tables"])
