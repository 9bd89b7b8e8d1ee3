"""GPU: several modification types in one call (pa_score_typed / score_typed).

A typed batch holds, for the same spectra, the rows of every modification type; each row is scored under its own
type's scorer while the spectra are copied and binned once.  The yardstick is the single-type call: the rows of type
t must equal `Scorer.score_batch` of scorer t on a batch of those rows alone, bit for bit in all seven result arrays,
and a sample of rows is checked against the live C oracle.  The counters must show the work done once per chunk
(binning, peak bytes) and once per type with PSMs in a chunk (the counting kernel).
"""
import ctypes as C

import numpy as np
import pytest

import _golden
from pyascore_b200 import Scorer, _lib, format_results, score_typed, synth

pytestmark = pytest.mark.gpu

RESULTS = ("best_sig", "best_score", "n_iso", "n_sites", "ascores", "alt_sites", "psm_status")
PHOSPHO = dict(bin_size=100., n_top=10, mod_group="STY", mod_mass=79.966331, mz_error=0.5, fragment_types="by")
ACETYL = dict(bin_size=100., n_top=10, mod_group="K", mod_mass=42.010565, mz_error=0.5, fragment_types="by")
OXIDATION = dict(bin_size=100., n_top=10, mod_group="M", mod_mass=15.9949, mz_error=0.5, fragment_types="by")
NON_TIMING = ("n_psm", "n_spec", "n_peaks", "n_retained", "n_isoforms", "n_fragment_lookups", "bytes_h2d", "bytes_d2h",
              "kernel_launches", "launches_bin", "launches_count", "launches_select", "launches_ascore", "n_chunks",
              "n_spec_exact", "launches_deep")


def gather(batch, rows):
    return synth.select_rows(batch, rows)


def typed_batch(base, extra, skip_below=0):
    return synth.typed_batch(base, [kw["mod_group"] for kw in extra], skip_below)


def make(kw, nl=(), device=0):
    s = Scorer(device=device, **kw)
    for g, m in nl:
        s.add_neutral_loss(g, m)
    return s


def rows_of(res, batch, sel):
    """the result rows `sel` of a result dict, in the layout a batch of those rows alone has"""
    idx, _ = synth._ragged(batch["mod_off"], np.asarray(sel, np.int64))
    out = {}
    for k in RESULTS:
        v = res[k] if isinstance(res[k], np.ndarray) else res[k].cpu().numpy()
        out[k] = v[idx] if k in ("ascores", "alt_sites") else v[sel]
    return out


def assert_same(a, b, what=""):
    for k in RESULTS:
        x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), (what, k)


def check_separate(scorers, batch, psm_type, res):
    """rows of type t == scorers[t].score_batch on those rows alone, bit for bit"""
    for t, sc in enumerate(scorers):
        sel = np.flatnonzero(psm_type == t)
        if sel.size == 0:
            continue
        alone = sc.score_batch(gather(batch, sel))
        assert_same(rows_of(res, batch, sel), alone, "type %d" % t)


def check_oracle(kws, nls, batch, psm_type, res, scorers, per_type=25):
    from oracle.cscorer import OraclePyAscore
    rng = np.random.default_rng(7)
    bad = []
    for t, (kw, nl) in enumerate(zip(kws, nls)):
        R = OraclePyAscore(**kw)
        for g, m in nl:
            R.add_neutral_loss(g, m)
        sel = np.flatnonzero(psm_type == t)
        for i in rng.choice(sel, size=min(per_type, sel.size), replace=False):
            R.score(*synth.psm_view(batch, int(i)))
            seq, best, asc, alts = format_results(scorers[t], batch, res, int(i))
            if seq != R.best_sequence or not _golden.same_bits(np.float32(best), np.float32(R.best_score)):
                bad.append((t, int(i), seq, R.best_sequence, best, R.best_score))
            if not _golden.same_bits(asc, np.asarray(R.ascores, np.float32)):
                bad.append((t, int(i), "ascores", asc, R.ascores))
            for j, alt in enumerate(R.alt_sites):
                if not np.array_equal(alts[j], np.asarray(alt, np.uint32)):
                    bad.append((t, int(i), "alt_sites", j, alts[j], alt))
    assert not bad, "%d mismatches against the oracle, first: %r" % (len(bad), bad[:3])


@pytest.fixture(scope="module")
def phospho():
    s = make(PHOSPHO)
    yield s
    s.close()


@pytest.fixture(scope="module")
def acetyl():
    s = make(ACETYL)
    yield s
    s.close()


@pytest.fixture(scope="module")
def mixed():
    base = synth.make_batch("lowres_phospho", 3000, seed=11)
    return typed_batch(base, [ACETYL])


def test_typed_equals_separate(phospho, acetyl, mixed):
    batch, psm_type = mixed
    assert 0 < (psm_type == 1).sum() < psm_type.size
    res = score_typed([phospho, acetyl], batch, psm_type)
    assert np.all(res["psm_status"] == 0)
    check_separate([phospho, acetyl], batch, psm_type, res)
    check_oracle([PHOSPHO, ACETYL], [(), ()], batch, psm_type, res, [phospho, acetyl])


@pytest.mark.parametrize("n_top", [10, 20])
def test_per_type_settings(n_top):
    """mz_error 0.02 vs 0.6 (both EG forms of K2: EG is mz_error > 0.5), "by" vs "cz", neutral losses on one type
    only; at n_top 20 also K2d and the DEEP forms of K3b / K3c per type"""
    k0 = dict(PHOSPHO, n_top=n_top, mz_error=0.02)
    k1 = dict(ACETYL, n_top=n_top, mz_error=0.6, fragment_types="cz")
    nl0, nl1 = [("st", 97.9769)], []
    s0, s1 = make(k0, nl0), make(k1, nl1)
    base = synth.make_batch("hires_phospho_nl", 1500, seed=12)
    batch, psm_type = typed_batch(base, [k1])
    res = score_typed([s0, s1], batch, psm_type)
    c = s0.counters()
    assert c["launches_deep"] == (2 * c["n_chunks"] if n_top > 10 else 0)
    check_separate([s0, s1], batch, psm_type, res)
    check_oracle([k0, k1], [nl0, nl1], batch, psm_type, res, [s0, s1], per_type=15)
    s0.close(); s1.close()


def test_small_batch_packed_path(phospho, acetyl):
    base = synth.make_batch("lowres_phospho", 60, seed=13)
    batch, psm_type = typed_batch(base, [ACETYL])
    res = score_typed([phospho, acetyl], batch, psm_type)
    c = phospho.counters()
    assert c["n_chunks"] == 1 and c["bytes_d2h"] > 0
    check_separate([phospho, acetyl], batch, psm_type, res)
    single = phospho.score_batch(batch)
    cs = phospho.counters()
    # the packed block: the type array (n_psm bytes, 16-byte aligned) is the only extra input
    assert 0 <= c["bytes_h2d"] - cs["bytes_h2d"] - batch["n_mod"].size < 16
    assert c["bytes_d2h"] == cs["bytes_d2h"]
    del single


def _chunk_per(n):
    return min(131072, max(16384, ((n + 7) // 8 + 1023) // 1024 * 1024))


def test_several_chunks_and_a_chunk_without_a_type(monkeypatch):
    """a host batch cut into several chunks, the first of which holds no acetyl rows; the work counters.  (Scorers
    that always narrow the m/z: the default decides per call by timing, which would make the byte counts of two calls
    differ.)"""
    monkeypatch.setenv("PA_NARROW", "1")
    phospho, acetyl = make(PHOSPHO), make(ACETYL)
    base = synth.make_batch("lowres_phospho", 40000, seed=14)
    batch, psm_type = typed_batch(base, [ACETYL], skip_below=20000)
    n = psm_type.size
    per = _chunk_per(n)
    assert not np.any(psm_type[:per] == 1) and np.all([np.any(psm_type[a:a + per] == 1) for a in range(per, n, per)])
    res = score_typed([phospho, acetyl], batch, psm_type)
    c = phospho.counters()
    n_chunks = (n + per - 1) // per
    assert c["n_chunks"] == n_chunks >= 3
    check_separate([phospho, acetyl], batch, psm_type, res)
    # work done once: binning and the peak bytes are those of a single-type call over the same rows
    phospho.score_batch(batch)
    cs = phospho.counters()
    assert c["launches_bin"] == cs["launches_bin"] and c["n_peaks"] == cs["n_peaks"] and c["n_chunks"] == cs["n_chunks"]
    assert c["bytes_h2d"] == cs["bytes_h2d"] + n                     # + one type byte per PSM, nothing else
    assert c["bytes_d2h"] == cs["bytes_d2h"]
    # the counting kernel once per type with PSMs in a chunk: chunk 0 has phospho rows only
    assert c["launches_count"] == 2 * n_chunks - 1
    assert c["launches_select"] == 2 * (2 * n_chunks - 1)
    # the separate calls copy and bin the peaks of the spectra the acetyl rows share a second time
    a0 = phospho.score_batch(gather(batch, np.flatnonzero(psm_type == 0)))
    b0 = phospho.counters()
    a1 = acetyl.score_batch(gather(batch, np.flatnonzero(psm_type == 1)))
    b1 = acetyl.counters()
    assert c["n_peaks"] < b0["n_peaks"] + b1["n_peaks"]
    assert c["bytes_h2d"] < b0["bytes_h2d"] + b1["bytes_h2d"]
    del a0, a1
    phospho.close(); acetyl.close()


def test_device_resident(phospho, acetyl, mixed):
    torch = pytest.importorskip("torch")
    batch, psm_type = mixed
    host = score_typed([phospho, acetyl], batch, psm_type)
    dev = {k: torch.from_numpy(v.view(np.int32) if v.dtype == np.uint32 else v).cuda()
           for k, v in batch.items() if k != "mod_off"}
    res = score_typed([phospho, acetyl], dev, torch.from_numpy(psm_type).cuda())
    torch.cuda.synchronize()
    got = {k: np.ascontiguousarray(res[k].cpu().numpy()).view(host[k].dtype) for k in RESULTS}
    assert_same(got, host, "device-resident")
    c = phospho.counters()
    assert c["n_chunks"] == 1 and c["bytes_h2d"] == 0 and c["launches_count"] == 2
    with pytest.raises(ValueError):
        score_typed([phospho, acetyl], dev, psm_type)               # the types must be where the batch is


def test_all_rows_of_one_type(phospho, acetyl, mixed):
    """type 0 has no PSMs at all: only the acetyl pass runs"""
    batch, psm_type = mixed
    sel = np.flatnonzero(psm_type == 1)
    sub = gather(batch, sel)
    ones = np.ones(sel.size, np.uint8)
    res = score_typed([phospho, acetyl], sub, ones)
    assert_same(res, acetyl.score_batch(sub), "only type 1")
    assert phospho.counters()["launches_count"] == phospho.counters()["n_chunks"]


def test_three_types(phospho, acetyl):
    ox = make(OXIDATION)
    base = synth.make_batch("lowres_phospho", 4000, seed=15)
    batch, psm_type = typed_batch(base, [ACETYL, OXIDATION])
    assert set(np.unique(psm_type)) == {0, 1, 2}
    res = score_typed([phospho, acetyl, ox], batch, psm_type)
    check_separate([phospho, acetyl, ox], batch, psm_type, res)
    check_oracle([PHOSPHO, ACETYL, OXIDATION], [(), (), ()], batch, psm_type, res, [phospho, acetyl, ox], per_type=10)
    ox.close()


@pytest.mark.parametrize("n", [60, 40000])
def test_no_types_is_score_batch(monkeypatch, n):
    """psm_type None: every PSM is type 0 -- the results and the counters of pa_score_batch on s[0] (scorers that
    always narrow, as above)"""
    monkeypatch.setenv("PA_NARROW", "1")
    phospho, acetyl = make(PHOSPHO), make(ACETYL)
    batch = synth.make_batch("lowres_phospho", n, seed=16)
    a = score_typed([phospho, acetyl], batch, None)
    ca = phospho.counters()
    b = phospho.score_batch(batch)
    cb = phospho.counters()
    assert_same(a, b, "psm_type None")
    assert {k: ca[k] for k in NON_TIMING} == {k: cb[k] for k in NON_TIMING}
    phospho.close(); acetyl.close()


def _raw(scorers, batch, psm_type, flags=0, n_types=None):
    s0 = scorers[0]
    pb, pr, out = s0._prepare(batch, None, RESULTS)
    handles = (C.c_void_p * len(scorers))(*[getattr(s, "h", s) for s in scorers])
    rc = _lib.load().pa_score_typed(handles, len(scorers) if n_types is None else n_types, C.byref(pb),
                                    None if psm_type is None else psm_type.ctypes.data, C.byref(pr), flags)
    return rc, out


def test_refusals(phospho, acetyl, mixed):
    L = _lib.load()
    batch, psm_type = mixed
    ERR_ARG, ERR_UNSUPPORTED, ERR_STATE = -2, -3, -4
    for n_types in (0, 256):
        rc, _ = _raw([phospho] * 256, batch, psm_type, n_types=n_types)
        assert rc == ERR_ARG and "n_types" in _lib.last_error(phospho.h)
    rc, _ = _raw([phospho, None], batch, psm_type)
    assert rc == ERR_ARG and "NULL" in _lib.last_error(phospho.h)
    h = C.c_void_p()
    assert L.pa_create_binner(100., 10, 0, C.byref(h)) == 0
    try:
        rc, _ = _raw([phospho, h.value], batch, psm_type)
        assert rc == ERR_ARG and "binner" in _lib.last_error(phospho.h)
    finally:
        L.pa_destroy(h)
    for kw in (dict(ACETYL, bin_size=50.), dict(ACETYL, n_top=20)):
        other = make(kw)
        rc, _ = _raw([phospho, other], batch, psm_type)
        assert rc == ERR_ARG and "bin_size" in _lib.last_error(phospho.h)
        with pytest.raises(ValueError):
            score_typed([phospho, other], batch, psm_type)
        other.close()
    rc, _ = _raw([phospho, acetyl], batch, psm_type, flags=_lib.PA_KEEP_ISOFORMS)
    assert rc == ERR_UNSUPPORTED and "PA_KEEP_ISOFORMS" in _lib.last_error(phospho.h)
    side = synth.make_batch("acetyl_k", 300, seed=17)
    acetyl.score_batch_async(side)
    try:
        rc, _ = _raw([phospho, acetyl], batch, psm_type)
        assert rc == ERR_STATE and "in flight" in _lib.last_error(phospho.h)
    finally:
        acetyl.wait()
    rc, _ = _raw([phospho, acetyl], batch, psm_type)                    # usable again
    assert rc == 0


def test_refusal_other_device(phospho, mixed):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("one visible GPU")
    batch, psm_type = mixed
    other = make(ACETYL, device=1)
    rc, _ = _raw([phospho, other], batch, psm_type)
    assert rc == -2 and "device" in _lib.last_error(phospho.h)
    other.close()


def test_type_out_of_range(phospho, acetyl, mixed):
    batch, psm_type = mixed
    good = score_typed([phospho, acetyl], batch, psm_type)
    bad_t = psm_type.copy()
    bad_rows = [5, int(np.flatnonzero(psm_type == 1)[3])]
    bad_t[bad_rows[0]] = 7
    bad_t[bad_rows[1]] = 2
    res = score_typed([phospho, acetyl], batch, bad_t)
    assert list(np.flatnonzero(res["psm_status"] != 0)) == sorted(bad_rows)
    assert np.all(res["psm_status"][bad_rows] == 7)                   # PA_PSM_BAD_INDEX
    keep = np.setdiff1d(np.arange(psm_type.size), bad_rows)
    assert_same(rows_of(res, batch, keep), rows_of(good, batch, keep), "other rows")


# ---- the CLI on BASELINE config 1 (the reference's example files, tests/golden/cli/config1.npz) ----

def _config1_files(tmp_path):
    import _msfiles
    from test_parsing import load_config1
    spectra, queries, expected = load_config1()
    spec, ident = str(tmp_path / "s.mzML"), str(tmp_path / "i.pep.xml")
    _msfiles.write_mzml(spec, spectra, inten_bits=32)
    _msfiles.write_pepxml(ident, queries)
    return spec, ident, expected


def _argv(over):
    out = []
    for k, v in over.items():
        out += ["--" + k, str(v)]
    return out


def test_cli_extra_mod_equals_reference(tmp_path):
    """--hit_depth 2 with oxidation on M as a second type: each file is the reference's TSV for that type alone"""
    from pyascore_b200.__main__ import main
    spec, ident, expected = _config1_files(tmp_path)
    out, ox = str(tmp_path / "o.tsv"), str(tmp_path / "ox.tsv")
    main(["--hit_depth", "2", "--extra_mod", "M:15.9949:" + ox, spec, ident, out])
    assert open(out).read() == expected["hit_depth2"]["tsv"]
    assert open(ox).read() == expected["oxidation"]["tsv"]
    # the same through a parameter file, with the chunks cut small (several typed batches)
    pf = tmp_path / "p.txt"
    out2, ox2 = str(tmp_path / "o2.tsv"), str(tmp_path / "ox2.tsv")
    pf.write_text("hit_depth = 2\nchunk_psms = 3\nextra_mod = M:15.9949:%s\n" % ox2)
    main(["--parameter_file", str(pf), spec, ident, out2])
    assert open(out2).read() == expected["hit_depth2"]["tsv"]
    assert open(ox2).read() == expected["oxidation"]["tsv"]


def test_cli_extra_mods_equal_separate_runs(tmp_path):
    """the hires_nl flags (neutral loss on st, all hits) plus acetyl on K and oxidation on M with its own neutral loss:
    each type's file equals a separate run of that type"""
    from pyascore_b200.__main__ import main
    spec, ident, expected = _config1_files(tmp_path)
    over = expected["hires_nl"]["args"]
    out, ac, ox = (str(tmp_path / n) for n in ("o.tsv", "ac.tsv", "ox.tsv"))
    main(_argv(over) + ["--extra_mod", "K:42.010565:" + ac, "--extra_mod", "M:15.9949:%s:m:63.998285" % ox,
                        spec, ident, out])
    assert open(out).read() == expected["hires_nl"]["tsv"]
    base = {k: v for k, v in over.items() if not k.startswith("neutral_loss")}
    for path, flags in ((ac, ["--residues", "K", "--mod_mass", "42.010565"]),
                        (ox, ["--residues", "M", "--mod_mass", "15.9949", "--neutral_loss_groups", "m",
                              "--neutral_loss_masses", "63.998285"])):
        alone = str(tmp_path / "alone.tsv")
        main(_argv(base) + flags + [spec, ident, alone])
        assert open(path).read() == open(alone).read(), path
    pf = tmp_path / "p.txt"
    pf.write_text("".join("%s = %s\n" % kv for kv in over.items()) +
                  "extra_mod = K:42.010565:%s\nextra_mod = M:15.9949:%s:m:63.998285\n" % (ac + "2", ox + "2"))
    main(["--parameter_file", str(pf), spec, ident, out + "2"])
    for a, b in ((out, out + "2"), (ac, ac + "2"), (ox, ox + "2")):
        assert open(a).read() == open(b).read()
