"""Host orchestration paths of the library that the parity suites do not reach.

Each case scores a fixed, seeded batch through one transfer path and compares every result it asked for, bit for bit,
with the same PSMs scored from host arrays through per-array copies (the "unpacked" form):
- a device-resident batch whose psm_spec is not in spectrum order (scored as one chunk over every spectrum);
- a device-resident PSM range that does not start at 0 (results at absolute positions, the rest left as it was);
- small host batches on the packed path (one block per direction), with some results not asked for;
- host batches just under and just over the packed input bound, and one whose results alone exceed the packed bound.

The byte counters tell which path ran.  Every counter that is not a timing must equal the value recorded from the
library at commit 2bece60 (PARENT below).
"""
import numpy as np
import pytest

from pyascore_b200 import Scorer, synth

pytestmark = pytest.mark.gpu

W = synth.WORKLOADS["lowres_phospho"]
PACK_MAX = 1 << 20
RESULTS = ("best_sig", "best_score", "n_iso", "n_sites", "ascores", "alt_sites", "psm_status")
COUNTERS = ("n_psm", "n_spec", "n_peaks", "n_retained", "n_isoforms", "n_fragment_lookups", "bytes_h2d", "bytes_d2h",
            "kernel_launches", "launches_bin", "launches_count", "launches_select", "launches_ascore", "n_chunks",
            "n_spec_exact")


def _counters(*values):
    return dict(zip(COUNTERS, values))


# recorded from the library at commit 2bece60 on a B200, in the order of COUNTERS
PARENT = {
    "device_range": {
        "device": _counters(1200, 3000, 333580, 0, 15529, 801196, 0, 0, 22, 2, 1, 2, 2, 1, 0),
        "host": _counters(1200, 3000, 333580, 0, 15529, 801196, 5402854, 55044, 19, 2, 1, 2, 2, 1, 0),
    },
    "device_unordered": {
        "device": _counters(2800, 3000, 842607, 0, 35265, 1802764, 0, 0, 22, 2, 1, 2, 2, 1, 0),
        "host": _counters(2800, 3000, 842607, 0, 35265, 1802764, 13635686, 128596, 19, 2, 1, 2, 2, 1, 0),
    },
    "pack_bound": {
        "over": _counters(236, 236, 65015, 0, 3246, 152320, 1053079, 10832, 18, 1, 1, 2, 2, 1, 0),
        "under": _counters(235, 235, 64602, 0, 3243, 152152, 1046432, 10828, 18, 1, 1, 2, 2, 1, 0),
    },
    "packed_some_results": {
        "full": _counters(40, 40, 13111, 0, 853, 64286, 212136, 1904, 18, 1, 1, 2, 2, 1, 0),
        "some": _counters(40, 40, 13111, 0, 853, 64286, 212136, 428, 18, 1, 1, 2, 2, 1, 0),
    },
    "results_over_bound": {
        "call": _counters(8000, 16, 4696, 0, 88000, 3872000, 395320, 1184000, 18, 1, 1, 2, 2, 1, 0),
    },
}


@pytest.fixture(scope="module")
def scorer():
    s = Scorer(device=0, **W["scorer"])
    yield s
    s.close()


def _take(batch, psms, n_spec=None):
    """the PSMs `psms` (in that order) of a host batch, over the batch's first `n_spec` spectra (default: all)"""
    psms = np.asarray(psms, np.int64)
    n_spec = batch["spec_off"].size - 1 if n_spec is None else n_spec
    so = batch["spec_off"][:n_spec + 1]
    out = dict(spec_off=so.copy(), mz=batch["mz"][:so[-1]].copy(), inten=batch["inten"][:so[-1]].copy(),
               psm_spec=batch["psm_spec"][psms].copy(), n_mod=batch["n_mod"][psms].copy(),
               max_charge=batch["max_charge"][psms].copy())
    for key, off in (("pep", "pep_off"), ("aux_pos", "aux_off")):
        lo, hi = batch[off][psms], batch[off][psms + 1]
        o = np.zeros(psms.size + 1, np.int32)
        np.cumsum(hi - lo, out=o[1:])
        out[off] = o
        idx = np.concatenate([np.arange(a, b) for a, b in zip(lo, hi)] + [np.zeros(0, np.int64)]).astype(np.int64)
        out[key] = batch[key][idx].copy()
        if key == "aux_pos":
            out["aux_mass"] = batch["aux_mass"][idx].copy()
    return out


def _head(batch, n):
    """the first n spectra of a batch with one PSM per spectrum, and their PSMs"""
    return _take(batch, np.arange(n), n)


def _with_mod_off(batch):
    b = dict(batch)
    b["mod_off"] = np.zeros(b["n_mod"].size + 1, np.int64)
    np.cumsum(np.maximum(b["n_mod"], 0), out=b["mod_off"][1:])
    return b


def _pack_bound(b):
    """the library's bound on a host batch's packed input block (every array at full size plus 16 bytes of alignment
    for each of 16)"""
    ns, npk, n = b["spec_off"].size - 1, int(b["spec_off"][-1] - b["spec_off"][0]), b["n_mod"].size
    return (ns + 1) * 8 + npk * 16 + n * 12 + (n + 1) * 16 + b["pep"].size + b["aux_pos"].size * 8 + 16 * 16


def _layout(sizes, start):
    """size of a packed block: the arrays one after another, each at a 16-byte aligned offset from `start`"""
    used = start
    for s in sizes:
        used = (used + 15) // 16 * 16 + s
    return used


def _in_sizes(b):
    """bytes of the host input arrays in the order the packed block holds them"""
    b = _with_mod_off(b)
    return [b[k].nbytes for k in ("spec_off", "mz", "inten", "psm_spec", "pep_off", "pep", "n_mod", "max_charge",
                                  "aux_off", "aux_pos", "aux_mass", "mod_off")]


def _out_sizes(b, want):
    b = _with_mod_off(b)
    n, nm = b["n_mod"].size, int(b["mod_off"][-1])
    per = dict(best_sig=8 * n, best_score=4 * n, n_iso=8 * n, n_sites=4 * n, ascores=4 * nm, alt_sites=8 * nm,
               psm_status=4 * n)
    return [per[k] for k in RESULTS if k in want]


def _host(v, key):
    if isinstance(v, np.ndarray):
        return v
    v = v.cpu().numpy()
    return v.view(np.uint64) if key in ("best_sig", "alt_sites") else v


def _score(s, batch, **kw):
    out = s.score_batch(dict(batch), **kw)
    c = s.counters()
    return {k: _host(v, k) for k, v in out.items()}, {k: c[k] for k in COUNTERS}


def _unpacked(s, batch, want=RESULTS):
    """results of the PSMs of a host batch scored with per-array copies: the batch followed by a filler batch that
    takes the call over the packed input bound"""
    filler = synth.make_batch(W, 512, seed=99)
    both = synth.concat_batches([batch, filler])
    assert _pack_bound(both) > PACK_MAX
    res, c = _score(s, both, want=want)
    assert c["bytes_h2d"] == sum(_in_sizes(both))
    n, nm = batch["n_mod"].size, int(np.maximum(batch["n_mod"], 0).sum())
    return {k: v[:nm] if k in ("ascores", "alt_sites") else v[:n] for k, v in res.items()}


def _same(got, ref, keys=RESULTS):
    for k in keys:
        assert got[k].dtype == ref[k].dtype and got[k].tobytes() == ref[k].tobytes(), k


def _to_dev(batch):
    import torch
    return {k: torch.from_numpy(v.view(np.int32) if v.dtype == np.uint32 else v).cuda() for k, v in batch.items()}


# ---- the cases: each returns the counters of the calls it checks ------------------------------------------------

def run_device_unordered(s):
    """A device-resident batch whose PSMs reference spectra out of order, and not the first or last ones: the whole
    spectrum array is binned as one chunk."""
    base = synth.make_batch(W, 3000, seed=11)
    order = np.random.default_rng(3).permutation(np.arange(100, 2900))
    b = _take(base, order)
    assert (np.diff(b["psm_spec"]) < 0).any()
    got, c = _score(s, _to_dev(b))
    ref, c_host = _score(s, b)
    _same(got, ref)
    assert c["n_chunks"] == 1 and c["n_peaks"] == int(b["spec_off"][-1])
    return {"device": c, "host": c_host}


def run_device_range(s):
    """pa_score_range on a device-resident batch with p_lo > 0: results land at absolute positions, values outside
    the range stay as they were."""
    import torch
    b = _with_mod_off(synth.make_batch(W, 3000, seed=12))
    lo, hi = 1000, 2200
    mlo, mhi = int(b["mod_off"][lo]), int(b["mod_off"][hi])
    n, nm = b["n_mod"].size, int(b["mod_off"][-1])
    fill = dict(best_sig=(0x5A5A5A5A5A5A5A5A, np.uint64), best_score=(-7.25, np.float32), n_iso=(-3, np.int64),
                n_sites=(-5, np.int32), ascores=(-9.5, np.float32), alt_sites=(0x3C3C3C3C3C3C3C3C, np.uint64),
                psm_status=(-11, np.int32))
    preset = {k: np.full(nm if k in ("ascores", "alt_sites") else n, v, t) for k, (v, t) in fill.items()}
    out_dev = {k: torch.from_numpy(v.view(np.int64) if v.dtype == np.uint64 else v.copy()).cuda()
               for k, v in preset.items()}
    out_host = {k: v.copy() for k, v in preset.items()}
    got, c = _score(s, _to_dev(b), out=out_dev, psm_range=(lo, hi))
    ref, c_host = _score(s, b, out=out_host, psm_range=(lo, hi))
    _same(got, ref)
    for k, v in got.items():
        a, z = (mlo, mhi) if k in ("ascores", "alt_sites") else (lo, hi)
        assert v[:a].tobytes() == preset[k][:a].tobytes() and v[z:].tobytes() == preset[k][z:].tobytes(), k
        assert v[a:z].tobytes() != preset[k][a:z].tobytes(), k
    assert c["n_psm"] == hi - lo
    return {"device": c, "host": c_host}


def run_packed_some_results(s):
    """A small host batch on the packed path that asks for two results: they equal those of a full call and of the
    unpacked form."""
    b = synth.make_batch(W, 40, seed=13)
    want = ("best_score", "ascores")
    got, c = _score(s, b, want=want)
    full, c_full = _score(s, b)
    ref = _unpacked(s, b)
    assert sorted(got) == sorted(want)
    _same(got, full, want)
    _same(full, ref)
    assert c["bytes_h2d"] == c_full["bytes_h2d"] == _layout(_in_sizes(b), 0)
    assert c["bytes_d2h"] == _layout(_out_sizes(b, want), 16)
    assert c_full["bytes_d2h"] == _layout(_out_sizes(b, RESULTS), 16)
    return {"some": c, "full": c_full}


def _split_at_pack_bound():
    base = synth.make_batch(W, 400, seed=14)
    lo, hi = 1, 400                          # the bound grows with the spectra taken: bisect for the last that fits
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if _pack_bound(_head(base, mid)) <= PACK_MAX else (lo, mid)
    return _head(base, lo), _head(base, lo + 1)


def run_pack_bound(s):
    """Host batches one spectrum under and one over the packed input bound."""
    under, over = _split_at_pack_bound()
    assert _pack_bound(under) <= PACK_MAX < _pack_bound(over)
    got_u, c_u = _score(s, under)
    got_o, c_o = _score(s, over)
    _same(got_u, _unpacked(s, under))
    _same(got_o, _unpacked(s, over))
    assert c_u["bytes_h2d"] == _layout(_in_sizes(under), 0)
    assert c_u["bytes_d2h"] == _layout(_out_sizes(under, RESULTS), 16)
    assert c_o["bytes_h2d"] == sum(_in_sizes(over)) and c_o["bytes_d2h"] == sum(_out_sizes(over, RESULTS))
    return {"under": c_u, "over": c_o}


def run_results_over_bound(s):
    """A host batch whose inputs fit the packed block and whose results do not: inputs go packed, results come back
    per array."""
    base = _head(synth.make_batch(W, 16, seed=15), 16)
    n = 8000
    pep = np.frombuffer(b"SSSSSSSSSSSK", np.uint8)
    b = dict(spec_off=base["spec_off"], mz=base["mz"], inten=base["inten"],
             psm_spec=np.repeat(np.arange(16, dtype=np.int32), n // 16),
             pep_off=(np.arange(n + 1) * pep.size).astype(np.int32), pep=np.tile(pep, n),
             n_mod=np.full(n, 10, np.int32), max_charge=np.full(n, 2, np.int32), aux_off=np.zeros(n + 1, np.int32),
             aux_pos=np.zeros(0, np.uint32), aux_mass=np.zeros(0, np.float32))
    nm = 10 * n
    assert _pack_bound(b) <= PACK_MAX < n * 32 + nm * 12 + 8 * 16
    got, c = _score(s, b)
    _same(got, _unpacked(s, b))
    assert c["bytes_h2d"] == _layout(_in_sizes(b), 0)
    assert c["bytes_d2h"] == sum(_out_sizes(b, RESULTS))
    return {"call": c}


CASES = {"device_unordered": run_device_unordered, "device_range": run_device_range,
         "packed_some_results": run_packed_some_results, "pack_bound": run_pack_bound,
         "results_over_bound": run_results_over_bound}


@pytest.mark.parametrize("case", sorted(CASES))
def test_orchestration(scorer, case):
    counters = CASES[case](scorer)
    assert counters == PARENT[case]
