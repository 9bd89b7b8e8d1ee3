"""CPU: the deep cases of tests/test_gpu_deep_limits.py, on the C oracle alone.  A case at n_top > 10 whose spectra hold
at most ten peaks per bin has no rank >= 10: K2d adds zeros, every deep column equals column 9 and a comparison with
the oracle passes however wrong the deep path is.  These tests show without a GPU that no deep case is vacuous -- each
reaches ranks >= 10 in its PSMs and Ascores taken at depths >= 10 -- that the deep variant matrix selects every kernel
instantiation, and that the default shape groups (tests/test_gpu_limits.py, tests/test_oracle_limits.py) still draw
the batches they drew before the deep helpers were added."""
import hashlib
import json

import numpy as np
import pytest

import _golden
import _limits
from test_gpu_deep_ntop import deep_reach

# SHA-256 of meta and batch of every default group, recorded before tests/_limits.py had the deep helpers
DEFAULT_DIGESTS = {
    "length": "960535d71aea577bdc086ca249ce53de5717942c498e4b731b76f0ea371b8221",
    "length_nl": "eadee952a2a57ff6c6e42ffa7700c43283f6b35a9195343e341523ea347720e7",
    "sites": "0b55acafaae66c7c24b4551d422dc0a3e6fb43671c975d9770568479ddf3ae05",
    "peaks_50": "393d68f8daa083c9e3bb2a0ff77727bfeff9b0e4eda5d5f6ff19e3a32895aa6f",
    "peaks_10": "216c02d96980f155aad62561c4780e86e212fe14f46b835942151a998409e98c",
    "peaks_7.3": "1098b27d91e906110f0ca11e92c1936ed1f4d13f831f23367f8268bdd31938d0",
    "charge": "5465eb32a2aaf546a19f234e03335ae8a92b34c5c16eff35d3c4648b3cb3c3dc",
    "charge_nl": "c4ac3f7f3ba9c9a30ad6c105461895d4d9a258ddcaec3ac678b8cdfe5cf45341",
    "fragments": "532ecd89f3979267c7af0edd3ff1a313ab946b648fd4286103ca264d87040496",
    "fragments_nl": "7d0ab99c497c4a10fb874a09b03c3fb87a96f9df8415ea9a9d579b322673fa2b",
    "isoforms": "665f4d4145a3a329bad85542f4dd0ea708b29350788b2ba0c2521a537ebc5a8b",
    "dense": "de78cfac7145fea689c624e05a3c4c776f25e6f1df57f4d0c5fdf36904af4fb6",
    "status": "31bf7ef71d6eb3482f8dec89fbc108d74e6f0b85d3a9fafff70a329f1a9bbd5d",
}
DEFAULT_GROUPS = {
    "length": _limits.length_group, "length_nl": lambda: _limits.length_group([("st", 97.9769)]),
    "sites": _limits.sites_group, "peaks_50": lambda: _limits.peaks_group(50.),
    "peaks_10": lambda: _limits.peaks_group(10.), "peaks_7.3": lambda: _limits.peaks_group(7.3),
    "charge": _limits.charge_group, "charge_nl": lambda: _limits.charge_group([("ST", 18.01528)]),
    "fragments": _limits.frag_group, "fragments_nl": _limits.frag_group_nl,
    "isoforms": _limits.isoform_group, "dense": _limits.dense_group, "status": _limits.status_group}


def group_digest(g):
    h = hashlib.sha256(json.dumps(g.meta, sort_keys=True).encode())
    b = g.batch()
    for k in sorted(b):
        h.update(k.encode())
        h.update(np.ascontiguousarray(b[k]).tobytes())
    return h.hexdigest()


def deep_rank_psms(ref, n_psm):
    """per PSM: some isoform's cumulative count at the last depth exceeds its count at depth 9 (a match of rank >= 10)"""
    off, c = ref["iso_off"], ref["iso_counts"]
    return [bool(np.any(c[off[i]:off[i + 1], -1] > c[off[i]:off[i + 1], 9])) for i in range(n_psm)]


def prove_deep(name, g, ref):
    """every PSM of a deep group matches a peak of rank >= 10, except the tied PSMs on two far-away peaks and the one- and
    two-residue PSMs of the default groups, whose spectra hold at most one ion of theirs (add_one_residue_deep's PSM is
    held to it); dense at n_top 64 brings the deep counts above 3000 and reads T_deep rows above 4000"""
    n = len(g.info)
    reach = deep_rank_psms(ref, n)
    off = ref["iso_off"]
    can = [int(ref["iso_total"][off[i]:off[i + 1]].max()) > 0 and not g.info[i].get("tied")
           and (g.info[i]["L"] > 2 or g.info[i].get("one_residue_deep")) for i in range(n)]
    assert any(can) and all(r for r, c in zip(reach, can) if c), [i for i in range(n) if can[i] and not reach[i]]
    if name == "length_nl":
        assert any(x.get("one_residue_deep") and r for x, r in zip(g.info, reach))
    if name == "dense" and g.meta["scorer"]["n_top"] == 64:
        assert ref["iso_counts"][:, 10:].max() > 3000 and ref["iso_total"].max() > 4000
    return reach


def test_default_groups_unchanged():
    for name, build in DEFAULT_GROUPS.items():
        assert group_digest(build()) == DEFAULT_DIGESTS[name], name


@pytest.mark.parametrize("name,n_top", _limits.DEEP_SHAPES, ids=["%s-%d" % c for c in _limits.DEEP_SHAPES])
def test_deep_groups_reach_deep_ranks(name, n_top):
    """each deep shape group reaches ranks >= 10 in every PSM that can match, and Ascores taken at depths >= 10 (but for
    the cases of DEEP_SHALLOW_ASCORES)"""
    g = _limits.deep_group(name, n_top)
    assert g.meta["scorer"]["n_top"] == n_top
    batch = g.batch()
    ref = _golden.oracle_ref(g.meta, batch)
    assert ref["iso_counts"].shape[1] == n_top
    prove_deep(name, g, ref)
    if (name, n_top) not in _limits.DEEP_SHALLOW_ASCORES:
        assert deep_reach(g.meta, batch, ref), "no Ascore of %s at n_top %d was taken at a depth >= 10" % (name, n_top)


def test_every_group_with_ascores_takes_one_deep():
    assert {n for n, t in _limits.DEEP_SHAPES if (n, t) not in _limits.DEEP_SHALLOW_ASCORES} == \
        {n for n, _ in _limits.DEEP_SHAPES} - {"dense"}


def test_deep_matrix_selects_every_instantiation():
    """the n_top 20 matrix takes both k_count_deep<HAS_NL> instantiations and all eight k_count_score ones, the n_top 64
    representatives one of each k_count_score instantiation"""
    at20 = {_limits.k2_instantiation(*_limits.VARIANTS[q]) for q, t in _limits.DEEP_MATRIX if t == 20}
    at64 = [_limits.k2_instantiation(*_limits.VARIANTS[q]) for q, t in _limits.DEEP_MATRIX if t == 64]
    assert len(at20) == 8 and {v[0] for v in at20} == {False, True}
    assert len(at64) == len(set(at64)) == 8


@pytest.mark.parametrize("q,n_top", _limits.DEEP_MATRIX, ids=["%d-%d" % c for c in _limits.DEEP_MATRIX])
def test_deep_matrix_reaches_deep_ranks(q, n_top):
    meta, batch = _limits.deep_variant_case(q, n_top)
    ref = _golden.oracle_ref(meta, batch)
    reach = deep_rank_psms(ref, batch["n_mod"].size)
    assert np.mean(reach) > 0.25, np.mean(reach)
