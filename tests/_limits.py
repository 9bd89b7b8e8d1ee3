"""Hand-built PSMs at the shape limits of the library (include/pyascore_b200.h and the capacities in
pyascore_b200/csrc/pa_device.cuh / pa_kernels.cuh), shared by tests/test_gpu_limits.py (GPU against the C oracle)
and tests/test_oracle_limits.py (the oracle against closed forms).

Every group is (meta, batch, info): `meta` is the scorer set-up in the layout of the golden files, `batch` a CSR
batch (one spectrum per PSM), `info` a list of per-PSM dicts with what the case is meant to reach.  The library has
no counter that says which kernel path ran, so each case carries the numbers the path choice is made from
(peptide length, site count, charge, ion types, neutral-loss variants) and the tests prove from those that both
sides of every limit were scored.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))

import make_golden  # noqa: E402

PHOS = dict(bin_size=100., n_top=10, mod_group="STY", mod_mass=79.966331, mz_error=0.5, fragment_types="by")
FILLER = "AGLVEPKRNQFIWHM"      # neither a phospho site (STY) nor a residue any group below gives a loss (D, S, T)
SITES = "STY"

# library limits the cases straddle (include/pyascore_b200.h, pa_device.cuh, pa_kernels.cuh)
MAX_PEPTIDE = 126
MAX_SITES = 63
MAX_FRAGMENTS = 4095
MAX_ISOFORMS = 1 << 26
LMAX_FAST = 64          # pa_walk_fast: 2 <= L <= 64 with staged peaks
RCAP = 255              # retained peaks staged in shared memory
ROW_MAX_BINS = 128      # K1's row form takes spectra of at most this many bins
LCAP = 256              # fragments per (isoform, ion type) list in shared memory (K3c)
SORTCAP = 256
SEL_THREAD_MAX = 512
UNIT = 1024
MAXSTREAM = 12

_MASS = {'G': 57.02146, 'A': 71.03711, 'S': 87.03203, 'P': 97.05276, 'V': 99.06841, 'T': 101.04768,
         'C': 103.00919, 'L': 113.08406, 'I': 113.08406, 'N': 114.04293, 'D': 115.02694, 'Q': 128.05858,
         'K': 128.09496, 'E': 129.04259, 'M': 131.04049, 'H': 137.05891, 'F': 147.06841, 'U': 150.95364,
         'R': 156.10111, 'Y': 163.06333, 'W': 186.07931, 'O': 237.14773}
_ION_SHIFT = {'b': 0., 'c': 17.026549, 'y': 18.010565, 'z': 18.010565 - 17.026549, 'Z': 18.010565 - 16.018724}


# ---- the k_count_score variant matrix: ion types x mz_error x neutral-loss sets
FTYPES = ["b", "y", "c", "by", "yb", "bcyzZ", "zbc"]
ERR_ABOVE_HALF = float(np.nextafter(np.float32(0.5), np.float32(1)))        # the first float32 above 0.5
ERRS = [0.02, 0.5, ERR_ABOVE_HALF, 0.75, 1.5]
NLS = [[], [("st", 97.9769)],
       [("st", 97.9769), ("ST", 18.01528), ("K", 17.026549), ("DE", 18.010565)]]     # PA_MAX_NL_MASSES distinct masses
# all pairs of the three settings: every (ion types, mz_error) pair once, the loss set cycling so that every
# (ion types, losses) and (mz_error, losses) pair occurs too
VARIANTS = [(f, e, NLS[(i + 2 * j) % 3]) for i, f in enumerate(FTYPES) for j, e in enumerate(ERRS)]


def k2_instantiation(ftypes, err, nl):
    """(HAS_NL, PAIR, EGH) of k_count_score for a scorer set-up, as pa_lib.cu picks it: neutral losses configured,
    exactly two ion types, mz_error > 0.5 in float32"""
    return bool(nl), len(ftypes) == 2, bool(np.float32(err) > np.float32(0.5))


def peptide(rng, L, site_idx, d_idx=()):
    """L residues of FILLER with S/T/Y at the 0-based indices `site_idx` and D at `d_idx`"""
    p = list(rng.choice(list(FILLER), size=L))
    for i in site_idx:
        p[i] = SITES[rng.integers(0, 3)]
    for i in d_idx:
        p[i] = "D"
    return "".join(p)


def ions(pep, mod_idx, types, Z, mod_mass=79.966331):
    """float64 m/z of the ions of the isoform with mods at residue indices `mod_idx` (only used to place peaks)"""
    m = np.array([_MASS[c] for c in pep]) + np.isin(np.arange(len(pep)), list(mod_idx)) * mod_mass
    b = np.cumsum(m)[:-1]
    y = m.sum() - b + 18.010565
    out = []
    for t in types:
        base = b + _ION_SHIFT[t] if t in "bc" else y - 18.010565 + _ION_SHIFT[t]
        for z in range(1, Z + 1):
            out.append((base + z * 1.007825) / z)
    return np.concatenate(out) if out else np.zeros(0)


def spectrum(rng, ion_mz, bin_size=100., lo=100., hi=2000., per_bin=None, n_noise=60, keep=0.6):
    """(mz, inten) sorted by m/z.  per_bin=None: the ions inside [lo, hi) kept with probability `keep`, jittered, plus
    uniform noise.  per_bin=array: exactly per_bin[b] peaks in bin b (bins counted from `lo`, a multiple of 100, as the
    reference does), the ions of that bin first, so the number of retained peaks is sum(min(per_bin, 10))."""
    bs = float(np.float32(bin_size))
    if per_bin is None:
        sig = ion_mz[(ion_mz > lo + 1.) & (ion_mz < hi - 1.)]
        sig = sig[rng.random(sig.size) < keep]
        sig = sig + rng.normal(0., 0.1, sig.size)
        mz = np.concatenate([sig, rng.uniform(lo + 1., hi - 1., n_noise)])
        is_sig = np.arange(mz.size) < sig.size
    else:
        parts, flags = [], []
        for b, c in enumerate(per_bin):
            a0, a1 = lo + b * bs + 0.02 * bs, lo + (b + 1) * bs - 0.02 * bs
            inside = ion_mz[(ion_mz > a0) & (ion_mz < a1)][:c]
            fill = rng.uniform(a0, a1, c - inside.size)
            parts += [inside, fill]
            flags += [np.ones(inside.size, bool), np.zeros(fill.size, bool)]
        mz, is_sig = np.concatenate(parts), np.concatenate(flags)
    inten = np.exp(np.where(is_sig, 6.0, 4.5) + rng.normal(0., 1., mz.size))
    inten = inten + np.arange(mz.size) * 1e-9          # distinct intensities (ties are implementation-defined)
    o = np.argsort(mz, kind="stable")
    return np.ascontiguousarray(mz[o]), np.ascontiguousarray(inten[o])


def even_bins(total, n_bins):
    """per-bin peak counts (each <= 10) adding up to `total`"""
    c = np.full(n_bins, total // n_bins)
    c[:total % n_bins] += 1
    assert c.max() <= 10
    return c


class Group:
    """PSMs of one scorer set-up"""

    def __init__(self, name, scorer, neutral_losses=()):
        self.name = name
        self.meta = dict(scorer=dict(scorer), neutral_losses=[list(x) for x in neutral_losses])
        self.psms, self.info = [], []

    def add(self, pep, k, Z, mz, inten, **info):
        self.psms.append(dict(mz=mz, inten=inten, peptide=pep, n_mod=k, max_charge=Z))
        info.update(L=len(pep), k=k, Z=Z, S=sum(c in self.meta["scorer"]["mod_group"] for c in pep))
        self.info.append(info)

    def batch(self):
        return make_golden.batch_from_psms(self.psms)


def _psm(g, rng, L, site_idx, mod_sites, Z, types="by", **kw):
    pep = peptide(rng, L, site_idx, kw.pop("d_idx", ()))
    mz, it = spectrum(rng, ions(pep, [site_idx[j] for j in mod_sites], types, Z))
    g.add(pep, len(mod_sites), Z, mz, it, **kw)


def length_group(neutral_losses=()):
    """peptide lengths 1 .. 126: pa_walk_fast (2 <= L <= 64) against pa_walk_isoform, the second site-mask word (`mhi`)
    in K2 and in K3b's stream set-up, PA_LMAX.  Sites on both sides of residue 64, the true mods past it."""
    rng = np.random.default_rng(64)
    g = Group("length" + ("_nl" if neutral_losses else ""), PHOS, neutral_losses)
    mz, it = spectrum(rng, ions("S", [], "by", 1))
    g.add("S", 1, 2, mz, it)
    mz, it = spectrum(rng, ions("ST", [1], "by", 2))
    g.add("ST", 1, 2, mz, it)
    g.add("SK", 1, 2, mz, it)
    for L in (63, 64, 65, 100, 126):
        sites = [i for i in (5, 30, 60, 62, 63, 64, 66, 70, 95, 120) if i < L]
        for Z in (2, 3):
            _psm(g, rng, L, sites, [len(sites) - 2, len(sites) - 1], Z)
    return g


def sites_group():
    """31 .. 63 modifiable residues, k = 1 and 2, the true sites at index >= 32: 64-bit signatures, pa_unrank,
    alternative sites and best_sequence past bit 31"""
    rng = np.random.default_rng(33)
    g = Group("sites", PHOS)
    for S in (31, 32, 33, 63):
        L = S + 7
        sites = sorted(rng.choice(np.arange(1, L - 1), S, replace=False).tolist())
        for mods in ([S - 1], [S - 4, S - 1]):
            _psm(g, rng, L, sites, mods, 2)
    return g


def peaks_group(bin_size):
    """254 / 255 / 256 (/ 1000) retained peaks: staged (<= PA_RCAP) against global peaks in K2; 7.3-Th bins over
    1500 Th give more than 128 bins, which K1's row form declines"""
    rng = np.random.default_rng(int(bin_size * 10))
    g = Group("peaks_%g" % bin_size, dict(PHOS, bin_size=bin_size))
    hi = {50.: 1500., 10.: 1200., 7.3: 1600.}[bin_size]
    n_bins = int((hi - 100.) // float(np.float32(bin_size))) - 1
    targets = (254, 255, 256) + ((1000,) if bin_size <= 10 else ())
    for t in targets:
        sites = [3, 7, 11, 15, 19, 22]
        pep = peptide(rng, 25, sites)
        mz, it = spectrum(rng, ions(pep, [7, 15], "by", 2), bin_size, 100., hi, per_bin=even_bins(t, n_bins))
        g.add(pep, 2, 2, mz, it, retained=t, n_bins=n_bins)
    return g


def charge_group(neutral_losses=()):
    """max fragment charge 1 .. 39: every K3b stream class (one / two / <= 4 / <= 12 streams), V*Z > 12 into K3c,
    K3c lists longer than PA_LCAP.  The one-residue PSMs have one site, so they are scored (K2, selection) but are
    unambiguous and give the Ascore kernels no work."""
    rng = np.random.default_rng(39)
    g = Group("charge" + ("_nl" if neutral_losses else ""), PHOS, neutral_losses)
    for Z in (1, 2, 3, 4, 5, 12, 13, 39):
        for k in (1, 2):
            _psm(g, rng, 14, [2, 5, 9, 12], [2] if k == 1 else [1, 2], Z)
        mz, it = spectrum(rng, ions("S", [0], "by", Z))
        g.add("T", 1, Z, mz, it)
    return g


def frag_group():
    """fragments per isoform 511 .. 4095 with one ion type ((L-1) * Z), which also grows the score table
    512 -> 1024 -> 2048 -> 4095 inside one call"""
    rng = np.random.default_rng(4095)
    g = Group("fragments", dict(PHOS, fragment_types="b"))
    for L, Z in ((74, 7), (65, 8), (28, 19), (65, 16), (42, 25), (65, 32), (106, 39)):
        sites = [1, L // 3, L // 2, L - 3]
        _psm(g, rng, L, sites, [1, 2], Z, types="b", n_frag=(L - 1) * Z)
    return g


def frag_group_nl():
    """2048 / 2049 fragments with five ion types and one loss-carrying residue D at index p:
    Z * (2 * (2m - p) + 3 * (m + p)) = Z * (7m + p) with m = L - 1"""
    rng = np.random.default_rng(2049)
    g = Group("fragments_nl", dict(PHOS, fragment_types="bcyzZ"), [("D", 18.010565)])
    for L, p, Z in ((74, 1, 4), (98, 4, 3)):
        sites = [10, 20, 30, L - 5]
        m = L - 1
        _psm(g, rng, L, sites, [0, 3], Z, types="bcyzZ", d_idx=(p,), n_frag=Z * (7 * m + p))
    return g


def isoform_group():
    """253 / 276, 496 / 528, 1001 / 1035 and 2002 isoforms per PSM (C(S, k) straddling PA_SORTCAP, PA_SEL_THREAD_MAX and
    PA_UNIT), with neutral losses and charge 3.  The best isoform is only picked by replaying std::sort when the top
    weighted score is tied -- in shared memory up to PA_SORTCAP isoforms, in global memory beyond -- so the PSMs at
    253 / 276 / 496 / 528 isoforms come again on a spectrum of two peaks far above every fragment (every isoform
    scores the same, as in make_golden.edge_cases)."""
    rng = np.random.default_rng(1025)
    g = Group("isoforms", PHOS, [("ST", 18.01528), ("st", 97.9769)])
    for S, k in ((23, 2), (24, 2), (32, 2), (33, 2), (14, 4), (46, 2), (14, 5)):
        L = S + 6
        sites = sorted(rng.choice(np.arange(1, L - 1), S, replace=False).tolist())
        _psm(g, rng, L, sites, list(range(S // 2, S // 2 + k)), 3)
    for S, k in ((23, 2), (24, 2), (32, 2), (33, 2)):
        L = S + 6
        sites = sorted(rng.choice(np.arange(1, L - 1), S, replace=False).tolist())
        g.add(peptide(rng, L, sites), k, 3, np.array([20000., 20001.]), np.array([1., 2.]), tied=True)
    return g


def dense_group():
    """4095 fragments per isoform at mz_error 1.5 on ~3000 retained peaks: most fragments match, the per-rank counts
    come near the 12-bit fields K2 packs them in"""
    rng = np.random.default_rng(12)
    g = Group("dense", dict(PHOS, fragment_types="b", mz_error=1.5, bin_size=10.))
    L, Z = 106, 39
    sites = [20, 50, 80]
    pep = peptide(rng, L, sites)
    mz, it = spectrum(rng, ions(pep, [50], "b", Z), 10., 0., 3000., per_bin=np.full(299, 10))
    g.add(pep, 1, Z, mz, it, n_frag=(L - 1) * Z)
    return g


def status_group():
    """inputs the library refuses per PSM (include/pyascore_b200.h: pa_psm_status) next to the largest accepted ones"""
    rng = np.random.default_rng(127)
    g = Group("status", dict(PHOS, fragment_types="b"))
    cases = [  # (L, sites, k, Z, status)
        (126, [3, 100], 1, 1, 0), (127, [3, 100], 1, 1, 2),
        (70, list(range(2, 65)), 1, 1, 0), (70, list(range(2, 66)), 1, 1, 3),
        (106, [3, 50], 1, 39, 0), (107, [3, 50], 1, 39, 8), (65, [3, 50], 1, 64, 8),
        (70, list(range(2, 65)), 6, 1, 4),        # C(63, 6) = 67 945 521 > 2^26
    ]
    for L, sites, k, Z, st in cases:
        pep = peptide(rng, L, sites)
        mz, it = spectrum(rng, ions(pep, sites[:k], "b", min(Z, 3)))
        g.add(pep, k, Z, mz, it, status=st)
    return g


def fragments_per_isoform(pep, state, types, Z, nl):
    """closed form of the theoretical fragments of one isoform (cpp/ModifiedPeptide.cpp:379-408, :500-524):
    per ion type, the sum over the L - 1 residue steps of its walk of the number of distinct sums of at most two of the
    losses passed so far (0 included) -- on a one-residue peptide one step with one variant fewer -- times Z.
    `state[i]` = 1 where residue i carries the variable mod; `nl` maps a letter (lower case: modified) to its loss."""
    L = len(pep)
    total = 0
    for t in types:
        order = range(L) if t in "bc" else range(L - 1, -1, -1)
        stack, n = [], 0
        for step, i in enumerate(order):
            if step == max(L - 1, 1):
                break
            key = pep[i].lower() if state[i] else pep[i]
            if nl.get(key, 0.) != 0.:
                stack.append(np.float32(nl[key]))
            sums = {np.float32(0.)}
            for a in range(len(stack)):
                s1 = np.float32(0.) + stack[a]
                sums.add(s1)
                for b2 in range(a + 1, len(stack)):
                    sums.add(np.float32(s1 + stack[b2]))
            n += len(sums) - (1 if L == 1 else 0)
        total += n * Z
    return total



# ---- deep peak depths (n_top 11 .. 64).  The groups above hold at most 10 peaks per bin (even_bins) or a handful per
# 100-Th bin (spectrum()), so at n_top > 10 they would give no rank >= 10 and K2d would only ever add zeros.  The helpers
# below give a built group's spectra denser bins from their own generator; the groups above keep their draws.
def at_n_top(g, n_top):
    """group `g` scored at peak depth `n_top` (the scorer set-up with n_top overridden, the same PSMs)"""
    out = Group(g.name, dict(g.meta["scorer"], n_top=n_top), g.meta["neutral_losses"])
    out.psms, out.info = list(g.psms), list(g.info)
    return out


def densify_spectrum(rng, mz, inten, bin_size, n_top, cap=None, stronger=True):
    """(mz, inten) with peaks added to the bins that hold peaks (bins as the reference counts them: from the spectrum's
    lowest m/z rounded down to a multiple of 100), from the lowest bin up, until each holds 11 .. n_top peaks.  The added
    peaks are stronger than every peak already in their bin, so those (the ions among them) move down by the number
    added -- ten or more where n_top leaves room -- to ranks >= 10.  Half the bins stay within five peaks of that, so
    that ions sit at depths near 10 as well as further down.  `cap`: stop before the retained peaks of the
    spectrum pass it.  stronger=False: the added peaks are weaker than those in their bin instead (the ions keep their
    ranks, the added peaks take 10 .. n_top-1).  Spectra of fewer than three peaks stay as they are."""
    if mz.size < 3:
        return mz, inten
    bs = float(np.float32(bin_size))
    lo, hi = np.floor(mz.min() / 100.) * 100., np.ceil(mz.max() / 100.) * 100.
    nb = int(np.ceil(np.float32((hi - lo) / bs)))
    b = np.minimum(np.floor((mz - lo) / bs).astype(np.int64), nb - 1)
    count = np.bincount(b, minlength=nb)
    retained = int(np.minimum(count, n_top).sum())
    add_mz, add_it = [mz], [inten]
    for q in np.flatnonzero((count > 0) & (count < n_top)):
        c = int(count[q])
        low = max(11, c + 10 if c + 10 <= n_top else c + 1)
        want = int(rng.integers(low, (n_top if rng.random() < 0.5 else min(n_top, low + 5)) + 1))
        if cap is not None and retained + want - c > cap:
            break
        a0 = lo + q * bs + 0.02 * bs
        a1 = min(lo + (q + 1) * bs, hi) - 0.02 * bs
        add_mz.append(rng.uniform(a0, a1, want - c))
        f = np.exp(rng.uniform(0.01, 2., want - c))
        add_it.append(inten[b == q].max() * f if stronger else inten[b == q].min() / f)
        retained += want - c
    mz, inten = np.concatenate(add_mz), np.concatenate(add_it)
    assert np.unique(inten).size == inten.size                  # distinct intensities (ties are implementation-defined)
    o = np.argsort(mz, kind="stable")
    return np.ascontiguousarray(mz[o]), np.ascontiguousarray(inten[o])


def densify(g, n_top, seed, cap=None, stronger=True):
    """group `g` at peak depth `n_top` on densified spectra (densify_spectrum, generator seeded by (seed, n_top))"""
    rng = np.random.default_rng([seed, n_top])
    out = at_n_top(g, n_top)
    bs = g.meta["scorer"]["bin_size"]
    out.psms = []
    for p in g.psms:
        mz, it = densify_spectrum(rng, p["mz"], p["inten"], bs, n_top, cap, stronger)
        out.psms.append(dict(p, mz=mz, inten=it))
    return out


def densify_batch(batch, bin_size, n_top, seed):
    """densify_spectrum over every spectrum of a CSR batch"""
    rng = np.random.default_rng([seed, n_top])
    off = batch["spec_off"]
    parts = [densify_spectrum(rng, batch["mz"][off[q]:off[q + 1]], batch["inten"][off[q]:off[q + 1]], bin_size, n_top)
             for q in range(off.size - 1)]
    out = dict(batch)
    out["mz"] = np.ascontiguousarray(np.concatenate([m for m, _ in parts]))
    out["inten"] = np.ascontiguousarray(np.concatenate([i for _, i in parts]))
    out["spec_off"] = np.concatenate([[0], np.cumsum([m.size for m, _ in parts])]).astype(np.int64)
    return out


def add_one_residue_deep(g, rng, letter="S", Z=2):
    """a one-residue PSM (k = 1) whose fragments (every loss variant of the group) sit at ranks 12 .. 13 of their bins:
    twelve stronger peaks away from them fill each bin.  Only K2d's one-step walk (L = 1) counts these matches."""
    m = _MASS[letter] + 79.966331
    losses = [0.] + [mass for grp, mass in g.meta["neutral_losses"] if letter.lower() in grp]
    ion = []
    for t in g.meta["scorer"]["fragment_types"]:          # as ions(): residue sum + the ion type's shift
        for nl in losses:
            for z in range(1, Z + 1):
                ion.append((m + _ION_SHIFT[t] - nl + z * 1.007825) / z)
    ion = np.unique(np.round(np.array(ion), 4))
    bs = float(np.float32(g.meta["scorer"]["bin_size"]))
    mz, it = [ion + rng.normal(0., 0.05, ion.size)], [np.exp(3. + rng.random(ion.size))]
    for q in np.unique(np.floor(ion / bs)):
        a0, a1 = q * bs, (q + 1) * bs
        cand = rng.uniform(a0 + 0.02 * bs, a1 - 0.02 * bs, 200)
        cand = cand[np.min(np.abs(cand[:, None] - ion[None, :]), axis=1) > 3.][:12]
        assert cand.size == 12
        mz.append(cand)
        it.append(np.exp(8. + rng.random(12)))
    mz, it = np.concatenate(mz), np.concatenate(it)
    o = np.argsort(mz)
    g.add(letter, 1, Z, np.ascontiguousarray(mz[o]), np.ascontiguousarray(it[o]), one_residue_deep=True)


def deep_peaks_group(n_top):
    """254 / 255 / 256 retained peaks (straddling PA_RCAP) from 18 bins of 100 Th holding 14 or 15 peaks each, i.e. more
    than ten retained peaks per bin, at peak depth n_top (>= 15)"""
    rng = np.random.default_rng(2550 + n_top)
    g = Group("peaks_deep", dict(PHOS, n_top=n_top))
    n_bins = 18
    for t in (254, 255, 256):
        sites = [3, 7, 11, 15, 19, 22]
        pep = peptide(rng, 25, sites)
        per_bin = np.full(n_bins, t // n_bins)
        per_bin[:t % n_bins] += 1
        assert 10 < per_bin.min() and per_bin.max() <= n_top
        mz, it = spectrum(rng, ions(pep, [7, 15], "by", 2), 100., 100., 100. + 100. * n_bins, per_bin=per_bin)
        g.add(pep, 2, 2, mz, it, retained=t, n_bins=n_bins)
    return g


# the deep cases of tests/test_gpu_deep_limits.py (GPU against the oracle) and tests/test_oracle_deep_limits.py (their
# reach, on the oracle alone)
DEEP_SEED = 1164


def deep_group(name, n_top):
    """the shape group `name` at peak depth n_top with bins of 11 .. n_top peaks.  The length groups stay within PA_RCAP
    retained peaks (their proof needs staged peaks), sites keeps its ions at the top ranks (its proof needs the true
    sites past index 31 to stay the best isoform's), and length_nl gets a one-residue PSM matched at deep ranks."""
    if name == "peaks_deep":
        return deep_peaks_group(n_top)
    build = {"length": length_group, "length_nl": lambda: length_group([("st", 97.9769)]), "sites": sites_group,
             "charge_nl": lambda: charge_group([("ST", 18.01528)]), "fragments": frag_group,
             "fragments_nl": frag_group_nl, "isoforms": isoform_group, "dense": dense_group}[name]
    g = densify(build(), n_top, DEEP_SEED, cap=RCAP if name.startswith("length") else None, stronger=name != "sites")
    if name == "length_nl":
        add_one_residue_deep(g, np.random.default_rng([DEEP_SEED, n_top, 1]))
    return g


DEEP_SHAPES = [(n, t) for n in ("length", "length_nl", "sites", "charge_nl", "fragments", "fragments_nl", "isoforms",
                                "dense") for t in (20, 64)] + [("peaks_deep", 20), ("peaks_deep", 40)]

# the shape cases none of whose Ascores is taken at a depth >= 10 (every group but dense has one that is: in dense,
# mz_error 1.5 over 10-Th bins, every 3-Th window holds peaks of rank < 10 and the score differences peak shallow)
DEEP_SHALLOW_ASCORES = {("sites", 20), ("fragments_nl", 64), ("dense", 20), ("dense", 64)}

# variant matrix at depth: every VARIANTS set-up at n_top 20, then the first set-up of each k_count_score
# instantiation at 64
DEEP_MATRIX = [(q, 20) for q in range(len(VARIANTS))] + \
    [(q, 64) for q in sorted({k2_instantiation(*v): i for i, v in reversed(list(enumerate(VARIANTS)))}.values())]


def deep_variant_case(q, n_top):
    """(meta, batch) of variant q at n_top: 160 synthetic PSMs (7..20 residues, charges 1..2) on densified spectra"""
    from pyascore_b200 import synth
    ftypes, err, nl = VARIANTS[q]
    w = dict(synth.WORKLOADS["lowres_phospho"], L=(7, 20), neutral_losses=nl,
             scorer=dict(PHOS, fragment_types=ftypes, mz_error=err, n_top=n_top))
    batch = synth.make_batch(w, 160, seed=2026, chunk_index=q)
    return dict(scorer=w["scorer"], neutral_losses=nl), densify_batch(batch, 100., n_top, DEEP_SEED + q)
