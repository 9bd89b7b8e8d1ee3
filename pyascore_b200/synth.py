"""Seeded synthetic PSM/spectrum batches in the CSR layout `score_batch` consumes.

The workloads are the ones BASELINE.json / SURVEY.md section 8(d) name (configs 2-5).  There is no
network for real data sets, so every benchmark and most parity tests run on these; the
generator is vectorised numpy so that a 1M-PSM batch is produced chunk by chunk from
`(seed, chunk_index)` without ever being materialised at once.

Batch layout (host numpy, all C-contiguous):
    spec_off  int64 [n_spec+1]   peak range of each spectrum in mz/inten
    mz, inten float64[n_peaks]   m/z sorted ascending inside a spectrum, intensities distinct
    psm_spec  int32 [n_psm]      spectrum index of each PSM (several PSMs may share one)
    pep_off   int32 [n_psm+1]    byte range of each peptide in pep
    pep       uint8 []           upper-case residue letters
    n_mod     int32 [n_psm]      number of unlocalised (variable) mods
    max_charge int32[n_psm]      max fragment charge (reference: min(cli_max, z-1), __main__.py:150-157)
    aux_off   int32 [n_psm+1]    range of fixed mods in aux_pos/aux_mass
    aux_pos   uint32[]           0 = N-term, else 1-based residue index
    aux_mass  float32[]
"""
import numpy as np

# float64 copies of the reference residue table (cpp/Types.h:7-30); only used to PLACE
# synthetic peaks near theoretical ions -- never for scoring.
_MASS = {'G': 57.02146, 'A': 71.03711, 'S': 87.03203, 'P': 97.05276, 'V': 99.06841, 'T': 101.04768,
         'C': 103.00919, 'L': 113.08406, 'I': 113.08406, 'N': 114.04293, 'D': 115.02694, 'Q': 128.05858,
         'K': 128.09496, 'E': 129.04259, 'M': 131.04049, 'H': 137.05891, 'F': 147.06841, 'U': 150.95364,
         'R': 156.10111, 'Y': 163.06333, 'W': 186.07931, 'O': 237.14773}
_MASS_LUT = np.zeros(256, np.float64)
for _c, _m in _MASS.items():
    _MASS_LUT[ord(_c)] = _m

WORKLOADS = {
    # config 2: low-res ion-trap phospho
    "lowres_phospho": dict(
        scorer=dict(bin_size=100., n_top=10, mod_group="STY", mod_mass=79.966331, mz_error=0.5,
                    fragment_types="by"), neutral_losses=[],
        alphabet="ADEFGHIKLMNPQRVW", site_alphabet="STY", L=(7, 30), k_vals=(1, 2, 3), k_p=(.6, .3, .1),
        max_sites=10, unamb_frac=0.05, z_vals=(2, 3), z_p=(.6, .4), max_frag_charge=99,
        jitter=0.15, keep_p=0.6, noise=(100, 400), nl_peak_p=0.0, hits=1, aux=None),
    # config 3: high-res HCD phospho with st neutral loss
    "hires_phospho_nl": dict(
        scorer=dict(bin_size=100., n_top=10, mod_group="STY", mod_mass=79.966331, mz_error=0.02,
                    fragment_types="by"), neutral_losses=[("st", 97.9769)],
        alphabet="ADEFGHIKLMNPQRVW", site_alphabet="STY", L=(7, 30), k_vals=(1, 2, 3), k_p=(.6, .3, .1),
        max_sites=10, unamb_frac=0.05, z_vals=(2, 3, 4), z_p=(.5, .35, .15), max_frag_charge=2,
        jitter=0.004, keep_p=0.6, noise=(100, 400), nl_peak_p=0.3, hits=1, aux=None),
    # config 4: combinatorial stress, C(20,5) = 15504 isoforms per PSM
    "stress": dict(
        scorer=dict(bin_size=100., n_top=10, mod_group="STY", mod_mass=79.966331, mz_error=0.5,
                    fragment_types="by"), neutral_losses=[],
        alphabet="ADEFGHIKLMNPQRVW", site_alphabet="STY", L=(40, 40), k_vals=(5,), k_p=(1.,),
        max_sites=20, fixed_sites=20, unamb_frac=0.0, z_vals=(2,), z_p=(1.,), max_frag_charge=1,
        jitter=0.15, keep_p=0.6, noise=(2000, 2000), total_peaks=2000, nl_peak_p=0.0, hits=1, aux=None),
    # config 5: acetyl-K with static carbamidomethyl C, 3 PSMs per spectrum
    "acetyl_k": dict(
        scorer=dict(bin_size=100., n_top=10, mod_group="K", mod_mass=42.0106, mz_error=0.02,
                    fragment_types="by"), neutral_losses=[],
        alphabet="ACDEFGHILMNPQRSTVWY", site_alphabet="K", L=(7, 30), k_vals=(1, 2, 3), k_p=(.6, .3, .1),
        max_sites=10, unamb_frac=0.05, z_vals=(2, 3, 4), z_p=(.5, .35, .15), max_frag_charge=3,
        jitter=0.004, keep_p=0.6, noise=(100, 400), nl_peak_p=0.0, hits=3, aux=("C", 57.021464)),
}


def _ranks(keys):
    """rank of every element inside its row (0 = smallest key)"""
    order = np.argsort(keys, axis=1, kind="stable")
    r = np.empty_like(order)
    np.put_along_axis(r, order, np.arange(keys.shape[1])[None, :].repeat(keys.shape[0], 0), axis=1)
    return r


def _peptides(rng, w, n):
    """-> residues uint8 (n, Lmax), L, k, site mask, true modified mask"""
    Lmin, Lmax = w["L"]
    L = rng.integers(Lmin, Lmax + 1, size=n)
    k = rng.choice(np.asarray(w["k_vals"]), size=n, p=np.asarray(w["k_p"]))
    if w.get("fixed_sites"):
        S = np.full(n, w["fixed_sites"])
    else:
        hi = np.minimum(w["max_sites"], L)
        S = k + 1 + (rng.random(n) * np.maximum(hi - k, 1)).astype(np.int64)
        S = np.minimum(S, hi)
        unamb = rng.random(n) < w["unamb_frac"]
        S = np.where(unamb, k, S)
        S = np.maximum(S, np.minimum(k, L))
    pos = np.arange(Lmax)[None, :]
    valid = pos < L[:, None]
    alpha = np.frombuffer(w["alphabet"].encode(), np.uint8)
    salpha = np.frombuffer(w["site_alphabet"].encode(), np.uint8)
    res = alpha[rng.integers(0, alpha.size, size=(n, Lmax))]
    key = rng.random((n, Lmax))
    key[~valid] = 2.0
    site = (_ranks(key) < S[:, None]) & valid
    res = np.where(site, salpha[rng.integers(0, salpha.size, size=(n, Lmax))], res)
    res = np.where(valid, res, 0).astype(np.uint8)
    key2 = rng.random((n, Lmax))
    key2[~site] = 2.0
    modified = (_ranks(key2) < k[:, None]) & site
    return res, L, k.astype(np.int32), site, modified


def make_batch(workload, n_psm, seed=20261017, chunk_index=0, return_truth=False):
    """Generate `n_psm` PSMs (n_psm // hits spectra) of the named workload."""
    w = WORKLOADS[workload] if isinstance(workload, str) else workload
    rng = np.random.default_rng([seed, chunk_index])
    hits = w["hits"]
    n_spec = max(n_psm // hits, 1)
    n_psm = n_spec * hits
    res, L, k, site, modified = _peptides(rng, w, n_spec)
    Lmax = res.shape[1]
    z = rng.choice(np.asarray(w["z_vals"]), size=n_spec, p=np.asarray(w["z_p"]))
    zf = np.minimum(w["max_frag_charge"], z - 1).astype(np.int32)
    Zmax = int(zf.max())

    # neutral masses of the true isoform's b / y ions
    m = _MASS_LUT[res]
    m = m + modified * w["scorer"]["mod_mass"]
    if w["aux"]:
        m = m + (res == ord(w["aux"][0])) * w["aux"][1]
    b = np.cumsum(m, axis=1)                                   # b_i = sum(res[0..i])
    tot = b[np.arange(n_spec), L - 1]
    y = tot[:, None] - b + 18.010565                           # y after cleaving bond i: res[i+1..]
    frag_ok = np.arange(Lmax)[None, :] < (L - 1)[:, None]
    sig = []
    sig_ok = []
    for ions, nl_count in ((b, np.cumsum(modified & np.isin(res, [83, 84]), axis=1)),
                           (y, (modified & np.isin(res, [83, 84])).sum(1)[:, None]
                            - np.cumsum(modified & np.isin(res, [83, 84]), axis=1))):
        for zz in range(1, Zmax + 1):
            ok = frag_ok & (zf >= zz)[:, None] & (rng.random((n_spec, Lmax)) < w["keep_p"])
            sig.append((ions + zz * 1.007825) / zz + rng.normal(0., w["jitter"], size=(n_spec, Lmax)))
            sig_ok.append(ok)
            if w["nl_peak_p"] > 0:
                for (_, nl_mass) in w["neutral_losses"]:
                    ok2 = frag_ok & (zf >= zz)[:, None] & (nl_count > 0) & (rng.random((n_spec, Lmax)) < w["nl_peak_p"])
                    sig.append((ions - nl_mass + zz * 1.007825) / zz
                               + rng.normal(0., w["jitter"], size=(n_spec, Lmax)))
                    sig_ok.append(ok2)
    sig = np.concatenate(sig, axis=1)
    sig_ok = np.concatenate(sig_ok, axis=1) & (sig > 50.)
    n_sig = sig_ok.sum(1)

    lo, hi = w["noise"]
    n_noise = rng.integers(lo, hi + 1, size=n_spec)
    if w.get("total_peaks"):
        n_noise = np.maximum(w["total_peaks"] - n_sig, 0)
    Nmax = int(n_noise.max())
    noise = rng.uniform(150., 2000., size=(n_spec, Nmax))
    noise_ok = np.arange(Nmax)[None, :] < n_noise[:, None]

    # one sortable key per peak: m/z with the lowest mantissa bit = "is signal"
    allmz = np.concatenate([sig, noise], axis=1)
    bits = allmz.view(np.uint64)
    bits &= ~np.uint64(1)
    bits[:, :sig.shape[1]] |= np.uint64(1)
    allmz[~np.concatenate([sig_ok, noise_ok], axis=1)] = np.inf
    allmz.sort(axis=1)
    cnt = (n_sig + n_noise).astype(np.int64)
    keep = np.arange(allmz.shape[1])[None, :] < cnt[:, None]
    mz = allmz[keep]
    is_sig = (mz.view(np.uint64) & np.uint64(1)).astype(bool)
    inten = np.exp(np.where(is_sig, 6.0, 4.5) + rng.normal(0., 1., size=mz.size))
    spec_off = np.zeros(n_spec + 1, np.int64)
    np.cumsum(cnt, out=spec_off[1:])
    # intensities must be distinct inside a spectrum (ties are implementation-defined in the
    # reference: SURVEY.md section 7.3); continuous draws collide with probability ~0, but make sure
    sid = np.repeat(np.arange(n_spec), cnt)
    o = np.lexsort((inten, sid))
    dup = (np.diff(inten[o]) == 0) & (np.diff(sid[o]) == 0)
    while dup.any():
        idx = o[1:][dup]
        inten[idx] = np.nextafter(inten[idx], np.inf)
        o = np.lexsort((inten, sid))
        dup = (np.diff(inten[o]) == 0) & (np.diff(sid[o]) == 0)

    # PSMs: hit 0 = the generating peptide, further hits = unrelated peptides on the same spectrum
    if hits > 1:
        res_all = np.zeros((n_spec, hits, Lmax), np.uint8)
        L_all = np.zeros((n_spec, hits), np.int64)
        k_all = np.zeros((n_spec, hits), np.int32)
        res_all[:, 0], L_all[:, 0], k_all[:, 0] = res, L, k
        for h in range(1, hits):
            r2, L2, k2, _, _ = _peptides(rng, w, n_spec)
            res_all[:, h], L_all[:, h], k_all[:, h] = r2, L2, k2
        res_p = res_all.reshape(n_psm, Lmax)
        L_p = L_all.reshape(n_psm)
        k_p = k_all.reshape(n_psm)
    else:
        res_p, L_p, k_p = res, L, k
    psm_spec = np.repeat(np.arange(n_spec, dtype=np.int32), hits)
    pep_off = np.zeros(n_psm + 1, np.int32)
    np.cumsum(L_p, out=pep_off[1:])
    pep = res_p[np.arange(Lmax)[None, :] < L_p[:, None]]
    if w["aux"]:
        is_aux = (res_p == ord(w["aux"][0])) & (np.arange(Lmax)[None, :] < L_p[:, None])
        aux_off = np.zeros(n_psm + 1, np.int32)
        np.cumsum(is_aux.sum(1), out=aux_off[1:])
        aux_pos = (np.nonzero(is_aux)[1] + 1).astype(np.uint32)
        aux_mass = np.full(aux_pos.size, w["aux"][1], np.float32)
    else:
        aux_off = np.zeros(n_psm + 1, np.int32)
        aux_pos = np.zeros(0, np.uint32)
        aux_mass = np.zeros(0, np.float32)
    batch = dict(spec_off=spec_off, mz=np.ascontiguousarray(mz), inten=inten, psm_spec=psm_spec,
                 pep_off=pep_off, pep=np.ascontiguousarray(pep), n_mod=np.ascontiguousarray(k_p, np.int32),
                 max_charge=np.repeat(zf, hits).astype(np.int32), aux_off=aux_off, aux_pos=aux_pos,
                 aux_mass=aux_mass)
    if return_truth:
        return batch, dict(modified=modified, site=site, L=L)
    return batch


def concat_batches(batches):
    """Concatenate CSR batches (offsets rebased)."""
    out = {}
    specs = 0
    peaks = 0
    peps = 0
    auxs = 0
    acc = {k: [] for k in batches[0]}
    for b in batches:
        acc["spec_off"].append(b["spec_off"][:-1] + peaks)
        acc["psm_spec"].append(b["psm_spec"] + specs)
        acc["pep_off"].append(b["pep_off"][:-1] + peps)
        acc["aux_off"].append(b["aux_off"][:-1] + auxs)
        for k in ("mz", "inten", "pep", "n_mod", "max_charge", "aux_pos", "aux_mass"):
            acc[k].append(b[k])
        specs += b["spec_off"].size - 1
        peaks += int(b["spec_off"][-1])
        peps += int(b["pep_off"][-1])
        auxs += int(b["aux_off"][-1])
    acc["spec_off"].append(np.array([peaks], np.int64))
    acc["pep_off"].append(np.array([peps], np.int32))
    acc["aux_off"].append(np.array([auxs], np.int32))
    for k, v in acc.items():
        out[k] = np.ascontiguousarray(np.concatenate(v))
    out["psm_spec"] = out["psm_spec"].astype(np.int32)
    return out


def batch_nbytes(batch):
    return int(sum(v.nbytes for v in batch.values()))


def psm_view(batch, i):
    """(mz, inten, peptide str, n_mod, max_charge, aux_pos, aux_mass) of PSM i -- what PyAscore.score takes"""
    s = int(batch["psm_spec"][i])
    a, b = int(batch["spec_off"][s]), int(batch["spec_off"][s + 1])
    pep = bytes(batch["pep"][batch["pep_off"][i]:batch["pep_off"][i + 1]]).decode()
    x, y = int(batch["aux_off"][i]), int(batch["aux_off"][i + 1])
    return (batch["mz"][a:b], batch["inten"][a:b], pep, int(batch["n_mod"][i]), int(batch["max_charge"][i]),
            batch["aux_pos"][x:y], batch["aux_mass"][x:y])


def _ragged(off, rows):
    """indices into the data of a CSR array for rows `rows`, and their offsets"""
    lens = (off[1:] - off[:-1])[rows].astype(np.int64)
    new_off = np.zeros(rows.size + 1, np.int64)
    np.cumsum(lens, out=new_off[1:])
    return np.repeat(off[:-1][rows].astype(np.int64) - new_off[:-1], lens) + np.arange(new_off[-1]), new_off


def select_rows(batch, rows, n_mod=None):
    """host batch of PSM rows `rows` of `batch` (in that order, repeats allowed) over the same spectra arrays; n_mod:
    the rows' n_mod (default: theirs)"""
    rows = np.asarray(rows, np.int64)
    out = {k: batch[k] for k in ("spec_off", "mz", "inten", "inten32") if k in batch}
    out["psm_spec"] = np.ascontiguousarray(batch["psm_spec"][rows])
    idx, off = _ragged(batch["pep_off"], rows)
    out["pep"], out["pep_off"] = np.ascontiguousarray(batch["pep"][idx]), off.astype(np.int32)
    idx, off = _ragged(batch["aux_off"], rows)
    out["aux_pos"], out["aux_mass"] = np.ascontiguousarray(batch["aux_pos"][idx]), np.ascontiguousarray(batch["aux_mass"][idx])
    out["aux_off"] = off.astype(np.int32)
    out["n_mod"] = np.ascontiguousarray(batch["n_mod"][rows] if n_mod is None else np.asarray(n_mod, np.int32))
    out["max_charge"] = np.ascontiguousarray(batch["max_charge"][rows])
    return out


def typed_batch(batch, groups, skip_below=0):
    """A batch of several modification types (pyascore_b200.score_typed) over the spectra of `batch`: type 0 = every
    PSM of `batch`; type t >= 1 = for every PSM at index >= skip_below whose peptide has a letter of groups[t-1], a row
    on the same spectrum with one such modification, right after the PSM's rows of the types before (psm_spec stays
    non-decreasing).  -> (batch, psm_type uint8)"""
    n = batch["n_mod"].size
    pep, off = batch["pep"], batch["pep_off"]
    rows, n_mod, typ = [np.arange(n)], [batch["n_mod"]], [np.zeros(n, np.uint8)]
    for t, letters in enumerate(groups, start=1):
        cs = np.concatenate([[0], np.cumsum(np.isin(pep, np.frombuffer(letters.encode(), np.uint8)))])
        r = np.flatnonzero((cs[off[1:]] - cs[off[:-1]] > 0) & (np.arange(n) >= skip_below))
        rows.append(r); n_mod.append(np.ones(r.size, np.int32)); typ.append(np.full(r.size, t, np.uint8))
    rows, n_mod, typ = np.concatenate(rows), np.concatenate(n_mod), np.concatenate(typ)
    order = np.lexsort((typ, rows))
    return select_rows(batch, rows[order], n_mod[order]), np.ascontiguousarray(typ[order])
