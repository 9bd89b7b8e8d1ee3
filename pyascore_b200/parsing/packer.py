"""PSM records + spectra -> CSR batches for `Scorer.score_batch`, and results -> TSV rows.

This replaces the body of the reference's per-PSM loop (pyascore/__main__.py:129-164): the
grouping by scan, `hit_depth`, the variable/fixed split of `process_mods` (:83-103) and the
fragment-charge rule (:138-145, :155-156) are applied while packing; scoring then happens once per
chunk on the GPU instead of once per PSM.  Spectra are never copied: every chunk refers to the
file-wide CSR block built by `SpectraParser.to_csr()` through `psm_spec`.
"""
import queue
import threading
from itertools import groupby

import numpy as np


def process_mods(residues, mod_mass, mod_correction_tol, zero_based, sequence, positions, masses):
    """reference: __main__.py:83-103 -> (fixed positions u32[], fixed masses f32[], n variable mods)"""
    n_variable = 0
    const_pos, const_mass = [], []
    shift = 1 if zero_based else 0
    for pos, mass in zip(positions, masses):
        pos = int(pos)
        aa = "n" if pos + shift == 0 else sequence[pos - 1 + shift]
        if np.isclose(mod_mass, mass, rtol=1e-6, atol=mod_correction_tol) and aa in residues:
            n_variable += 1
        else:
            const_pos.append(pos + shift)
            const_mass.append(mass)
    return np.array(const_pos, dtype=np.uint32), np.array(const_mass, dtype=np.float32), n_variable


def fragment_charge(match_charge, precursor_charge, max_fragment_charge):
    """reference: __main__.py:138-145 + :155-156"""
    if match_charge is not None and match_charge != 0:
        z = match_charge
    elif precursor_charge is not None and precursor_charge != 0:
        z = precursor_charge
    else:
        z = 2
    return min(max_fragment_charge, max(int(z), 2) - 1)


class PsmPacker:
    """Accumulates the PSMs that will be scored (n_variable > 0) of scan-sorted match records.

    `types` (default: the one type (residues, mod_mass)) lists the (residues, mod_mass) of every modification type of
    a typed batch (`score_typed`): a record added as type t is split by process_mods with types[t], and with more
    than one type every flushed batch carries `psm_type` (uint8, one per row)."""

    def __init__(self, spectra, residues="STY", mod_mass=79.966331, mod_correction_tol=1., zero_based=False,
                 max_fragment_charge=5, hit_depth=1, types=None):
        self.spectra = spectra
        self.types = list(types) if types is not None else [(residues, mod_mass)]
        self.residues, self.mod_mass = self.types[0]
        self.tol = mod_correction_tol
        self.zero_based, self.max_z, self.hit_depth = zero_based, max_fragment_charge, hit_depth
        self._reset()

    def _reset(self):
        self.scans, self.psm_spec, self.peps, self.n_mod, self.max_charge = [], [], [], [], []
        self.aux_pos, self.aux_mass, self.psm_type = [], [], []

    def __len__(self):
        return len(self.scans)

    def add(self, match, t=0):
        """pack one PSM record as type t; returns True when it carries variable mods of that type (i.e. will be
        scored)"""
        idx = self.spectra.index_of(match["scan"])
        if idx < 0:
            raise KeyError(match["scan"])            # the reference indexes spectra_map[scan] (:133)
        residues, mod_mass = self.types[t]
        cpos, cmass, n_var = process_mods(residues, mod_mass, self.tol, self.zero_based,
                                          match["peptide"], match["mod_positions"], match["mod_masses"])
        if n_var <= 0:
            return False
        self.psm_type.append(t)
        self.scans.append(int(match["scan"]))
        self.psm_spec.append(idx)
        self.peps.append(match["peptide"].encode("ascii"))
        self.n_mod.append(n_var)
        self.max_charge.append(fragment_charge(match["charge_state"], int(self.spectra.precursor_charge[idx]),
                                               self.max_z))
        self.aux_pos.append(cpos)
        self.aux_mass.append(cmass)
        return True

    def add_scan_sorted(self, psms):
        """the reference's double loop: group by scan, keep the first `hit_depth` hits of each group
        (hit_depth < 0: all of them)"""
        for _, group in groupby(psms, lambda m: m["scan"]):
            for ind, match in enumerate(group):
                if ind == self.hit_depth:
                    break
                self.add(match)

    def flush(self):
        """-> (scan numbers, batch dict) of everything added since the last flush"""
        n = len(self.scans)
        pep_off = np.zeros(n + 1, np.int32)
        np.cumsum([len(p) for p in self.peps], out=pep_off[1:])
        aux_off = np.zeros(n + 1, np.int32)
        np.cumsum([a.size for a in self.aux_pos], out=aux_off[1:])
        sp = self.spectra
        batch = dict(
            spec_off=sp.spec_off, mz=sp.mz, **({"inten": sp.inten} if sp.inten is not None else {"inten32": sp.inten32}),
            psm_spec=np.array(self.psm_spec, np.int32), pep_off=pep_off,
            pep=np.frombuffer(b"".join(self.peps), np.uint8).copy() if n else np.zeros(0, np.uint8),
            n_mod=np.array(self.n_mod, np.int32), max_charge=np.array(self.max_charge, np.int32), aux_off=aux_off,
            aux_pos=np.concatenate(self.aux_pos).astype(np.uint32) if n else np.zeros(0, np.uint32),
            aux_mass=np.concatenate(self.aux_mass).astype(np.float32) if n else np.zeros(0, np.float32))
        if len(self.types) > 1:
            batch["psm_type"] = np.array(self.psm_type, np.uint8)
        scans = np.array(self.scans, np.int64)
        self._reset()
        return scans, batch


def iter_batches(spectra, psms, chunk_psms=65536, **packer_kw):
    """scan-sorted PSM records -> (scans, batch) chunks cut on scan boundaries.

    With `types` of more than one entry (see PsmPacker), `psms` holds one scan-sorted record list per type -- the
    same identifications, mass-corrected for that type -- and every scan contributes its hit_depth hits of type 0,
    then those of type 1, and so on: psm_spec stays non-decreasing."""
    packer = PsmPacker(spectra, **packer_kw)
    if len(packer.types) == 1:
        for _, group in groupby(psms, lambda m: m["scan"]):
            for ind, match in enumerate(group):
                if ind == packer.hit_depth:
                    break
                packer.add(match)
            if len(packer) >= chunk_psms:
                yield packer.flush()
    else:
        if len(psms) != len(packer.types):
            raise ValueError("%d record lists for %d modification types" % (len(psms), len(packer.types)))
        for groups in zip(*(groupby(p, lambda m: m["scan"]) for p in psms), strict=True):
            if any(scan != groups[0][0] for scan, _ in groups):
                raise ValueError("the record lists of the modification types do not list the same scans")
            for t, (_, group) in enumerate(groups):
                for ind, match in enumerate(group):
                    if ind == packer.hit_depth:
                        break
                    packer.add(match, t)
            if len(packer) >= chunk_psms:
                yield packer.flush()
    if len(packer):
        yield packer.flush()


def score_stream(scorer, batches, depth=2):
    """Score (scans, batch) chunks on the GPU while a producer thread packs the next ones.  `scorer`: a Scorer /
    MultiScorer, or a function batch -> results (e.g. around `score_typed`).

    `pa_score_batch` is a blocking C call that releases the GIL (ctypes), so host-side
    parsing/packing of chunk c+1 overlaps the H2D copies and kernels of chunk c.  Yields
    (scans, batch, results) in order.  If scoring raises or the consumer abandons the generator,
    the producer is told to stop and joined, so no thread is left blocked on the bounded queue."""
    q = queue.Queue(maxsize=depth)
    stop = threading.Event()

    def put(item):
        while not stop.is_set():
            try:
                q.put(item, timeout=0.1)
                return True
            except queue.Full:
                continue
        return False

    def producer():
        try:
            for item in batches:
                if not put(item):
                    return
            put(None)
        except BaseException as e:      # surfaced in the consumer
            put(e)

    t = threading.Thread(target=producer, daemon=True)
    t.start()
    try:
        while True:
            item = q.get()
            if item is None:
                break
            if isinstance(item, BaseException):
                raise item
            scans, batch = item
            yield scans, batch, (scorer(batch) if callable(scorer) else scorer.score_batch(batch))
    finally:
        stop.set()
        t.join(timeout=30)


def result_rows(scorer, scans, batch, res, rows_of=None):
    """-> [scan, LocalizedSequence, PepScore, Ascores, AltSites] rows with the reference's string
    formatting (__main__.py:158-164): ascores `str(np.float32)` joined by ';', alternative sites
    joined by ',' inside a mod and ';' between mods.  rows_of: the batch rows to format (default: all), e.g. the rows
    of one type of a typed batch, formatted with that type's scorer"""
    from ..batch import format_results
    from .._lib import PSM_STATUS
    rows = []
    for i in range(scans.size) if rows_of is None else rows_of:
        status = int(res["psm_status"][i])
        if status != 0:
            import warnings
            pep = bytes(batch["pep"][batch["pep_off"][i]:batch["pep_off"][i + 1]]).decode()
            warnings.warn("scan %d, %s: not scored (%s)" % (scans[i], pep, PSM_STATUS.get(status, status)))
            continue
        seq, best, asc, alts = format_results(scorer, batch, res, i)
        rows.append([int(scans[i]), seq, best, ";".join(str(s) for s in asc),
                     ";".join(",".join(str(site) for site in site_list) for site_list in alts)])
    return rows


TSV_COLUMNS = ["Scan", "LocalizedSequence", "PepScore", "Ascores", "AltSites"]


def write_tsv(path, rows):
    """what `DataFrame(rows, columns=...).to_csv(path, sep="\\t", index=False)` writes
    (__main__.py:166-172): header line, python `repr` floats, no quoting needed for these fields"""
    with open(path, "w", newline="") as dst:
        dst.write("\t".join(TSV_COLUMNS) + "\n")
        for scan, seq, best, asc, alt in rows:
            dst.write("%d\t%s\t%s\t%s\t%s\n" % (scan, seq, repr(float(best)), asc, alt))
