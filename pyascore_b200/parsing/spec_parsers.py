"""Spectra files -> the scan records the scoring path consumes, and straight into CSR arrays.

Mirror of the reference's `SpectraParser` (pyascore/parsing/spec_parsers.py:175-282): same
constructor arguments, `to_list()` / `to_dict()` and record schema
`{scan, ms_level, precursor_mz, precursor_charge, mz_values f64[], intensity_values f64[]}`.
New here: `to_csr()` packs every retained scan into one pinned CSR block (spec_off / mz / inten),
the layout `pa_score_batch` reads, so no per-spectrum copy happens between the file and the GPU.
"""
import numpy as np

from . import _xml

_READERS = {"mzML": _xml.iter_mzml, "mzXML": _xml.iter_mzxml}


class SpectraCSR:
    """All retained scans of one file: scans ascending, peaks of scan i at mz[spec_off[i]:spec_off[i+1]]."""

    def __init__(self, scans, precursor_mz, precursor_charge, spec_off, mz, inten, inten32=None):
        self.scans = scans                          # int64[n_spec], ascending
        self.precursor_mz = precursor_mz            # float64[n_spec], NaN = missing
        self.precursor_charge = precursor_charge    # int32[n_spec], 0 = missing
        self.spec_off = spec_off                    # int64[n_spec+1]
        self.mz = mz                                # float64[n_peaks]  (pinned when a GPU library is loaded)
        self.inten = inten                          # float64[n_peaks], or None when every intensity of the file is a
        self.inten32 = inten32                      #   float32 value: then float32[n_peaks] here (pa_batch.inten32)
        self._index = None

    def __len__(self):
        return self.scans.size

    def index_of(self, scan):
        """position of `scan`, or -1 (last one wins for duplicated scan numbers, like dict building)"""
        if self._index is None:
            self._index = {int(s): i for i, s in enumerate(self.scans)}
        return self._index.get(int(scan), -1)

    def spectrum(self, i):
        a, b = int(self.spec_off[i]), int(self.spec_off[i + 1])
        return self.mz[a:b], (self.inten if self.inten is not None else self.inten32)[a:b]


class SpectraParser:
    """Read MSn spectra from mzML / mzXML (reference: spec_parsers.py:175-282)."""

    def __init__(self, spec_file_name, spec_file_format, ms_level=2, custom_filter=None):
        if spec_file_format not in _READERS:
            raise ValueError("{} not supported at this time."
                             " Should be one of: mzML or mzXML".format(spec_file_format))
        self._path, self._reader = spec_file_name, _READERS[spec_file_format]
        if ms_level >= 0:
            self.ms_level = ms_level
        else:
            raise ValueError("ms_level must be an integer greater than or equal to 0")
        # the reference tests `callable(ms_level)` here (spec_parsers.py:226), which rejects every
        # custom filter; the evident intent is implemented instead
        if custom_filter is not None and not callable(custom_filter):
            raise ValueError("custom_filter must be callable.")
        self.custom_filter = custom_filter
        self._spectra = []

    def _records(self):
        for scan, ms_level, pmz, pz, mz, inten in self._reader(self._path):
            if self.ms_level and ms_level != self.ms_level:
                continue
            rec = {"scan": scan, "ms_level": ms_level, "precursor_mz": pmz, "precursor_charge": pz,
                   "mz_values": mz, "intensity_values": inten}
            if self.custom_filter is not None and not self.custom_filter(rec):
                continue
            yield rec

    def _get_spectra(self):
        if not self._spectra:
            self._spectra = sorted(self._records(), key=lambda s: s["scan"])

    def to_list(self):
        """List of scans from the file sorted by scan number"""
        self._get_spectra()
        return self._spectra

    def to_dict(self):
        """{scan number : spectrum without its "scan" key} (the reference pops the key out of its cached records,
        spec_parsers.py:281, so a second call fails there; the cache is left intact here)"""
        self._get_spectra()
        return {spec["scan"]: {k: v for k, v in spec.items() if k != "scan"} for spec in self._spectra}

    def to_csr(self, pinned=True, narrow_intensity=True):
        """Pack the retained scans into one CSR block (pinned host memory by default).

        narrow_intensity: when every intensity of the file is exactly a float32 value (mzML / mzXML files usually
        store 32-bit intensity arrays) the block carries them as float32 (`inten32`, `inten` = None): a quarter
        fewer bytes over the host link, same ranks (pa_batch.inten32)."""
        self._get_spectra()
        recs = self._spectra
        n = len(recs)
        spec_off = np.zeros(n + 1, np.int64)
        np.cumsum([r["mz_values"].size for r in recs], out=spec_off[1:])
        total = int(spec_off[-1])
        narrow = narrow_intensity and total > 0 and all(
            np.array_equal(r["intensity_values"].astype(np.float32), r["intensity_values"]) for r in recs)
        idt = np.float32 if narrow else np.float64
        if pinned:
            from ..batch import pinned_empty
            mz, inten = pinned_empty(total, np.float64), pinned_empty(total, idt)
        else:
            mz, inten = np.empty(total, np.float64), np.empty(total, idt)
        for i, r in enumerate(recs):
            a, b = spec_off[i], spec_off[i + 1]
            mz[a:b] = r["mz_values"]
            inten[a:b] = r["intensity_values"]
        scans = np.array([r["scan"] for r in recs], np.int64)
        pmz = np.array([np.nan if r["precursor_mz"] is None else r["precursor_mz"] for r in recs], np.float64)
        pz = np.array([0 if r["precursor_charge"] is None else r["precursor_charge"] for r in recs], np.int32)
        return SpectraCSR(scans, pmz, pz, spec_off, mz, None if narrow else inten, inten if narrow else None)

    def to_device(self, device=0, narrow_intensity=True):
        """The CSR block of `to_csr(narrow_intensity=...)`, bit for bit, decoded on CUDA device `device`: the host reads
        the XML structure only, the GPU decodes the binary arrays (parsing/mzml_gpu.py).  `spec_off`, `mz` and `inten` /
        `inten32` are CUDA tensors; `scans`, `precursor_mz` and `precursor_charge` numpy arrays.  mzML only, without a
        custom_filter (it runs on decoded arrays in Python); a file this path cannot decode exactly as the stdlib reader
        does raises ValueError with the reason, and `to_csr()` reads it."""
        if self._reader is not _xml.iter_mzml:
            raise ValueError("to_device decodes mzML files only; read mzXML with to_csr()")
        if self.custom_filter is not None:
            raise ValueError("to_device cannot apply a custom_filter (it runs in Python on decoded arrays); use to_csr()")
        from .mzml_gpu import mzml_to_device
        return mzml_to_device(self._path, self.ms_level, device, narrow_intensity)
