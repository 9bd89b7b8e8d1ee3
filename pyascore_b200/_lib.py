"""ctypes binding of libpyascore_b200.so (C ABI: include/pyascore_b200.h).

The library is built in-tree by pyascore_b200/csrc/build.py.  There is no CPU path: if the
shared object is missing, or no CUDA device is usable, every entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PYASCORE_B200_LIB selects another build of the same library (tuning variants under build/)
SO_PATH = os.environ.get("PYASCORE_B200_LIB") or os.path.join(_HERE, "libpyascore_b200.so")

PA_N_TOP = 10          # depths the reference weights (and the default scoring depth)
PA_MAX_N_TOP = 64      # deepest n_top a scorer takes (include/pyascore_b200.h)
PA_KEEP_ISOFORMS = 1

PSM_STATUS = {
    0: "ok", 1: "unknown residue letter", 2: "peptide longer than 126 residues",
    3: "more than 63 modifiable residues", 4: "more than 2^26 positional isoforms", 5: "empty spectrum",
    6: "fixed-mod position beyond the peptide", 7: "bad spectrum index / negative n_of_mod or charge",
    8: "more than 4095 theoretical fragments per isoform",
}

vp = C.c_void_p


class PaBatch(C.Structure):
    _fields_ = [("n_spec", C.c_int64), ("spec_off", vp), ("mz", vp), ("inten", vp), ("n_psm", C.c_int64),
                ("psm_spec", vp), ("pep_off", vp), ("pep", vp), ("n_mod", vp), ("max_charge", vp),
                ("aux_off", vp), ("aux_pos", vp), ("aux_mass", vp), ("mod_off", vp), ("inten32", vp)]


class PaResults(C.Structure):
    _fields_ = [("best_sig", vp), ("best_score", vp), ("n_iso", vp), ("n_sites", vp), ("ascores", vp),
                ("alt_sites", vp), ("psm_status", vp)]


class PaMzmlArray(C.Structure):
    _fields_ = [("text_off", C.c_int64), ("text_len", C.c_int64), ("out_off", C.c_int64), ("count", C.c_int64),
                ("spec", C.c_int64), ("dtype", C.c_int32), ("flags", C.c_int32)]


class PaMzmlIndex(C.Structure):
    _fields_ = [("n_spec", C.c_int64), ("scan", vp), ("ms_level", vp), ("precursor_mz", vp), ("precursor_charge", vp),
                ("spec_off", vp), ("n_arrays", C.c_int64), ("arrays", C.POINTER(PaMzmlArray))]


class PaCounters(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_psm", "n_spec", "n_peaks", "n_retained", "n_isoforms",
                                         "n_fragment_lookups", "bytes_h2d", "bytes_d2h", "kernel_launches")] + \
               [(n, C.c_float) for n in ("ms_bin", "ms_plan", "ms_count", "ms_select", "ms_total")] + \
               [(n, C.c_int64) for n in ("launches_bin", "launches_count", "launches_select", "launches_ascore")] + \
               [(n, C.c_float) for n in ("ms_ascore", "ms_narrow_wait")] + [("n_chunks", C.c_int64), ("n_spec_exact", C.c_int64)] + \
               [("launches_deep", C.c_int64), ("ms_deep", C.c_float)]


EXPORTS = ["pa_create", "pa_add_neutral_loss", "pa_destroy", "pa_last_error", "pa_score_batch",
           "pa_fetch_pep_scores", "pa_calculate_ambiguity", "pa_format_sequence", "pa_site_positions",
           "pa_bin_spectra", "pa_tail_table", "pa_counters", "pa_alloc_pinned", "pa_free_pinned", "pa_version",
           "pa_create_binner", "pa_bin_spectra_ex", "pa_fragment_table", "pa_site_determining_ions", "pa_log_math",
           "pa_power_set_sums", "pa_score_range", "pa_score_batch_async", "pa_wait", "pa_shard_ranges", "pa_shard_ranges_for", "pa_alloc_pinned_ex", "pa_narrow_mz", "pa_score_typed",
           "pa_mzml_index", "pa_mzml_index_free", "pa_decode_arrays", "pa_inflate_host"]

_lib = None


def load():
    """Load the shared library (no CUDA call is made until pa_create)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            "pyascore_b200: %s is missing. Build it with `python pyascore_b200/csrc/build.py` "
            "(nvcc, sm_100a). There is no CPU fallback." % SO_PATH)
    L = C.CDLL(SO_PATH)
    L.pa_create.restype = C.c_int
    L.pa_create.argtypes = [C.c_float, C.c_int, C.c_char_p, C.c_float, C.c_float, C.c_char_p, C.c_int, C.POINTER(vp)]
    L.pa_add_neutral_loss.restype = C.c_int
    L.pa_add_neutral_loss.argtypes = [vp, C.c_char_p, C.c_float]
    L.pa_destroy.restype = None
    L.pa_destroy.argtypes = [vp]
    L.pa_last_error.restype = C.c_char_p
    L.pa_last_error.argtypes = [vp]
    L.pa_score_batch.restype = C.c_int
    L.pa_score_batch.argtypes = [vp, C.POINTER(PaBatch), C.POINTER(PaResults), C.c_uint32]
    L.pa_score_typed.restype = C.c_int
    L.pa_score_typed.argtypes = [C.POINTER(vp), C.c_int32, C.POINTER(PaBatch), vp, C.POINTER(PaResults), C.c_uint32]
    L.pa_score_range.restype = C.c_int
    L.pa_score_range.argtypes = [vp, C.POINTER(PaBatch), C.POINTER(PaResults), C.c_int64, C.c_int64, C.c_uint32]
    L.pa_score_batch_async.restype = C.c_int
    L.pa_score_batch_async.argtypes = [vp, C.POINTER(PaBatch), C.POINTER(PaResults), C.c_int64, C.c_int64, C.c_uint32, vp]
    L.pa_wait.restype = C.c_int
    L.pa_wait.argtypes = [vp]
    L.pa_shard_ranges.restype = C.c_int
    L.pa_shard_ranges.argtypes = [vp, C.POINTER(PaBatch), C.c_int32, C.c_double, vp, vp]
    L.pa_shard_ranges_for.restype = C.c_int
    L.pa_shard_ranges_for.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.POINTER(PaBatch), C.c_int32, C.c_double, vp, vp]
    L.pa_fetch_pep_scores.restype = C.c_int64
    L.pa_fetch_pep_scores.argtypes = [vp, C.c_int64, C.c_int64, vp, vp, vp, vp, vp]
    L.pa_calculate_ambiguity.restype = C.c_int
    L.pa_calculate_ambiguity.argtypes = [vp, C.c_int64, C.c_uint64, vp, C.c_float, C.c_uint64, vp, C.c_float, vp]
    L.pa_format_sequence.restype = C.c_int
    L.pa_format_sequence.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, C.c_int32, C.c_uint64, C.c_char_p, C.c_int32]
    L.pa_site_positions.restype = C.c_int
    L.pa_site_positions.argtypes = [vp, vp, C.c_int32, vp, C.c_int32]
    L.pa_bin_spectra.restype = C.c_int
    L.pa_bin_spectra.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp]
    L.pa_tail_table.restype = C.c_int
    L.pa_tail_table.argtypes = [vp, C.c_int32, vp]
    L.pa_counters.restype = C.c_int
    L.pa_counters.argtypes = [vp, C.POINTER(PaCounters)]
    L.pa_alloc_pinned.restype = vp
    L.pa_alloc_pinned.argtypes = [C.c_int64]
    L.pa_alloc_pinned_ex.restype = vp
    L.pa_alloc_pinned_ex.argtypes = [C.c_int64, C.c_uint32]
    L.pa_narrow_mz.restype = C.c_int64
    L.pa_narrow_mz.argtypes = [vp, vp, C.c_int64, C.c_float, vp, vp]
    L.pa_free_pinned.restype = None
    L.pa_free_pinned.argtypes = [vp]
    L.pa_version.restype = C.c_int
    L.pa_create_binner.restype = C.c_int
    L.pa_create_binner.argtypes = [C.c_float, C.c_int, C.c_int, C.POINTER(vp)]
    L.pa_bin_spectra_ex.restype = C.c_int
    L.pa_bin_spectra_ex.argtypes = [vp, C.c_int64] + [vp] * 9
    L.pa_fragment_table.restype = C.c_int
    L.pa_fragment_table.argtypes = [vp, vp, C.c_int32, vp, vp, C.c_int32, C.c_uint64, C.c_char, C.c_int32, vp, vp]
    L.pa_site_determining_ions.restype = C.c_int
    L.pa_site_determining_ions.argtypes = [vp, vp, C.c_int32, vp, vp, C.c_int32, C.c_uint64, C.c_uint64, C.c_char,
                                           C.c_int32, vp, C.POINTER(C.c_int32), vp, C.POINTER(C.c_int32), C.c_int32]
    L.pa_log_math.restype = C.c_int
    L.pa_log_math.argtypes = [vp, C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_float, vp]
    L.pa_power_set_sums.restype = C.c_int64
    L.pa_power_set_sums.argtypes = [vp, C.c_int32, C.c_int32, vp, C.c_int64]
    L.pa_mzml_index.restype = C.c_int
    L.pa_mzml_index.argtypes = [vp, C.c_int64, C.c_int32, C.POINTER(C.POINTER(PaMzmlIndex)), C.c_char_p, C.c_int32]
    L.pa_mzml_index_free.restype = None
    L.pa_mzml_index_free.argtypes = [C.POINTER(PaMzmlIndex)]
    L.pa_decode_arrays.restype = C.c_int
    L.pa_decode_arrays.argtypes = [C.c_int, vp, vp, C.c_int64, vp, vp, vp, vp, C.c_char_p, C.c_int32]
    L.pa_inflate_host.restype = C.c_int64
    L.pa_inflate_host.argtypes = [vp, C.c_int64, vp, C.c_int64]
    _lib = L
    return L


def last_error(handle=None):
    msg = load().pa_last_error(handle)
    return msg.decode("utf8", "replace") if msg else ""
