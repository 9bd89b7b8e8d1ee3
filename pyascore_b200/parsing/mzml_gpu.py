"""mzML spectra decoded on the GPU: the file is read once into pinned host memory, `pa_mzml_index` walks its XML
structure on the host (no payload is touched there), the bytes go to the device in one copy, and `pa_decode_arrays`
decodes every retained binary array (base64, zlib, dtype conversion) straight into the CSR peak arrays in HBM.

The result is the `SpectraCSR` that `SpectraParser(path, "mzML").to_csr()` builds, bit for bit, with `spec_off`, `mz`
and `inten` / `inten32` as CUDA tensors.  A file whose decoding could differ from the stdlib reader's is refused with a
ValueError that says why (see include/pyascore_b200.h, pa_mzml_index / pa_decode_arrays)."""
import ctypes as C
import os

import numpy as np

from .. import _lib

_ERR_CAP = 1024
_ARRAY_DTYPE = np.dtype([("text_off", "<i8"), ("text_len", "<i8"), ("out_off", "<i8"), ("count", "<i8"),
                         ("spec", "<i8"), ("dtype", "<i4"), ("flags", "<i4")])
ZLIB, INTENSITY = 1, 2
DECODE_STATUS = {1: "base64 text that b64decode rejects (or non-ASCII text, an entity, data after the padding)",
                 2: "a zlib stream that zlib.decompress rejects",
                 3: "a decoded length other than the array length the file states"}


def _copy(ptr, n, ctype, dtype):
    if n == 0:
        return np.zeros(0, dtype)
    return np.frombuffer((ctype * n).from_address(ptr), dtype).copy()


def index_mzml(data, ms_level=2):
    """The retained spectra of the mzML file bytes `data` (bytes or a uint8 array) in scan order, with the byte ranges
    of their binary arrays: dict(scans, ms_level, precursor_mz, precursor_charge, spec_off, arrays).  `arrays` is a
    structured array (text_off, text_len, out_off, count, spec, dtype, flags), m/z then intensity per spectrum that has both.
    Raises ValueError with the stdlib reader's text (several precursors, numpress) or the reason for refusing."""
    L = _lib.load()
    buf = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data, np.uint8)
    out = C.POINTER(_lib.PaMzmlIndex)()
    err = C.create_string_buffer(_ERR_CAP)
    rc = L.pa_mzml_index(buf.ctypes.data if buf.size else None, buf.size, int(ms_level), C.byref(out), err, _ERR_CAP)
    if rc != 0:
        raise ValueError(err.value.decode("utf8", "replace"))
    try:
        ix = out.contents
        n, na = ix.n_spec, ix.n_arrays
        res = dict(scans=_copy(ix.scan, n, C.c_int64, np.int64), ms_level=_copy(ix.ms_level, n, C.c_int32, np.int32),
                   precursor_mz=_copy(ix.precursor_mz, n, C.c_double, np.float64),
                   precursor_charge=_copy(ix.precursor_charge, n, C.c_int32, np.int32),
                   spec_off=_copy(ix.spec_off, n + 1, C.c_int64, np.int64))
        res["arrays"] = (np.frombuffer((C.c_char * (na * _ARRAY_DTYPE.itemsize)).from_address(C.addressof(ix.arrays.contents)),
                                       _ARRAY_DTYPE).copy() if na else np.zeros(0, _ARRAY_DTYPE))
    finally:
        L.pa_mzml_index_free(out)
    return res


def read_pinned(path):
    """the bytes of `path` in one pinned host block (uint8 array)"""
    from ..batch import pinned_empty
    size = os.path.getsize(path)
    buf = pinned_empty(size, np.uint8)
    with open(path, "rb") as f:
        got = f.readinto(memoryview(buf)) if size else 0
    if got != size:
        raise OSError("%s: read %d of %d bytes" % (path, got, size))
    return buf


def mzml_to_device(path, ms_level=2, device=0, narrow_intensity=True):
    """File -> SpectraCSR with its peak arrays on CUDA device `device` (see the module text)."""
    import torch

    from .spec_parsers import SpectraCSR
    L = _lib.load()
    data = read_pinned(path)
    ix = index_mzml(data, ms_level)
    dev = torch.device("cuda", int(device))
    arrays = ix["arrays"]
    total = int(ix["spec_off"][-1])
    file_dev = torch.empty(max(data.size, 1), dtype=torch.uint8, device=dev)
    if data.size:
        file_dev[:data.size].copy_(torch.from_numpy(data), non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()       # the pinned block is released on return
    mz = torch.empty(total, dtype=torch.float64, device=dev)
    inten = torch.empty(total, dtype=torch.float64, device=dev)
    status = torch.zeros(max(arrays.size, 1), dtype=torch.int32, device=dev)
    inexact = torch.zeros(1, dtype=torch.int32, device=dev)
    err = C.create_string_buffer(_ERR_CAP)
    rc = L.pa_decode_arrays(int(device), file_dev.data_ptr(), arrays.ctypes.data if arrays.size else None, arrays.size,
                            mz.data_ptr(), inten.data_ptr(), status.data_ptr(), inexact.data_ptr(), err, _ERR_CAP)
    if rc != 0:
        msg = err.value.decode("utf8", "replace")
        raise (RuntimeError if rc == -1 else ValueError)("pyascore_b200: " + msg)
    del file_dev
    st = status[:arrays.size].cpu().numpy()
    bad = np.flatnonzero(st)
    if bad.size:
        j = int(bad[0])
        raise ValueError("%s: %d binary array(s) cannot be decoded on the GPU; the first (%s array of scan %d): %s" % (
            path, bad.size, "intensity" if arrays["flags"][j] & INTENSITY else "m/z", ix["scans"][arrays["spec"][j]],
            DECODE_STATUS.get(int(st[j]), int(st[j]))))
    narrow = narrow_intensity and total > 0 and int(inexact.item()) == 0
    spec_off = torch.from_numpy(ix["spec_off"]).to(dev)
    if narrow:
        return SpectraCSR(ix["scans"], ix["precursor_mz"], ix["precursor_charge"], spec_off, mz, None,
                          inten.to(torch.float32))
    return SpectraCSR(ix["scans"], ix["precursor_mz"], ix["precursor_charge"], spec_off, mz, inten)

