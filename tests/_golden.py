"""Helpers shared by the golden-vector tests (oracle on CPU, CUDA library on GPU)."""
import glob
import json
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def load(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    meta = json.loads(bytes(z["meta"]).decode())
    batch = {k[3:]: np.ascontiguousarray(z[k]) for k in z.files if k.startswith("in_")}
    ref = {k[4:]: z[k] for k in z.files if k.startswith("ref_")}
    return meta, batch, _finish_ref(ref, batch)


def _finish_ref(ref, batch):
    n = batch["n_mod"].size
    seqs = bytes(ref["best_sequence"]).decode().split("\n")
    if len(seqs) != n:          # all-empty edge: "".split -> ['']
        seqs = (seqs + [""] * n)[:n]
    ref["best_sequence"] = seqs
    ref["iso_off"] = np.concatenate([[0], np.cumsum(ref["n_iso"])]).astype(np.int64)
    ref["mod_off"] = np.concatenate([[0], np.cumsum(batch["n_mod"])]).astype(np.int64)
    return ref


def oracle_ref(meta, batch):
    """the C oracle run live over a host batch -> reference results in the layout load() returns (whole pep_scores
    tables included), for test_gpu_parity.check_against_ref"""
    import sys
    sys.path.insert(0, GOLDEN_DIR)
    import make_golden
    from oracle.cscorer import OraclePyAscore
    ref = make_golden.run_reference(meta["scorer"], meta["neutral_losses"], batch, OraclePyAscore)
    return _finish_ref(ref, batch)


def ref_alt(ref, i, j):
    q = int(ref["mod_off"][i]) + j
    return ref["alt"][ref["alt_off"][q]:ref["alt_off"][q + 1]]


def same_bits(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def rel_close(a, b, tol=1e-6):
    """|a-b| <= tol*|b| elementwise, with inf/nan required to match exactly."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    if a.shape != b.shape:
        return False
    fin = np.isfinite(b)
    if not np.array_equal(np.isfinite(a), fin):
        return False
    if not np.array_equal(a[~fin], b[~fin], equal_nan=True):
        return False
    return bool(np.all(np.abs(a[fin] - b[fin]) <= tol * np.abs(b[fin])))


BIG_DIR = os.path.join(GOLDEN_DIR, "big")


def big_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(BIG_DIR, "*.npz")))


def load_big(name):
    """goldens of tests/golden/make_golden_big.py: per-PSM results + SHA-256 of the whole pep_scores table"""
    z = np.load(os.path.join(BIG_DIR, name + ".npz"))
    meta = json.loads(bytes(z["meta"]).decode())
    batch = {k[3:]: np.ascontiguousarray(z[k]) for k in z.files if k.startswith("in_")}
    ref = {k[4:]: z[k] for k in z.files if k.startswith("ref_")}
    n = batch["n_mod"].size
    seqs = bytes(ref["best_sequence"]).decode().split("\n")
    ref["best_sequence"] = (seqs + [""] * n)[:n]
    ref["table_sha256"] = bytes(ref["table_sha256"]).decode().split("\n")
    ref["mod_off"] = np.concatenate([[0], np.cumsum(batch["n_mod"])]).astype(np.int64)
    return meta, batch, ref


def table_digest(bits, cnt, sc, w, tot):
    import hashlib
    h = hashlib.sha256()
    for a, dt in ((bits, np.uint64), (cnt, np.int32), (sc, np.float32), (w, np.float32), (tot, np.int32)):
        h.update(np.ascontiguousarray(a, dt).tobytes())
    return h.hexdigest()


def sig_bits(sig):
    bits = np.zeros(sig.shape[0], np.uint64)
    for j in range(sig.shape[1]):
        bits |= sig[:, j].astype(np.uint64) << np.uint64(j)
    return bits
