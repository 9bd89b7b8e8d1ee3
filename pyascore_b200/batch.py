"""Batched scoring over CSR arrays -- the entry point the CLI loop of the reference
(pyascore/__main__.py:129-164) is replaced with.

`Scorer` owns one pa_scorer handle (one GPU).  `Scorer.score_batch(batch)` takes the dict of
arrays described in pyascore_b200/synth.py (numpy arrays in host memory -- ideally allocated
with `pinned_empty` -- or torch CUDA tensors already resident in HBM) and returns the result
arrays; `format_results` turns them into the reference's strings / lists.
"""
import ctypes as C

import numpy as np

from . import _lib

_IN_KEYS = ("spec_off", "mz", "inten", "psm_spec", "pep_off", "pep", "n_mod", "max_charge",
            "aux_off", "aux_pos", "aux_mass", "mod_off", "inten32")
_IN_DTYPES = dict(spec_off=np.int64, mz=np.float64, inten=np.float64, psm_spec=np.int32, pep_off=np.int32,
                  pep=np.uint8, n_mod=np.int32, max_charge=np.int32, aux_off=np.int32, aux_pos=np.uint32,
                  aux_mass=np.float32, mod_off=np.int64, inten32=np.float32)
_OUT_DTYPES = dict(best_sig=np.uint64, best_score=np.float32, n_iso=np.int64, n_sites=np.int32,
                   ascores=np.float32, alt_sites=np.uint64, psm_status=np.int32)


_WANT_ALL = ("best_sig", "best_score", "n_iso", "n_sites", "ascores", "alt_sites", "psm_status")


class _Pinned:
    """numpy view over cudaMallocHost memory; freed when the last view dies."""

    def __init__(self, nbytes, flags=0):
        self.L = _lib.load()
        self.ptr = self.L.pa_alloc_pinned_ex(max(int(nbytes), 1), int(flags))
        if not self.ptr:
            raise MemoryError("pa_alloc_pinned(%d) failed" % nbytes)
        self.nbytes = int(nbytes)

    def __del__(self):
        if getattr(self, "ptr", None):
            self.L.pa_free_pinned(self.ptr)
            self.ptr = None


PINNED_WRITE_COMBINED, PINNED_PORTABLE = 1, 2


def pinned_empty(shape, dtype, flags=0):
    """numpy array over page-locked host memory (pa_alloc_pinned_ex; flags: PINNED_WRITE_COMBINED | PINNED_PORTABLE)"""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) if not np.isscalar(shape) else int(shape)
    owner = _Pinned(n * dtype.itemsize, flags)
    buf = (C.c_char * max(n * dtype.itemsize, 1)).from_address(owner.ptr)
    buf._pa_owner = owner            # the numpy view keeps `buf` (its base) and so the pinned block alive
    return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)


def pin_batch(batch, flags=0, peak_flags=None):
    """Copy a host batch into pinned memory (so H2D copies overlap compute).  `peak_flags`: placement flags of the two
    big arrays (m/z, intensities) when they differ from the rest, e.g. write-combined pages."""
    out = {}
    for k, v in batch.items():
        a = pinned_empty(v.shape, v.dtype, (peak_flags if peak_flags is not None and k in ("mz", "inten") else flags))
        a[...] = v
        out[k] = a
    return out


def add_mod_off(batch):
    if "mod_off" not in batch:
        n_mod = batch["n_mod"]
        if isinstance(n_mod, np.ndarray):
            mo = np.zeros(n_mod.size + 1, np.int64)
            np.cumsum(np.maximum(n_mod, 0), out=mo[1:])      # (a negative n_mod is reported per PSM, not laid out)
        else:  # torch tensor
            import torch
            mo = torch.zeros(n_mod.numel() + 1, dtype=torch.int64, device=n_mod.device)
            mo[1:] = torch.cumsum(n_mod.to(torch.int64).clamp_(min=0), 0)
        batch["mod_off"] = mo
    return batch


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()          # torch tensor


def _check(name, a):
    want = _IN_DTYPES[name]
    if isinstance(a, np.ndarray):
        if a.dtype != want:
            raise ValueError("Buffer dtype mismatch for %s, expected '%s' but got '%s'" % (name, np.dtype(want), a.dtype))
        if not a.flags.c_contiguous:
            raise ValueError("ndarray is not C-contiguous (%s)" % name)
    else:
        import torch
        tmap = {np.int64: torch.int64, np.float64: torch.float64, np.int32: torch.int32, np.uint8: torch.uint8,
                np.uint32: torch.int32, np.float32: torch.float32}
        if a.dtype != tmap[want] and not (want is np.uint32 and a.dtype == torch.uint32):
            raise ValueError("tensor dtype mismatch for %s: %s" % (name, a.dtype))
        if not a.is_contiguous():
            raise ValueError("tensor is not contiguous (%s)" % name)


class Scorer:
    """One pa_scorer: PyAscore's constructor arguments (Ascore.pyx:64-73) + a CUDA device.  n_top: 10 .. 64
    (_lib.PA_N_TOP .. _lib.PA_MAX_N_TOP); the per-depth arrays of the probes below are n_top wide."""

    def __init__(self, bin_size, n_top, mod_group, mod_mass, mz_error=.5, fragment_types="by", device=0):
        self.L = _lib.load()
        h = C.c_void_p()
        rc = self.L.pa_create(bin_size, int(n_top), mod_group.encode("utf8"), mod_mass, mz_error,
                              fragment_types.encode("utf8"), int(device), C.byref(h))
        if rc != 0:
            msg = _lib.last_error(None)
            if rc == -1:
                raise RuntimeError("pyascore_b200: " + msg)
            raise ValueError("pyascore_b200: " + msg)
        self.h = h
        self.device = int(device)
        self.mod_group = mod_group
        self.n_top = int(n_top)

    def close(self):
        if getattr(self, "h", None):
            self.L.pa_destroy(self.h)
            self.h = None

    __del__ = close

    def _raise(self, rc):
        msg = _lib.last_error(self.h)
        if rc == -1:
            raise RuntimeError("pyascore_b200 (CUDA): " + msg)
        raise ValueError("pyascore_b200: " + msg)

    def add_neutral_loss(self, group, mass):
        rc = self.L.pa_add_neutral_loss(self.h, group.encode("utf8"), mass)
        if rc != 0:
            self._raise(rc)

    def _prepare(self, batch, out, want):
        """checked ctypes views of a batch + result arrays (allocated on the side the inputs live on)"""
        add_mod_off(batch)
        for k in _IN_KEYS:
            if k in batch and batch[k] is not None:
                _check(k, batch[k])
        n_psm = int(batch["n_mod"].shape[0])
        n_spec = int(batch["spec_off"].shape[0]) - 1
        on_dev = not isinstance(batch["mz"], np.ndarray)
        pb = _lib.PaBatch()
        pb.n_spec, pb.n_psm = n_spec, n_psm
        for k in _IN_KEYS:
            setattr(pb, k, _ptr(batch.get(k)))
        if out is None:
            out = {}
            if on_dev:
                import torch
                tm = dict(best_sig=torch.int64, best_score=torch.float32, n_iso=torch.int64, n_sites=torch.int32,
                          ascores=torch.float32, alt_sites=torch.int64, psm_status=torch.int32)
                n_modtot = int(batch["mod_off"][-1].item())
                for k in want:
                    n = n_modtot if k in ("ascores", "alt_sites") else n_psm
                    out[k] = torch.empty(max(n, 1), dtype=tm[k], device=batch["mz"].device)[:n]
            else:
                n_modtot = int(batch["mod_off"][-1])
                for k in want:
                    n = n_modtot if k in ("ascores", "alt_sites") else n_psm
                    out[k] = np.empty(n, _OUT_DTYPES[k])
        pr = _lib.PaResults()
        for k in _OUT_DTYPES:
            setattr(pr, k, _ptr(out.get(k)))
        return pb, pr, out

    def score_batch(self, batch, out=None, keep_isoforms=False, want=_WANT_ALL, psm_range=None):
        """Score every PSM of `batch` (or PSMs [lo, hi) with psm_range=(lo, hi): results land at their absolute
        positions); returns dict of result arrays (same side as the inputs)."""
        pb, pr, out = self._prepare(batch, out, want)
        flags = _lib.PA_KEEP_ISOFORMS if keep_isoforms else 0
        if psm_range is None:
            rc = self.L.pa_score_batch(self.h, C.byref(pb), C.byref(pr), flags)
        else:
            rc = self.L.pa_score_range(self.h, C.byref(pb), C.byref(pr), int(psm_range[0]), int(psm_range[1]), flags)
        if rc != 0:
            self._raise(rc)
        return out

    def score_batch_async(self, batch, out=None, want=_WANT_ALL, psm_range=None, stream=None):
        """Start scoring and return at once (pa_score_batch_async); `wait()` completes the call.  `stream`: a CUDA
        stream handle (int / torch.cuda.Stream) whose queued work must finish before the inputs are read."""
        pb, pr, out = self._prepare(batch, out, want)
        lo, hi = (0, -1) if psm_range is None else (int(psm_range[0]), int(psm_range[1]))
        if stream is not None and not isinstance(stream, int):
            stream = stream.cuda_stream
        self._inflight = (batch, out)            # the arrays must outlive the call
        rc = self.L.pa_score_batch_async(self.h, C.byref(pb), C.byref(pr), lo, hi, 0, stream)
        if rc != 0:
            self._inflight = None
            self._raise(rc)
        return out

    def wait(self):
        rc = self.L.pa_wait(self.h)
        self._inflight = None
        if rc != 0:
            self._raise(rc)

    def shard_ranges(self, batch, world, peak_weight=55., share=None):
        """-> [(p0, p1)] * world: contiguous PSM ranges of a host batch cut on spectrum boundaries and balanced by
        estimated cost (pa_shard_ranges)"""
        add_mod_off(batch)
        pb = _lib.PaBatch()
        pb.n_spec, pb.n_psm = int(batch["spec_off"].shape[0]) - 1, int(batch["n_mod"].shape[0])
        for k in _IN_KEYS:
            setattr(pb, k, _ptr(batch.get(k)))
        cuts = np.zeros(world + 1, np.int64)
        sh = None if share is None else np.ascontiguousarray(share, np.float64)
        rc = self.L.pa_shard_ranges(self.h, C.byref(pb), int(world), float(peak_weight),
                                    None if sh is None else sh.ctypes.data, cuts.ctypes.data)
        if rc != 0:
            raise ValueError("pyascore_b200: cannot shard this batch (host arrays with non-decreasing psm_spec needed)")
        return [(int(cuts[r]), int(cuts[r + 1])) for r in range(world)]

    def counters(self):
        c = _lib.PaCounters()
        self.L.pa_counters(self.h, C.byref(c))
        return {n: getattr(c, n) for n, _ in c._fields_}

    # ---- stage probes ----
    def bin_spectra(self, spec_off, mz, inten):
        spec_off = np.ascontiguousarray(spec_off, np.int64)
        mz = np.ascontiguousarray(mz, np.float64)
        inten = np.ascontiguousarray(inten, np.float64)
        n = spec_off.size - 1
        omz = np.zeros(mz.size, np.float32)
        ork = np.zeros(mz.size, np.uint8)
        ocnt = np.zeros(max(n, 1), np.int32)
        rc = self.L.pa_bin_spectra(self.h, n, spec_off.ctypes.data, mz.ctypes.data, inten.ctypes.data,
                                   omz.ctypes.data, ork.ctypes.data, ocnt.ctypes.data)
        if rc != 0:
            self._raise(rc)
        return omz, ork, ocnt[:n]

    def tail_table(self, n_max):
        out = np.zeros(((n_max + 1) * (n_max + 2) // 2, self.n_top), np.float32)
        rc = self.L.pa_tail_table(self.h, n_max, out.ctypes.data)
        if rc != 0:
            self._raise(rc)
        return out

    # ---- per-PSM detail of a kept batch ----
    def fetch_pep_scores(self, psm):
        n = self.L.pa_fetch_pep_scores(self.h, psm, 0, None, None, None, None, None)
        if n < 0:
            self._raise(int(n))
        sig = np.zeros(n, np.uint64)
        cnt = np.zeros((n, self.n_top), np.int32)
        sc = np.zeros((n, self.n_top), np.float32)
        w = np.zeros(n, np.float32)
        tot = np.zeros(n, np.int32)
        if n:
            m = self.L.pa_fetch_pep_scores(self.h, psm, n, sig.ctypes.data, cnt.ctypes.data, sc.ctypes.data,
                                           w.ctypes.data, tot.ctypes.data)
            if m < 0:
                self._raise(int(m))
        return sig, cnt, sc, w, tot

    def calculate_ambiguity(self, psm, sig_a, scores_a, w_a, sig_b, scores_b, w_b):
        sa = np.ascontiguousarray(scores_a, np.float32)
        sb = np.ascontiguousarray(scores_b, np.float32)
        if sa.size != self.n_top or sb.size != self.n_top:
            raise ValueError("scores must have n_top = %d entries" % self.n_top)
        out = C.c_float()
        rc = self.L.pa_calculate_ambiguity(self.h, psm, int(sig_a), sa.ctypes.data, w_a, int(sig_b), sb.ctypes.data,
                                           w_b, C.byref(out))
        if rc != 0:
            self._raise(rc)
        return out.value

    def format_sequence(self, pep, n_mod, aux_pos, aux_mass, sig):
        pb = pep if isinstance(pep, (bytes, bytearray)) else bytes(pep)
        ap = np.ascontiguousarray(aux_pos, np.uint32) if aux_pos is not None else np.zeros(0, np.uint32)
        am = np.ascontiguousarray(aux_mass, np.float32) if aux_mass is not None else np.zeros(0, np.float32)
        buf = C.create_string_buffer(16 * len(pb) + 64)
        arr = np.frombuffer(pb, np.uint8)
        n = self.L.pa_format_sequence(self.h, arr.ctypes.data, len(pb), int(n_mod), ap.ctypes.data, am.ctypes.data,
                                      ap.size, int(sig), buf, len(buf))
        if n < 0:
            raise ValueError("pa_format_sequence failed")
        return buf.value.decode("utf8")

    def site_positions(self, pep):
        pb = pep if isinstance(pep, (bytes, bytearray)) else bytes(pep)
        arr = np.frombuffer(pb, np.uint8)
        pos = np.zeros(max(len(pb), 1), np.int32)
        n = self.L.pa_site_positions(self.h, arr.ctypes.data, len(pb), pos.ctypes.data, pos.size)
        return pos[:n]


class MultiScorer:
    """One scorer per GPU of the box behind the interface of `Scorer`: a host batch is cut into contiguous PSM
    ranges on spectrum boundaries (balanced by estimated cost), every GPU scores its range concurrently and writes
    its slice of ONE set of result arrays -- no collective, no gather (SURVEY.md section 8e: the sharded form of
    the loop in pyascore/__main__.py:129-164)."""

    def __init__(self, bin_size, n_top, mod_group, mod_mass, mz_error=.5, fragment_types="by", devices=(0,)):
        self.devices = [int(d) for d in devices]
        if not self.devices:
            raise ValueError("MultiScorer needs at least one device")
        self.scorers = [Scorer(bin_size, n_top, mod_group, mod_mass, mz_error, fragment_types, device=d)
                        for d in self.devices]
        self.mod_group = mod_group
        self.last_ranges = None
        # share of a batch's cost each GPU gets; starts equal and follows the rates measured on the calls so far (the
        # GPUs of a box do not get the same host-link bandwidth when all of them copy at once)
        self.share = np.ones(len(self.devices))
        self.adapt = True

    def close(self):
        for sc in self.scorers:
            sc.close()

    def add_neutral_loss(self, group, mass):
        for sc in self.scorers:
            sc.add_neutral_loss(group, mass)

    def score_batch(self, batch, out=None, want=_WANT_ALL, peak_weight=55.):
        if not isinstance(batch["mz"], np.ndarray):
            raise ValueError("MultiScorer shards host batches; device-resident batches belong to one GPU")
        n = len(self.scorers)
        if n == 1:
            self.last_ranges = [(0, int(batch["n_mod"].shape[0]))]
            return self.scorers[0].score_batch(batch, out=out, want=want)
        try:
            self.last_ranges = ranges = self.scorers[0].shard_ranges(batch, n, peak_weight, self.share)
        except ValueError:                  # PSMs not in spectrum order: cannot be cut on spectrum boundaries
            self.last_ranges = [(0, int(batch["n_mod"].shape[0]))]
            return self.scorers[0].score_batch(batch, out=out, want=want)
        started = []
        err = None
        for sc, r in zip(self.scorers, ranges):
            try:
                out = sc.score_batch_async(batch, out=out, want=want, psm_range=r)     # rank 0 allocates `out`
                started.append(sc)
            except Exception as e:          # noqa: BLE001 -- the ranks already started must still be waited for
                err = e
                break
        for sc in started:
            try:
                sc.wait()
            except Exception as e:          # noqa: BLE001
                err = err or e
        if err is not None:
            raise err
        if self.adapt:
            # rate of every GPU on this call (cost units per millisecond, cost = its share of the cut); the next cut
            # follows a smoothed version of it
            ms = np.array([max(sc.counters()["ms_total"], 1e-3) for sc in self.scorers])
            if np.all(np.array([b - a for a, b in ranges]) > 0):
                rate = self.share / self.share.sum() / ms
                self.share = 0.5 * self.share / self.share.sum() + 0.5 * rate / rate.sum()
        return out

    def counters(self):
        return [sc.counters() for sc in self.scorers]

    # string / site helpers are host arithmetic: any scorer serves
    def format_sequence(self, *a):
        return self.scorers[0].format_sequence(*a)

    def site_positions(self, pep):
        return self.scorers[0].site_positions(pep)


def score_typed(scorers, batch, psm_type, out=None, want=_WANT_ALL):
    """Score PSM i of `batch` under scorers[psm_type[i]] (pa_score_typed): several modification types in one call, with
    the spectra copied and binned once for all of them.  `scorers`: `Scorer` objects on one device with the same
    bin_size and n_top; `psm_type`: uint8 per PSM on the side of the batch's arrays (numpy / CUDA tensor), or None
    (every PSM is type 0).  Returns the dict of `Scorer.score_batch`; the rows of type t equal scorers[t].score_batch on
    those rows alone, and `format_results` takes scorers[psm_type[i]] for row i."""
    scorers = list(scorers)
    if not scorers:
        raise ValueError("score_typed needs at least one scorer")
    s0 = scorers[0]
    pb, pr, out = s0._prepare(batch, out, want)
    if psm_type is not None:
        n_psm = int(batch["n_mod"].shape[0])
        if tuple(psm_type.shape) != (n_psm,):
            raise ValueError("psm_type must hold one entry per PSM (%d), not %s" % (n_psm, tuple(psm_type.shape)))
        if isinstance(psm_type, np.ndarray):
            if psm_type.dtype != np.uint8 or not psm_type.flags.c_contiguous:
                raise ValueError("psm_type must be a C-contiguous uint8 array")
            if not isinstance(batch["mz"], np.ndarray):
                raise ValueError("psm_type must live where the batch's arrays live (a CUDA tensor here)")
        else:
            import torch
            if psm_type.dtype != torch.uint8 or not psm_type.is_contiguous():
                raise ValueError("psm_type must be a contiguous uint8 tensor")
            if isinstance(batch["mz"], np.ndarray):
                raise ValueError("psm_type must live where the batch's arrays live (a host array here)")
    handles = (C.c_void_p * len(scorers))(*[sc.h for sc in scorers])
    rc = s0.L.pa_score_typed(handles, len(scorers), C.byref(pb), _ptr(psm_type), C.byref(pr), 0)
    if rc != 0:
        s0._raise(rc)
    return out


def format_results(scorer, batch, res, i):
    """Reference-style view of PSM i: (best_sequence, best_score, ascores, alt_sites)."""
    pep = bytes(batch["pep"][batch["pep_off"][i]:batch["pep_off"][i + 1]])
    k = int(batch["n_mod"][i])
    a0, a1 = int(batch["aux_off"][i]), int(batch["aux_off"][i + 1])
    n_iso = int(res["n_iso"][i])
    if n_iso == 0:
        seq = ""
    else:
        seq = scorer.format_sequence(pep, k, batch["aux_pos"][a0:a1], batch["aux_mass"][a0:a1], int(res["best_sig"][i]))
    mo = int(batch["mod_off"][i])
    asc = np.array(res["ascores"][mo:mo + k], np.float32)
    sites = scorer.site_positions(pep)
    alts = []
    for j in range(k):
        m = int(res["alt_sites"][mo + j])
        alts.append(np.array([sites[u] for u in range(len(sites)) if (m >> u) & 1], np.uint32))
    return seq, float(res["best_score"][i]), asc, alts
