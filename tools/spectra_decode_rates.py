"""File -> SpectraCSR rates of the stdlib mzML reader and of the GPU decoder, and the CLI's wall clock per stage with
and without --gpu_decode.

    python tools/spectra_decode_rates.py [--ms2 200000] [--reps 3] [--out profiles/FILE.json]

Workload: seeded synthetic mzML files of `--ms2` MS2 spectra (100-300 peaks, float64 m/z, float32 intensities), with one
MS1 scan of ~3000 peaks before every 10 MS2 scans, written twice (zlib-compressed and uncompressed arrays), and the
matching pepXML (one phospho PSM per MS2 scan); see tests/test_gpu_decode.py::synthetic_run.  Per file:
  stdlib:    SpectraParser(path, "mzML").to_csr() (pinned, as the CLI calls it), once -- it is the slow side;
  index:     pa_mzml_index alone on the file bytes already in memory, and the read of the file into pinned memory;
  to_device: the whole SpectraParser.to_device(0) with the device synchronised, `--reps` times after a warm-up;
  CLI:       python -m pyascore_b200 without and with --gpu_decode, wall clock between the CLI's own stage log lines
             (spectra, identifications, scoring + rows + TSV); the two TSVs are checked byte-identical.
The GPU's name and power limit are read in the same run.  Files go to a temporary directory.  Needs a CUDA device.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def cli_stages(argv):
    """run the CLI; -> seconds of its stages, from the wall clock at each of its log lines"""
    from pyascore_b200.__main__ import build_parser, run
    from pyascore_b200.config import validate_args
    marks = []
    args = build_parser().parse_args(argv)
    validate_args(args)
    t0 = time.perf_counter()
    run(args, log=lambda line: marks.append((time.perf_counter(), line)))
    t1 = time.perf_counter()
    at = {k: next(t for t, line in marks if k in line) for k in ("Reading spectra", "Reading identifications", "Anlyzing")}
    refused = [line for _, line in marks if "GPU decoding refused" in line]
    return dict(spectra_s=at["Reading identifications"] - at["Reading spectra"],
                identifications_s=at["Anlyzing"] - at["Reading identifications"],
                scoring_rows_tsv_s=t1 - at["Anlyzing"], total_s=t1 - t0, refused=refused)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ms2", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "spectra_decode_rates.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("spectra_decode_rates.py needs a CUDA device")
    import _msfiles
    from typed_rates import gpu_info
    from test_gpu_decode import synthetic_run
    from pyascore_b200.parsing import SpectraParser
    from pyascore_b200.parsing.mzml_gpu import index_mzml, read_pinned

    res = dict(gpu=gpu_info(0), ms2=a.ms2, ms1_every=10, files={})
    spectra, queries = synthetic_run(a.ms2, seed=2024, ms1_every=10, peaks=(100, 300))
    res["ms1"] = sum(s["ms_level"] == 1 for s in spectra)
    res["ms2_peaks"] = int(sum(s["mz"].size for s in spectra if s["ms_level"] == 2))
    res["ms1_peaks"] = int(sum(s["mz"].size for s in spectra if s["ms_level"] == 1))
    with tempfile.TemporaryDirectory() as tmp:
        ident = os.path.join(tmp, "i.pep.xml")
        _msfiles.write_pepxml(ident, queries)
        warm = os.path.join(tmp, "warm.mzML")
        _msfiles.write_mzml(warm, spectra[:2000], compress=True)
        SpectraParser(warm, "mzML").to_device(0)
        for compress in (True, False):
            name = "zlib" if compress else "uncompressed"
            spec = os.path.join(tmp, name + ".mzML")
            _msfiles.write_mzml(spec, spectra, compress=compress, inten_bits=32)
            size = os.path.getsize(spec)
            r = dict(file_bytes=size)
            p = SpectraParser(spec, "mzML")
            t = time.perf_counter()
            host = p.to_csr()
            r["stdlib_to_csr_s"] = time.perf_counter() - t
            t = time.perf_counter()
            data = read_pinned(spec)
            r["read_pinned_s"] = time.perf_counter() - t
            idx = []
            for _ in range(a.reps):
                t = time.perf_counter()
                index_mzml(data, 2)
                idx.append(time.perf_counter() - t)
            del data
            dev_s = []
            for _ in range(a.reps):
                torch.cuda.synchronize()
                t = time.perf_counter()
                dev = p.to_device(0)
                torch.cuda.synchronize()
                dev_s.append(time.perf_counter() - t)
            r["index_s"], r["to_device_s"] = idx, dev_s
            r["identical"] = bool(dev.spec_off.cpu().numpy().tobytes() == host.spec_off.tobytes() and
                                  dev.mz.cpu().numpy().tobytes() == np.asarray(host.mz).tobytes() and
                                  (dev.inten32 is None) == (host.inten32 is None) and
                                  (dev.inten32 if dev.inten32 is not None else dev.inten).cpu().numpy().tobytes() ==
                                  np.asarray(host.inten32 if host.inten32 is not None else host.inten).tobytes())
            del dev, host
            for key, s in (("stdlib_to_csr", r["stdlib_to_csr_s"]), ("index", statistics.median(idx)),
                           ("to_device", statistics.median(dev_s))):
                r[key + "_mb_s"] = size / s / 1e6
                r[key + "_kspectra_s"] = len(spectra) / s / 1e3
            outs = {}
            for flag in ([], ["--gpu_decode"]):
                out = os.path.join(tmp, "o%d.tsv" % len(flag))
                r["cli_gpu_decode" if flag else "cli_host"] = cli_stages(flag + [spec, ident, out])
                outs[bool(flag)] = open(out, "rb").read()
            r["cli_tsv_identical"] = outs[True] == outs[False]
            r["cli_rows"] = outs[True].count(b"\n") - 1
            res["files"][name] = r
            print(json.dumps({name: r}, indent=1), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
