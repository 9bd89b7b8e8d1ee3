"""GPU: mzML spectra decoded on the device (SpectraParser.to_device) against the stdlib reader's to_csr, bit for bit, on
the file matrix of tests/test_mzml_index.py and a large mixed-compression file; refused files; and the CLI with
--gpu_decode writing the same TSV as without it."""
import gc

import numpy as np
import pytest

import _msfiles
from pyascore_b200.parsing import SpectraParser
from pyascore_b200.parsing._xml import STD_AA_MASS
from test_mzml_index import MATRIX, SPECTRA, make_spectra, write_mzml_variant

pytestmark = pytest.mark.gpu
PHOSPHO = 79.966331


def assert_same_csr(dev, host):
    """host fields equal, peak arrays equal bit for bit, and the same float32 / float64 intensity choice"""
    import torch
    assert isinstance(dev.mz, torch.Tensor) and dev.mz.is_cuda
    assert isinstance(dev.scans, np.ndarray) and dev.scans.dtype == host.scans.dtype
    assert dev.scans.tobytes() == host.scans.tobytes()
    assert dev.precursor_mz.tobytes() == host.precursor_mz.tobytes()
    assert dev.precursor_charge.dtype == host.precursor_charge.dtype
    assert dev.precursor_charge.tobytes() == host.precursor_charge.tobytes()
    assert dev.spec_off.cpu().numpy().tobytes() == host.spec_off.tobytes()
    assert dev.mz.cpu().numpy().tobytes() == np.asarray(host.mz).tobytes()
    assert (dev.inten is None) == (host.inten is None) and (dev.inten32 is None) == (host.inten32 is None)
    if host.inten is not None:
        assert dev.inten.dtype == torch.float64 and dev.inten.cpu().numpy().tobytes() == np.asarray(host.inten).tobytes()
    else:
        assert dev.inten32.dtype == torch.float32 and dev.inten32.cpu().numpy().tobytes() == np.asarray(host.inten32).tobytes()


@pytest.mark.parametrize("name", sorted(MATRIX))
def test_to_device_equals_to_csr(tmp_path, name):
    path = str(tmp_path / "s.mzML")
    write_mzml_variant(path, make_spectra(300, seed=len(name), **SPECTRA), **MATRIX[name])
    for level in (2, 0):
        p = SpectraParser(path, "mzML", ms_level=level)
        for narrow in (True, False):
            assert_same_csr(p.to_device(0, narrow_intensity=narrow), p.to_csr(narrow_intensity=narrow))


def test_to_device_config1_and_empty_file(tmp_path):
    from test_parsing import load_config1
    spectra, _, _ = load_config1()
    path = str(tmp_path / "c.mzML")
    for compress in (False, True):
        _msfiles.write_mzml(path, spectra, compress=compress, inten_bits=32)
        p = SpectraParser(path, "mzML")
        assert_same_csr(p.to_device(0), p.to_csr())
    _msfiles.write_mzml(path, [])
    p = SpectraParser(path, "mzML")
    got = p.to_device(0)
    assert len(got) == 0 and got.mz.numel() == 0 and got.inten is not None       # to_csr keeps float64 without peaks
    assert_same_csr(got, p.to_csr())


def test_to_device_large_mixed_compression(tmp_path):
    """>= 100 000 spectra, zlib and uncompressed arrays interleaved, MS1 scans interleaved"""
    path = str(tmp_path / "big.mzML")
    write_mzml_variant(path, make_spectra(110000, seed=1, ms1_every=10, max_peaks=60, dup_scans=True), compress="mixed")
    p = SpectraParser(path, "mzML")
    got = p.to_device(0)
    assert len(got) >= 99000
    assert_same_csr(got, p.to_csr())


def _corrupt_first_zlib_array(text, how):
    import base64
    import zlib
    a = text.index("<binary>", text.index("<spectrum ")) + len("<binary>")
    b = text.index("</binary>", a)
    raw = base64.b64decode(text[a:b])
    zlib.decompress(raw)
    raw = raw[:-1] + bytes([raw[-1] ^ 1]) if how == "adler" else raw[:len(raw) // 2]
    return text[:a] + base64.b64encode(raw).decode() + text[b:]


def test_refused_files_leave_nothing_behind(tmp_path):
    import torch
    path = str(tmp_path / "r.mzML")
    write_mzml_variant(path, make_spectra(40, seed=9, empty=False), compress=True)
    text = open(path).read()
    at = text.index('defaultArrayLength="') + len('defaultArrayLength="')
    bad = {"length": text[:at] + "1" + text[at:],                        # 10x the peaks the arrays hold
           "adler": _corrupt_first_zlib_array(text, "adler"),
           "truncated": _corrupt_first_zlib_array(text, "truncated")}
    want = {"length": "decoded length", "adler": "zlib", "truncated": "zlib"}
    gc.collect()
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated(0)
    for what, t in bad.items():
        open(path, "w").write(t)
        with pytest.raises(ValueError, match=want[what]):
            SpectraParser(path, "mzML").to_device(0)
    gc.collect()
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated(0) == before
    # the refusals of the path itself
    write_mzml_variant(path, make_spectra(5, seed=2))
    with pytest.raises(ValueError, match="custom_filter"):
        SpectraParser(path, "mzML", custom_filter=lambda r: True).to_device(0)
    _msfiles.write_mzxml(str(tmp_path / "x.mzXML"), make_spectra(5, seed=2, missing=False))
    with pytest.raises(ValueError, match="mzML files only"):
        SpectraParser(str(tmp_path / "x.mzXML"), "mzXML").to_device(0)


# ---------------------------------------------------------------------------------------------
# CLI
# ---------------------------------------------------------------------------------------------
def synthetic_run(n_ms2, seed=0, ms1_every=10, peaks=(100, 300)):
    """(spectra in file order, pepXML queries): one phospho peptide per MS2 scan (one mod on an S/T/Y, sometimes an
    oxidised M) with peaks at some of its b/y fragments plus noise, and an MS1 scan of ~3000 peaks before every
    `ms1_every` MS2 scans"""
    rng = np.random.default_rng(seed)
    letters = np.array(list("ACDEFGHIKLMNPQRSTVWY"))
    spectra, queries = [], []
    scan = 0
    for i in range(n_ms2):
        if ms1_every and i % ms1_every == 0:
            scan += 1
            k = int(rng.integers(2800, 3200))
            spectra.append(dict(scan=scan, ms_level=1, mz=np.sort(rng.uniform(300, 1800, k)),
                                inten=rng.uniform(1e3, 1e7, k).astype(np.float32)))
        scan += 1
        pep = "".join(rng.choice(letters, int(rng.integers(7, 20)))) + "K"
        sites = [j for j, c in enumerate(pep) if c in "STY"]
        if not sites:
            pep = pep[:2] + "S" + pep[3:]
            sites = [2]
        site = int(rng.choice(sites))
        mods = [(site + 1, STD_AA_MASS[pep[site]] + PHOSPHO)]
        mods += [(j + 1, STD_AA_MASS["M"] + 15.9949) for j, c in enumerate(pep) if c == "M" and rng.random() < 0.5]
        z = int(rng.integers(2, 4))
        prefix = np.cumsum([STD_AA_MASS[c] for c in pep]) + np.array([PHOSPHO if j == site else 0. for j in range(len(pep))]).cumsum()
        frags = np.concatenate([prefix[:-1] + 1.00728, prefix[-1] - prefix[:-1] + 19.01784])
        k = int(rng.integers(*peaks))
        mz = np.concatenate([rng.choice(frags, min(k // 3, frags.size), replace=False), rng.uniform(150, 1800, k - min(k // 3, frags.size))])
        spectra.append(dict(scan=scan, ms_level=2, mz=np.sort(mz), inten=rng.exponential(1e4, mz.size).astype(np.float32),
                            precursor_mz=float((prefix[-1] + 18.0106 + z * 1.00728) / z), precursor_charge=z))
        queries.append(dict(scan=scan, charge=z, hits=[dict(peptide=pep, score=float(rng.uniform(1, 5)),
                                                            mods=sorted(mods))]))
    return spectra, queries


def _run_both(tmp_path, argv, outs):
    """run the CLI without and with --gpu_decode; -> the TSV texts of both runs, per output file"""
    from pyascore_b200.__main__ import main
    texts = {}
    for flag in ([], ["--gpu_decode"]):
        main(flag + argv)
        texts[bool(flag)] = [open(o).read() for o in outs]
    return texts[False], texts[True]


def test_cli_gpu_decode_config1(tmp_path):
    from test_gpu_cli import _argv
    from test_parsing import load_config1
    spectra, queries, expected = load_config1()
    spec, ident, out = str(tmp_path / "s.mzML"), str(tmp_path / "i.pep.xml"), str(tmp_path / "o.tsv")
    _msfiles.write_mzml(spec, spectra, inten_bits=32, compress=True)
    _msfiles.write_pepxml(ident, queries)
    for setting in ("default", "hires_nl"):
        host, dev = _run_both(tmp_path, _argv(expected[setting]["args"]) + [spec, ident, out], [out])
        assert dev == host == [expected[setting]["tsv"]]


def test_cli_gpu_decode_synthetic_20000(tmp_path):
    spectra, queries = synthetic_run(20000, seed=4, ms1_every=0, peaks=(40, 120))
    spec, ident, out = str(tmp_path / "s.mzML"), str(tmp_path / "i.pep.xml"), str(tmp_path / "o.tsv")
    _msfiles.write_mzml(spec, spectra, compress=True)
    _msfiles.write_pepxml(ident, queries)
    host, dev = _run_both(tmp_path, ["--chunk_psms", "6000", spec, ident, out], [out])
    assert dev == host and host[0].count("\n") > 15000


def test_cli_gpu_decode_two_types_and_parameter_file(tmp_path):
    spectra, queries = synthetic_run(3000, seed=5, ms1_every=7, peaks=(40, 120))
    spec, ident = str(tmp_path / "s.mzML"), str(tmp_path / "i.pep.xml")
    out, ox = str(tmp_path / "p.tsv"), str(tmp_path / "ox.tsv")
    _msfiles.write_mzml(spec, spectra, compress=True)
    _msfiles.write_pepxml(ident, queries)
    host, dev = _run_both(tmp_path, ["--extra_mod", "M:15.9949:" + ox, "--chunk_psms", "1000", spec, ident, out], [out, ox])
    assert dev == host and host[1].count("\n") > 100
    from pyascore_b200.__main__ import main
    pf = tmp_path / "p.txt"
    pf.write_text("gpu_decode = 1\nextra_mod = M:15.9949:%s\n" % ox)
    main(["--parameter_file", str(pf), spec, ident, out])
    assert [open(out).read(), open(ox).read()] == host


def test_cli_gpu_decode_refused_file_falls_back(tmp_path):
    from pyascore_b200.__main__ import main
    spectra, queries = synthetic_run(300, seed=6, ms1_every=0, peaks=(40, 80))
    spec, ident, out = str(tmp_path / "s.mzML"), str(tmp_path / "i.pep.xml"), str(tmp_path / "o.tsv")
    _msfiles.write_mzml(spec, spectra)
    _msfiles.write_pepxml(ident, queries)
    main([spec, ident, out])
    want = open(out).read()
    text = open(spec).read()
    open(spec, "w").write(text.replace("<binary>", "<binary><!-- note -->", 1))
    logs = []
    from pyascore_b200.__main__ import build_parser, run
    run(build_parser().parse_args(["--gpu_decode", spec, ident, out]), log=logs.append)
    assert open(out).read() == want
    assert sum("GPU decoding refused" in line for line in logs) == 1
