"""CPU: the host half of GPU mzML decoding -- pa_mzml_index against the stdlib reader (iter_mzml + SpectraParser) on a
matrix of mzML files, and pa_inflate_host (the inflate core of the decode kernel) against Python's zlib.

`write_mzml_variant` and `MATRIX` are shared with tests/test_gpu_decode.py, which decodes the same files on the GPU."""
import base64
import zlib

import numpy as np
import pytest

from pyascore_b200.parsing import SpectraParser
from pyascore_b200.parsing.mzml_gpu import index_mzml

_DT = {"f8": ("MS:1000523", "<f8"), "f4": ("MS:1000521", "<f4"), "i4": ("MS:1000519", "<i4"), "i8": ("MS:1000522", "<i8")}
_ZLIB, _NONE = "MS:1000574", "MS:1000576"


def _payload(values, dt, compress, wrap):
    raw = np.asarray(values).astype(_DT[dt][1]).tobytes()
    if compress:
        raw = zlib.compress(raw)
    text = base64.b64encode(raw).decode()
    if wrap:          # newlines (and indentation) inside <binary>: b64decode skips them
        text = "\n    ".join(text[i:i + 76] for i in range(0, len(text), 76))
    return text


def make_spectra(n, seed=0, ms1_every=0, max_peaks=40, dup_scans=False, missing=True, empty=True):
    """seeded spectra in file order: unsorted scans (duplicates with dup_scans), some without charge / precursor /
    peaks, every ms1_every-th an MS1 scan with many peaks"""
    rng = np.random.default_rng(seed)
    scans = rng.permutation(np.arange(1, n + 1) * 3)
    if dup_scans:
        scans[rng.integers(0, n, n // 4)] = scans[rng.integers(0, n, n // 4)]
    out = []
    for i in range(n):
        ms1 = ms1_every and i % ms1_every == 0
        k = int(rng.integers(200, 400)) if ms1 else int(rng.integers(1, max_peaks))
        if empty and not ms1 and i % 11 == 5:
            k = 0
        s = dict(scan=int(scans[i]), ms_level=1 if ms1 else 2, mz=np.sort(rng.uniform(100, 2000, k)),
                 inten=rng.uniform(0, 1e5, k).astype(np.float32), precursor_mz=float(rng.uniform(300, 1500)),
                 precursor_charge=int(rng.integers(1, 5)))
        if missing and i % 7 == 3:
            s["precursor_charge"] = None
        if missing and i % 13 == 4:
            s["precursor_mz"] = None
        out.append(s)
    return out


def write_mzml_variant(path, spectra, compress=False, mz_dt="f8", in_dt="f4", groups=False, wrap=False, comments=False,
                       entities=False, indexed=True, quote='"', inten_f64_values=False):
    """mzML writer covering what the stdlib reader resolves: compress True / False / "mixed" (per spectrum), array
    types f8/f4/i4/i8, cvParams direct or through referenceableParamGroup (also the ms level), wrapped base64,
    comments and processing instructions between elements, entities in the id, indexed or plain, either quote style"""
    q = quote
    out = ['<?xml version="1.0" encoding="utf-8"?>']
    if indexed:
        out.append('<indexedmzML xmlns="http://psi.hupo.org/ms/mzml">')
    out.append('<mzML xmlns="http://psi.hupo.org/ms/mzml" id="t" version="1.1.0">')
    cv = lambda acc, val="": '<cvParam cvRef=%sMS%s accession=%s%s%s name=%sx%s value=%s%s%s/>' % (q, q, q, acc, q, q, q, q, val, q)
    out.append('<referenceableParamGroupList count="4">'
               '<referenceableParamGroup id="mz_z">%s%s%s</referenceableParamGroup>'
               '<referenceableParamGroup id="mz_n">%s%s%s</referenceableParamGroup>'
               '<referenceableParamGroup id="in_z">%s%s%s</referenceableParamGroup>'
               '<referenceableParamGroup id="in_n">%s%s%s</referenceableParamGroup>'
               '<referenceableParamGroup id="ms2">%s</referenceableParamGroup></referenceableParamGroupList>'
               % (cv(_DT[mz_dt][0]), cv(_ZLIB), cv("MS:1000514"), cv(_DT[mz_dt][0]), cv(_NONE), cv("MS:1000514"),
                  cv(_DT[in_dt][0]), cv(_ZLIB), cv("MS:1000515"), cv(_DT[in_dt][0]), cv(_NONE), cv("MS:1000515"),
                  cv("MS:1000511", "2")))
    out.append('<run id="r"><spectrumList count="%d">' % len(spectra))
    for i, s in enumerate(spectra):
        comp = (i % 3 != 1) if compress == "mixed" else bool(compress)
        sid = "controllerType=0 controllerNumber=1 scan=%d" % s["scan"]
        if entities:
            sid = "controllerType=0 &amp; x=&quot;1&quot; scan=&#%d;%s" % (ord(str(s["scan"])[0]), str(s["scan"])[1:])
        lvl = s.get("ms_level", 2)
        out.append('<spectrum index=%s%d%s id=%s%s%s defaultArrayLength=%s%d%s>' % (q, i, q, q, sid, q, q, len(s["mz"]), q))
        if comments:
            out.append('<!-- spectrum %d <not a tag> --><?pi x?>' % i)
        out.append('<referenceableParamGroupRef ref="ms2"/>' if groups and lvl == 2 else cv("MS:1000511", str(lvl)))
        if lvl > 1 and s.get("precursor_mz") is not None:
            out.append('<precursorList count="1"><precursor><selectedIonList count="1"><selectedIon>' +
                       cv("MS:1000744", repr(float(s["precursor_mz"]))))
            if s.get("precursor_charge") is not None:
                out.append(cv("MS:1000041", str(s["precursor_charge"])))
            out.append('</selectedIon></selectedIonList></precursor></precursorList>')
        inten = s["inten"].astype(np.float64) * (1 + 1e-9) if inten_f64_values else s["inten"]
        vals = dict(mz=s["mz"] * (1000 if mz_dt[0] == "i" else 1), inten=inten)
        out.append('<binaryDataArrayList count="2">')
        for kind, dt, acc in (("mz", mz_dt, "MS:1000514"), ("in", in_dt, "MS:1000515")):
            if groups:
                params = '<referenceableParamGroupRef ref="%s_%s"/>' % (kind, "z" if comp else "n")
            else:
                params = cv(_DT[dt][0]) + cv(_ZLIB if comp else _NONE) + cv(acc)
            if comments:
                params += '<!-- array -->'
            out.append('<binaryDataArray encodedLength="0">%s<binary>%s</binary></binaryDataArray>'
                       % (params, _payload(vals["mz" if kind == "mz" else "inten"], dt, comp, wrap)))
        out.append('</binaryDataArrayList></spectrum>')
    out.append('</spectrumList></run></mzML>')
    if indexed:
        out.append('<indexList count="1"><index name="spectrum"><offset idRef="x">0</offset></index></indexList>'
                   '<indexListOffset>0</indexListOffset></indexedmzML>')
    with open(path, "w") as f:
        f.write("\n".join(out))


MATRIX = {
    "plain_f8_f4": dict(),
    "zlib_f8_f4": dict(compress=True),
    "mixed_groups": dict(compress="mixed", groups=True),
    "zlib_f4_f8": dict(compress=True, mz_dt="f4", in_dt="f8"),
    "ints_i8_i4": dict(mz_dt="i8", in_dt="i4"),
    "zlib_i4_i8": dict(compress=True, mz_dt="i4", in_dt="i8"),
    "wrapped_comments": dict(compress="mixed", wrap=True, comments=True),
    "entities_plain_file": dict(entities=True, indexed=False, quote="'"),
    "f8_intensities": dict(compress=True, in_dt="f8", inten_f64_values=True),
}
SPECTRA = dict(ms1_every=4, dup_scans=True)


def _compare_index(path, ms_level):
    ix = index_mzml(open(path, "rb").read(), ms_level)
    recs = SpectraParser(path, "mzML", ms_level=ms_level).to_list()
    assert ix["scans"].tolist() == [r["scan"] for r in recs]
    assert ix["ms_level"].tolist() == [r["ms_level"] for r in recs]
    pmz = np.array([np.nan if r["precursor_mz"] is None else r["precursor_mz"] for r in recs], np.float64)
    assert pmz.tobytes() == ix["precursor_mz"].tobytes()
    assert ix["precursor_charge"].tolist() == [0 if r["precursor_charge"] is None else r["precursor_charge"] for r in recs]
    assert np.diff(ix["spec_off"]).tolist() == [r["mz_values"].size for r in recs]
    # the payload ranges decode, with Python's base64 / zlib, to the stdlib reader's arrays
    data = open(path, "rb").read()
    seen = 0
    for a in ix["arrays"]:
        raw = base64.b64decode(data[a["text_off"]:a["text_off"] + a["text_len"]])
        if a["flags"] & 1 and raw:
            raw = zlib.decompress(raw)
        vals = np.frombuffer(raw, ["<f8", "<f4", "<i4", "<i8"][a["dtype"]]).astype(np.float64)
        r = recs[a["spec"]]
        assert vals.size == a["count"] == r["mz_values"].size and a["out_off"] == ix["spec_off"][a["spec"]]
        want = r["intensity_values"] if a["flags"] & 2 else r["mz_values"]
        assert vals.tobytes() == want.tobytes()
        seen += 1
    return ix, recs, seen


@pytest.mark.parametrize("name", sorted(MATRIX))
def test_index_matches_stdlib_reader(tmp_path, name):
    path = str(tmp_path / "s.mzML")
    write_mzml_variant(path, make_spectra(60, seed=len(name), **SPECTRA), **MATRIX[name])
    for level in (2, 1, 0):
        ix, recs, seen = _compare_index(path, level)
        assert len(recs) > 0 and seen == 2 * len(recs)          # every spectrum of the writer has both arrays
    assert set(index_mzml(open(path, "rb").read(), 2)["ms_level"]) == {2}


def test_index_edge_spectra(tmp_path):
    """precursor without charge, precursor without m/z value, no precursorList, no arrays, one array only, a later
    array of the same kind wins, first precursor's first selectedIon only, scan-less id"""
    path = tmp_path / "e.mzML"
    arr = lambda acc, vals: ('<binaryDataArray><cvParam accession="MS:1000523"/><cvParam accession="%s"/><binary>%s'
                             '</binary></binaryDataArray>' % (acc, base64.b64encode(np.float64(vals).tobytes()).decode()))
    lvl = '<cvParam accession="MS:1000511" value="2"/>'
    ion = lambda *cvs: ('<precursorList count="1"><precursor><selectedIonList><selectedIon>%s</selectedIon>'
                        '<selectedIon><cvParam accession="MS:1000744" value="9"/><cvParam accession="MS:1000041" value="9"/>'
                        '</selectedIon></selectedIonList></precursor></precursorList>' % "".join(cvs))
    body = [
        ('id="scan=5" defaultArrayLength="2"', lvl + ion('<cvParam accession="MS:1000744" value="500.5"/>') +
         '<binaryDataArrayList>%s%s</binaryDataArrayList>' % (arr("MS:1000514", [1, 2]), arr("MS:1000515", [3, 4]))),
        ('id="scan=4" defaultArrayLength="2"', lvl + ion('<cvParam accession="MS:1000744"/>', '<cvParam accession="MS:1000041" value="2"/>') +
         '<binaryDataArrayList>%s</binaryDataArrayList>' % arr("MS:1000514", [1, 2])),
        ('id="scan=3" defaultArrayLength="1"', lvl + '<binaryDataArrayList>%s%s%s</binaryDataArrayList>' % (
            arr("MS:1000514", [7, 8]), arr("MS:1000515", [5]), arr("MS:1000514", [6]))),
        ('id="nothing here" defaultArrayLength="0"', lvl + ion('<cvParam accession="MS:1000041" value=" 3 "/>',
                                                               '<cvParam accession="MS:1000744" value=" 1e3 "/>')),
        ('id="scan=x scan=2" defaultArrayLength="0"', lvl + '<precursorList count="0"/>'),
    ]
    text = '<?xml version="1.0"?><mzML><run><spectrumList>%s</spectrumList></run></mzML>' % "".join(
        "<spectrum %s>%s</spectrum>" % b for b in body)
    path.write_text(text)
    ix, recs, seen = _compare_index(str(path), 2)
    assert ix["scans"].tolist() == [-1, 2, 3, 4, 5] and seen == 4
    assert ix["precursor_charge"].tolist() == [3, 0, 0, 0, 0]


def _refusal(path):
    with pytest.raises(ValueError) as want:
        SpectraParser(path, "mzML").to_list()
    with pytest.raises(ValueError) as got:
        index_mzml(open(path, "rb").read(), 2)
    return str(want.value), str(got.value)


def test_same_refusals_as_stdlib(tmp_path):
    spectra = make_spectra(6, seed=3)
    path = str(tmp_path / "m.mzML")
    write_mzml_variant(path, spectra)
    text = open(path).read()
    # several precursors (also announced by count only)
    bad = text.replace('<precursorList count="1">', '<precursorList count="2">', 1)
    open(path, "w").write(bad)
    want, got = _refusal(path)
    assert want == got == "Multiple precursors not supported at this time"
    bad = text.replace('</precursor></precursorList>', '</precursor><precursor/></precursorList>', 1).replace(
        '<precursorList count="1">', '<precursorList>', 1)
    open(path, "w").write(bad)
    assert _refusal(path)[0] == _refusal(path)[1]
    # numpress, also on an MS1 spectrum the level filter drops
    for level in ("2", "1"):
        bad = text.replace('accession="MS:1000511" name="x" value="2"', 'accession="MS:1000511" name="x" value="%s"' % level, 1)
        at = bad.index("<spectrum ")
        bad = bad[:at] + bad[at:].replace('accession="MS:1000576"', 'accession="MS:1002312"', 1)
        open(path, "w").write(bad)
        want, got = _refusal(path)
        assert want == got and "numpress" in got


def test_refusals_of_this_path(tmp_path):
    """files the stdlib reader reads but whose raw payload bytes are not its text, or whose layout is unknown"""
    path = str(tmp_path / "r.mzML")
    write_mzml_variant(path, make_spectra(4, seed=5, empty=False))
    text = open(path).read()
    cases = {
        "markup": text.replace("<binary>", "<binary><!-- c -->", 1),
        "different lengths": text.replace('<binaryDataArray encodedLength="0">', '<binaryDataArray arrayLength="1">', 1),
        "arrayLength": text.replace('defaultArrayLength', 'otherLength', 1),
        "DOCTYPE": text.replace('?>', '?><!DOCTYPE indexedmzML [<!ENTITY e "x">]>', 1),
    }
    for what, bad in cases.items():
        open(path, "w").write(bad)
        SpectraParser(path, "mzML").to_list()
        with pytest.raises(ValueError):
            index_mzml(bad.encode(), 2)


def test_index_of_the_config1_file(tmp_path):
    from test_parsing import load_config1
    import _msfiles
    spectra, _, _ = load_config1()
    path = str(tmp_path / "c.mzML")
    for compress in (False, True):
        _msfiles.write_mzml(path, spectra, compress=compress, inten_bits=32)
        ix, recs, seen = _compare_index(path, 2)
        assert len(recs) == len(spectra)


# ---------------------------------------------------------------------------------------------
# pa_inflate_host against zlib
# ---------------------------------------------------------------------------------------------
def _inflate(data, cap):
    import ctypes as C
    from pyascore_b200 import _lib
    L = _lib.load()
    src = np.frombuffer(data, np.uint8) if data else np.zeros(1, np.uint8)
    out = np.zeros(max(cap, 1), np.uint8)
    n = L.pa_inflate_host(src.ctypes.data, len(data), out.ctypes.data, cap)
    return n, out[:max(n, 0)].tobytes()


def _inputs():
    rng = np.random.default_rng(11)
    return {"random": rng.bytes(70000),
            "floats": np.sort(rng.uniform(100, 2000, 9000)).tobytes() + rng.uniform(0, 1e5, 9000).astype(np.float32).tobytes(),
            "repetitive": b"\x00" * 50000 + b"ab" * 20000 + bytes(range(256)) * 100 + b"xyz" * 7,
            "tiny": b"a", "empty": b""}


@pytest.mark.parametrize("strategy", ["Z_DEFAULT_STRATEGY", "Z_FILTERED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FIXED"])
def test_inflate_matches_zlib(strategy):
    for name, data in _inputs().items():
        for level in range(10):
            c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, getattr(zlib, strategy))
            comp = c.compress(data) + c.flush()
            n, out = _inflate(comp, len(data))
            assert n == len(data) and out == data, (name, level, strategy)
            if level in (0, 6):
                assert _inflate(zlib.compress(data, level), len(data))[1] == data
                assert _inflate(zlib.compress(data, level) + b"trailing", len(data))[1] == data   # ignored, as zlib does


def test_inflate_rejects_what_zlib_rejects():
    data = _inputs()["floats"]
    comp = zlib.compress(data, 6)

    def rejected(bad):
        with pytest.raises(zlib.error):
            zlib.decompress(bad)
        return _inflate(bad, len(data))[0] == -1

    for cut in (1, 2, 10, len(comp) // 2, len(comp) - 5, len(comp) - 1):
        assert rejected(comp[:cut])                                        # truncated
    assert rejected(bytes([comp[0] ^ 0x10]) + comp[1:])                  # bad header (method / check bits)
    assert rejected(comp[:-1] + bytes([comp[-1] ^ 1]))                   # bad Adler-32
    assert rejected(b"\x78\x9c\xff" + comp[3:])                           # reserved block type
    assert rejected(b"\x78\xbb" + comp[2:])                               # preset dictionary
    stored = zlib.compress(data[:1000], 0)
    assert rejected(stored[:3] + bytes([stored[3] ^ 0xff]) + stored[4:])  # stored block LEN / NLEN disagree
    assert _inflate(comp, len(data) - 1)[0] == -2                         # output beyond the capacity


def test_gpu_decode_option():
    from pyascore_b200.config import args_from_file, build_parser, validate_args
    p = build_parser()
    parse = lambda extra: p.parse_args(extra + ["s.mzML", "i.pep.xml", "o.tsv"])
    assert parse([]).gpu_decode is False and parse(["--gpu_decode"]).gpu_decode is True
    validate_args(parse(["--gpu_decode", "--device", "1"]))
    with pytest.raises(ValueError, match="--gpu_decode cannot be combined with --devices"):
        validate_args(parse(["--gpu_decode", "--devices", "0,1"]))
    with pytest.raises(ValueError, match="--gpu_decode reads mzML files only"):
        validate_args(parse(["--gpu_decode", "--spec_file_type", "mzXML"]))
    validate_args(parse(["--devices", "0,1"]))
    validate_args(parse(["--spec_file_type", "mzXML"]))


def test_gpu_decode_parameter_file(tmp_path):
    from pyascore_b200.config import args_from_file, build_parser
    p = build_parser()
    for value, want in (("1", True), ("0", False)):
        pf = tmp_path / "p.txt"
        pf.write_text("hit_depth = 2\ngpu_decode = %s\n" % value)
        a = p.parse_args(args_from_file(str(pf)) + ["s", "i", "o"])
        assert a.gpu_decode is want and a.hit_depth == 2 and a.spec_file == "s"
