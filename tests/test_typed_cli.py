"""CPU: the host side of several modification types per run -- the packer's row order and types, and the
--extra_mod option (parsing, validation, parameter files, the refusal of --devices)."""
import numpy as np
import pytest

from pyascore_b200.config import args_from_file, build_parser, parse_extra_mod, validate_args
from pyascore_b200.parsing import iter_batches
from pyascore_b200.parsing.spec_parsers import SpectraCSR

PH, AC, OX = 79.966331, 42.010565, 15.9949


def _csr():
    rng = np.random.default_rng(0)
    off = np.array([0, 5, 5, 14, 18], np.int64)
    return SpectraCSR(np.array([10, 20, 30, 40]), np.full(4, np.nan), np.array([3, 0, 2, 0], np.int32), off,
                      rng.uniform(100, 900, off[-1]), rng.uniform(1, 9, off[-1]))


def _records():
    return [dict(scan=10, charge_state=0, peptide="ASTK", mod_positions=[2], mod_masses=[PH]),
            dict(scan=10, charge_state=0, peptide="AKTK", mod_positions=[2], mod_masses=[AC]),
            dict(scan=10, charge_state=0, peptide="ASKM", mod_positions=[3, 4], mod_masses=[AC, OX]),
            dict(scan=30, charge_state=4, peptide="CSYK", mod_positions=[1, 2], mod_masses=[57.021464, PH]),
            dict(scan=40, charge_state=None, peptide="MSKK", mod_positions=[1, 3], mod_masses=[OX, AC])]


def test_packer_types_row_order():
    csr, recs = _csr(), _records()
    types = [("STY", PH), ("K", AC), ("M", OX)]
    (scans, b), = list(iter_batches(csr, [recs, recs, recs], hit_depth=-1, types=types))
    # per scan: the hits of type 0, then type 1, then type 2; a row only where the type has a variable mod
    assert list(scans) == [10, 10, 10, 10, 30, 40, 40]
    assert list(b["psm_type"]) == [0, 1, 1, 2, 0, 1, 2] and b["psm_type"].dtype == np.uint8
    assert list(b["psm_spec"]) == [0, 0, 0, 0, 2, 3, 3]
    assert bytes(b["pep"]) == b"ASTKAKTKASKMASKMCSYKMSKKMSKK" and list(b["n_mod"]) == [1, 1, 1, 1, 1, 1, 1]
    # the other type's mod is a fixed mod of the row
    assert list(b["aux_off"]) == [0, 0, 0, 1, 2, 3, 4, 5] and list(b["aux_pos"]) == [4, 3, 1, 1, 3]
    np.testing.assert_array_equal(b["aux_mass"], np.float32([OX, AC, 57.021464, OX, AC]))
    # hit_depth counts hits per type (the first hit of scan 10 has no acetyl: no type-1 row there), chunks are cut on
    # scan boundaries
    chunks = list(iter_batches(csr, [recs, recs], hit_depth=1, types=types[:2], chunk_psms=1))
    assert [list(s) for s, _ in chunks] == [[10], [30], [40]]
    assert [list(c["psm_type"]) for _, c in chunks] == [[0], [0], [1]]
    (scans, b), = list(iter_batches(csr, [recs, recs], hit_depth=2, types=types[:2]))
    assert list(scans) == [10, 10, 30, 40] and list(b["psm_type"]) == [0, 1, 0, 1]
    # one type: today's batches, without a psm_type array
    (_, one), = list(iter_batches(csr, recs, hit_depth=-1, types=types[:1]))
    (_, dflt), = list(iter_batches(csr, recs, hit_depth=-1))
    assert "psm_type" not in one and one.keys() == dflt.keys()
    assert all(np.array_equal(one[k], dflt[k]) for k in one if k not in ("mz", "inten", "spec_off"))
    with pytest.raises(ValueError):
        list(iter_batches(csr, [recs], types=types[:2]))
    with pytest.raises(ValueError):
        list(iter_batches(csr, [recs, recs[:3]], types=types[:2], hit_depth=-1))


def _args(extra):
    p = build_parser()
    return p.parse_args(extra + ["s.mzML", "i.pep.xml", "o.tsv"])


def test_extra_mod_parsing():
    assert parse_extra_mod("K:42.010565:acetyl.tsv") == dict(
        residues="K", mod_mass=42.010565, out_file="acetyl.tsv", neutral_loss_groups="", neutral_loss_masses="")
    assert parse_extra_mod("ST:79.966331:p.tsv:st,y:97.9769,-1.5") == dict(
        residues="ST", mod_mass=79.966331, out_file="p.tsv", neutral_loss_groups="st,y",
        neutral_loss_masses="97.9769,-1.5")
    for bad in ("K:42.01", "K:x:a.tsv", ":42.01:a.tsv", "K:42.01:", "K:42.01:a.tsv:st", "K:42.01:a.tsv:st,y:97.9",
                "K:42.01:a.tsv:st:abc"):
        with pytest.raises(ValueError):
            parse_extra_mod(bad)
    a = _args(["--extra_mod", "K:42.010565:ac.tsv", "--extra_mod", "M:15.9949:ox.tsv"])
    assert a.extra_mod == ["K:42.010565:ac.tsv", "M:15.9949:ox.tsv"]
    validate_args(a)
    assert _args([]).extra_mod is None
    validate_args(_args([]))


def test_extra_mod_residues_validated_like_residues():
    with pytest.raises(ValueError, match="The residue inputed, X, is not allowed"):
        validate_args(_args(["--extra_mod", "KX:42.01:ac.tsv"]))
    with pytest.raises(ValueError, match="The residue inputed, X, is not allowed"):
        validate_args(_args(["--residues", "X"]))


def test_extra_mod_parameter_file(tmp_path):
    pf = tmp_path / "p.txt"
    pf.write_text("hit_depth = 2\nextra_mod = K:42.010565:acetyl.tsv\n# a comment\nextra_mod = M:15.9949:ox.tsv:m:63.998285\n")
    p = build_parser()
    argv = ["--parameter_file", str(pf), "s", "i", "o"]
    a = p.parse_args(args_from_file(str(pf)) + argv)
    assert a.extra_mod == ["K:42.010565:acetyl.tsv", "M:15.9949:ox.tsv:m:63.998285"] and a.hit_depth == 2
    validate_args(a)
    # the command line adds types to those of the file
    a = p.parse_args(args_from_file(str(pf)) + ["--extra_mod", "Y:1.0:y.tsv"] + argv)
    assert len(a.extra_mod) == 3


def test_extra_mod_refused_with_devices():
    with pytest.raises(ValueError, match="--extra_mod cannot be combined with --devices"):
        validate_args(_args(["--extra_mod", "K:42.010565:ac.tsv", "--devices", "0,1"]))
    validate_args(_args(["--devices", "0,1"]))
