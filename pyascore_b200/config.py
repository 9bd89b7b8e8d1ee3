"""Command-line options of `python -m pyascore_b200`: the reference's flag set
(pyascore/config.py:19-93: same names, types and defaults, so parameter files and scripts carry
over) plus `--device` / `--chunk_psms` for the GPU pipeline, `--extra_mod` for more modification types per run and `--gpu_decode`
to decode mzML spectra on the GPU."""
import argparse
import re

# (flag, type, default, help) -- one row per reference option (config.py:31-91)
_OPTIONS = [
    ("--residues", str, "STY", "Residues that can carry the modification."),
    ("--mod_mass", float, 79.966331, "Exact modification mass (search engines often report it rounded)."),
    ("--mz_error", float, 0.5, "m/z tolerance for matching a spectral peak to a theoretical fragment."),
    ("--mod_correction_tol", float, 1., "Mass tolerance for recognising a reported modification as the "
                                        "variable one (wide values absorb rounding)."),
    # type=bool as in the reference (config.py:49): any non-empty string enables it
    ("--zero_based", bool, False, "Reported mod positions are 0-based (default: 1-based)."),
    ("--neutral_loss_groups", str, "", "Comma separated residue groups with a neutral loss; lower case = "
                                       "the modified residue loses it ('st' vs 'ST')."),
    ("--neutral_loss_masses", str, "", "Comma separated loss masses, one per group (negative = gain)."),
    ("--static_mod_groups", str, "C", "Comma separated residue groups that always carry a fixed modification."),
    ("--static_mod_masses", str, "57.021464", "Comma separated masses, one per static group."),
    ("--fragment_types", str, "by", "Fragment ion series to score, any of b c y z Z (Z = z+H)."),
    ("--max_fragment_charge", int, 5, "Upper limit of the fragment charge (never above precursor charge - 1)."),
    ("--hit_depth", int, 1, "PSMs taken per scan; negative = all."),
    ("--parameter_file", str, "", "File of 'name = value' lines; command-line flags override it."),
    ("--spec_file_type", str, "mzML", "mzML or mzXML."),
    ("--ident_file_type", str, "pepXML", "pepXML, mzIdentML, percolatorTXT or mokapotTXT."),
]


_SWITCHES = ("gpu_decode",)     # flags without a value on the command line


def args_from_file(file_path):
    """'name = value' lines ('#' starts a comment) -> ['--name', 'value', ...] (config.py:5-17)"""
    out = []
    with open(file_path, "r") as src:
        for line in src:
            m = re.search(r"^([^\s]+)\s*=\s*([^\s]+)$", line.split("#")[0].strip())
            if m is not None:
                if m.group(1) in _SWITCHES:          # 'gpu_decode = 1' turns the switch on, '= 0' leaves it off
                    out += ["--" + m.group(1)] if m.group(2) not in ("0", "False", "false") else []
                else:
                    out += ["--" + m.group(1), m.group(2)]
    return out


def build_parser():
    p = argparse.ArgumentParser(
        prog="pyascore_b200",
        description="PTM localisation with the Ascore algorithm, scored in batches on a B200 GPU. "
                    "Reads spectra (mzML/mzXML) and identifications (pepXML/mzIdentML/percolator/mokapot), "
                    "writes one row per scored PSM.")
    p.add_argument("--match_save", action="store_true",
                   help="Dump the inputs of the scored PSMs (spectra CSR + PSM arrays) to dump_batch.npz.")
    for flag, typ, default, text in _OPTIONS:
        p.add_argument(flag, type=typ, default=default, help=text)
    p.add_argument("--device", type=int, default=0, help="CUDA device ordinal.")
    p.add_argument("--devices", type=str, default="", help="Comma separated CUDA device ordinals: every batch is "
                   "sharded over these GPUs (overrides --device).")
    p.add_argument("--chunk_psms", type=int, default=65536, help="PSMs packed per GPU batch.")
    p.add_argument("--extra_mod", action="append", default=None, metavar="RESIDUES:MASS:OUT_FILE[:NL_GROUPS:NL_MASSES]",
                   help="One more modification type to localise in the same run, written to its own OUT_FILE (the "
                        "spectra are read, copied and binned once for all types). NL_GROUPS / NL_MASSES are comma "
                        "separated as in --neutral_loss_groups / --neutral_loss_masses. Repeatable; in a parameter "
                        "file, one 'extra_mod = ...' line per type. Not combinable with --devices.")
    p.add_argument("--gpu_decode", action="store_true",
                   help="Decode the mzML spectra on the GPU (--device): the host reads the XML structure, the GPU the "
                        "binary arrays, and every batch is scored from device memory. Same output; a file this path "
                        "cannot decode exactly is read by the standard reader instead. 'gpu_decode = 1' in a parameter "
                        "file. Not combinable with --devices or mzXML.")
    p.add_argument("spec_file", type=str, help="MS spectra file.")
    p.add_argument("ident_file", type=str, help="Results of the database search.")
    p.add_argument("out_file", type=str, help="Destination of the tab-separated results.")
    return p


def _validate_residues(residues):
    """reference: __main__.py:49-53"""
    allowed_residues = "ncACDEFGHIKLMNOPQRSTUVWY"
    for aa in residues:
        if aa not in allowed_residues:
            raise ValueError("The residue inputed, {}, is not allowed."
                             " Must be one of: {}".format(aa, allowed_residues))


def parse_extra_mod(text):
    """'RESIDUES:MASS:OUT_FILE[:NL_GROUPS:NL_MASSES]' -> dict(residues, mod_mass, out_file, neutral_loss_groups,
    neutral_loss_masses)"""
    parts = text.split(":")
    if len(parts) not in (3, 5) or not parts[0] or not parts[2]:
        raise ValueError("--extra_mod {!r}: expected RESIDUES:MASS:OUT_FILE or "
                         "RESIDUES:MASS:OUT_FILE:NL_GROUPS:NL_MASSES".format(text))
    try:
        mass = float(parts[1])
    except ValueError:
        raise ValueError("--extra_mod {!r}: the mass {!r} is not a number".format(text, parts[1])) from None
    groups, masses = (parts[3], parts[4]) if len(parts) == 5 else ("", "")
    if len(groups.split(",")) != len(masses.split(",")):
        raise ValueError("--extra_mod {!r}: {} neutral-loss groups but {} masses".format(
            text, len(groups.split(",")), len(masses.split(","))))
    for m in masses.split(",") if masses else ():
        try:
            float(m)
        except ValueError:
            raise ValueError("--extra_mod {!r}: the neutral-loss mass {!r} is not a number".format(text, m)) from None
    return dict(residues=parts[0], mod_mass=mass, out_file=parts[2], neutral_loss_groups=groups,
                neutral_loss_masses=masses)


def validate_args(args):
    """reference: __main__.py:48-65, plus the --extra_mod types"""
    _validate_residues(args.residues)
    extra = getattr(args, "extra_mod", None) or []
    for text in extra:
        _validate_residues(parse_extra_mod(text)["residues"])
    if extra and getattr(args, "devices", ""):
        raise ValueError("--extra_mod cannot be combined with --devices: a run with several modification types "
                         "scores on one GPU (choose it with --device)")
    if getattr(args, "gpu_decode", False):
        if getattr(args, "devices", ""):
            raise ValueError("--gpu_decode cannot be combined with --devices: the spectra are decoded into the memory of "
                             "one GPU (choose it with --device)")
        if args.spec_file_type != "mzML":
            raise ValueError("--gpu_decode reads mzML files only, not {}".format(args.spec_file_type))
    allowed_fragments = "cbyzZ"
    for frag in args.fragment_types:
        if frag not in allowed_fragments:
            raise ValueError("The fragment type inputed, {}, is not allowed."
                             " Must be one of: {}".format(frag, allowed_fragments))
    if args.max_fragment_charge < 1:
        raise ValueError("The max fragment charge must be greater than or equal to 1")
