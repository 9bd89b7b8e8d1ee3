"""`python -m pyascore_b200 spec_file ident_file out_file [options]` -- the reference's CLI
(pyascore/__main__.py:114-173) with the per-PSM Python loop replaced by batched GPU scoring:

    parse spectra -> one pinned CSR block        (SpectraParser.to_csr)
    parse identifications, sort by scan          (IdentificationParser.to_list)
    pack chunks of PSMs (hit_depth, mod split, charge rule)  ||  score previous chunk on the GPU
    format rows, write the TSV (same columns and number formatting)

With --extra_mod, the spectra are parsed once and each batch holds the rows of every modification type, scored in
one GPU call (score_typed); each type writes its own TSV.  With --gpu_decode, the spectra of an mzML file are decoded on
the GPU (SpectraParser.to_device) and every batch is scored from device memory.
"""
import sys
from datetime import datetime

import numpy as np

from .batch import MultiScorer, Scorer, add_mod_off, score_typed
from .config import args_from_file, build_parser, parse_extra_mod, validate_args
from .parsing import (COMMON_MODS, IdentificationParser, MassCorrector, SpectraParser, iter_batches, result_rows,
                      score_stream, write_tsv)


def _stamp():
    return datetime.now().strftime("%m/%d/%y %H:%M:%S")


def static_mod_dict(args):
    """reference: __main__.py:26-29"""
    out = {}
    for group, mass in zip(args.static_mod_groups.split(","), args.static_mod_masses.split(",")):
        out.update({aa: float(mass) for aa in group})
    return out


def parse_identifications(args, residues=None, mod_mass=None):
    """reference: __main__.py:22-45 -> scan-sorted PSM records, mass-corrected for the variable modification
    (residues, mod_mass) -- default: --residues / --mod_mass"""
    residues = args.residues if residues is None else residues
    mod_mass = args.mod_mass if mod_mass is None else mod_mass
    static_mods = static_mod_dict(args)
    mods = COMMON_MODS.copy()
    mods.update({aa: mod_mass for aa in residues})
    mods.update(static_mods)
    parser = IdentificationParser(args.ident_file, args.ident_file_type, MassCorrector(mod_mass_dict=mods),
                                  static_mods=static_mods)
    return sorted(parser.to_list(), key=lambda m: m["scan"])


def build_scorer(args):
    """reference: __main__.py:68-80 (bin_size 100, n_top 10 are fixed there too)"""
    devices = [int(d) for d in getattr(args, "devices", "").split(",") if d.strip() != ""]
    if devices:
        scorer = MultiScorer(100., 10, args.residues, args.mod_mass, args.mz_error, args.fragment_types, devices=devices)
    else:
        scorer = Scorer(100., 10, args.residues, args.mod_mass, args.mz_error, args.fragment_types, device=args.device)
    if args.neutral_loss_groups and args.neutral_loss_masses:
        for g, m in zip(args.neutral_loss_groups.split(","), args.neutral_loss_masses.split(",")):
            scorer.add_neutral_loss(g, float(m))
    return scorer


def read_spectra(args, log=print):
    """The run's spectra: with --gpu_decode decoded on the GPU (--device), else -- or when that path refuses the file, which
    is logged -- the pinned CSR block of the stdlib reader"""
    parser = SpectraParser(args.spec_file, args.spec_file_type)
    if getattr(args, "gpu_decode", False):
        try:
            return parser.to_device(args.device)
        except ValueError as e:
            log("{} -- GPU decoding refused, reading the spectra on the host: {}".format(_stamp(), e))
    return parser.to_csr()


def score_on_device(score, spectra):
    """`score` (batch -> results) as the CLI calls it: unchanged for host spectra; for spectra on a GPU each batch's PSM
    arrays go to that device, `score` takes the device-resident path and the results come back to the host"""
    if isinstance(spectra.mz, np.ndarray):
        return score
    import torch
    dev = spectra.mz.device

    def run(batch):
        add_mod_off(batch)
        on_dev = {k: torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v for k, v in batch.items()}
        torch.cuda.current_stream(dev).synchronize()
        return {k: v.cpu().numpy() for k, v in score(on_dev).items()}
    return run


def _host_arrays(batch):
    return {k: v if isinstance(v, np.ndarray) else v.cpu().numpy() for k, v in batch.items() if v is not None}


def mod_types(args):
    """the modification types of a run: type 0 = --residues / --mod_mass / the neutral-loss flags / out_file, then one
    per --extra_mod"""
    return [dict(residues=args.residues, mod_mass=args.mod_mass, out_file=args.out_file,
                 neutral_loss_groups=args.neutral_loss_groups, neutral_loss_masses=args.neutral_loss_masses)] + \
        [parse_extra_mod(text) for text in args.extra_mod]


def run_typed(args, log=print):
    """A run with --extra_mod: the spectra are parsed once and every batch is scored for all modification types in
    one GPU call (score_typed); each type's rows go to its own TSV, the same file a run of that type alone writes."""
    types = mod_types(args)
    log("{} -- Ascore Started".format(_stamp()))
    log("{} -- Reading spectra from: {}".format(_stamp(), args.spec_file))
    spectra = read_spectra(args, log)
    log("{} -- Reading identifications from: {}".format(_stamp(), args.ident_file))
    psms = [parse_identifications(args, t["residues"], t["mod_mass"]) for t in types]
    log("{} -- Anlyzing PSMs".format(_stamp()))
    scorers = []
    rows = [[] for _ in types]
    n_psm = [0] * len(types)
    saved = []
    try:
        for t in types:
            scorers.append(Scorer(100., 10, t["residues"], t["mod_mass"], args.mz_error, args.fragment_types,
                                  device=args.device))
            if t["neutral_loss_groups"] and t["neutral_loss_masses"]:
                for g, m in zip(t["neutral_loss_groups"].split(","), t["neutral_loss_masses"].split(",")):
                    scorers[-1].add_neutral_loss(g, float(m))
        batches = iter_batches(spectra, psms, chunk_psms=args.chunk_psms,
                               types=[(t["residues"], t["mod_mass"]) for t in types],
                               mod_correction_tol=args.mod_correction_tol, zero_based=args.zero_based,
                               max_fragment_charge=args.max_fragment_charge, hit_depth=args.hit_depth)
        score = score_on_device(lambda b: score_typed(scorers, b, b["psm_type"]), spectra)
        for scans, batch, res in score_stream(score, batches):
            for t, sc in enumerate(scorers):
                sel = np.flatnonzero(batch["psm_type"] == t)
                rows[t].extend(result_rows(sc, scans, batch, res, rows_of=sel))
                n_psm[t] += int(sel.size)
            if args.match_save:
                saved.append((scans, batch))
    finally:
        for sc in scorers:
            sc.close()
    if args.match_save and saved:
        scans, batch = saved[-1]
        np.savez("dump_batch.npz", scans=scans, **_host_arrays(batch))
    for t, typ in enumerate(types):
        if len(rows[t]) != n_psm[t]:
            log("{} -- {} of {} PSMs of {} could not be scored (see the warnings) and have no row in the output".format(
                _stamp(), n_psm[t] - len(rows[t]), n_psm[t], typ["out_file"]))
        write_tsv(typ["out_file"], rows[t])
    log("{} -- Ascore Completed".format(_stamp()))
    return rows


def run(args, log=print):
    if getattr(args, "extra_mod", None):
        return run_typed(args, log)
    log("{} -- Ascore Started".format(_stamp()))
    log("{} -- Reading spectra from: {}".format(_stamp(), args.spec_file))
    spectra = read_spectra(args, log)
    log("{} -- Reading identifications from: {}".format(_stamp(), args.ident_file))
    psms = parse_identifications(args)
    log("{} -- Anlyzing PSMs".format(_stamp()))
    scorer = build_scorer(args)
    batches = iter_batches(spectra, psms, chunk_psms=args.chunk_psms, residues=args.residues,
                           mod_mass=args.mod_mass, mod_correction_tol=args.mod_correction_tol,
                           zero_based=args.zero_based, max_fragment_charge=args.max_fragment_charge,
                           hit_depth=args.hit_depth)
    rows = []
    saved = []
    n_psm = 0
    try:
        for scans, batch, res in score_stream(score_on_device(scorer.score_batch, spectra), batches):
            rows.extend(result_rows(scorer, scans, batch, res))
            n_psm += int(scans.size)
            if args.match_save:
                saved.append((scans, batch))
    finally:
        scorer.close()
    if args.match_save and saved:
        scans, batch = saved[-1]
        np.savez("dump_batch.npz", scans=scans, **_host_arrays(batch))
    if len(rows) != n_psm:
        # the reference would have written a row for these (or crashed on them): make the difference visible
        log("{} -- {} of {} PSMs could not be scored (see the warnings) and have no row in the output".format(
            _stamp(), n_psm - len(rows), n_psm))
    write_tsv(args.out_file, rows)
    log("{} -- Ascore Completed".format(_stamp()))
    return rows


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.parameter_file:
        args = parser.parse_args(args_from_file(args.parameter_file) + argv)
    validate_args(args)
    run(args)


if __name__ == "__main__":
    main()
