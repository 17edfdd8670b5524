#! /usr/bin/env python
"""Drop-in for scripts/metalign.py of nlapier2/Metalign: same flags; database selection runs on the GPU
(metalign_b200.select_db), then the reference's own alignment/profiling stage (scripts/map_and_profile.py,
minimap2 -- out of scope here, used unchanged if it is importable) runs on the files selection wrote.
With --select_only, or when map_and_profile is not importable, it stops after selection and keeps temp_dir.
Under torchrun every rank takes part in the selection (metalign_b200.select_db) and rank 0 alone maps and profiles."""
from __future__ import annotations

import argparse
import shutil
import sys

from . import select_db as select


def metalign_parseargs(argv=None):
    p = argparse.ArgumentParser(description="Metalign pipeline with B200-native database selection.")
    p.add_argument("reads", help="reads file")
    p.add_argument("data", help="data/ directory")
    p.add_argument("--cutoff", type=float, default=0.01)
    p.add_argument("--db_dir", default="AUTO")
    p.add_argument("--dbinfo_in", default="AUTO")
    p.add_argument("--keep_temp_files", action="store_true")
    p.add_argument("--input_type", default="AUTO", choices=["fastq", "fasta", "AUTO"])
    p.add_argument("--length_normalize", action="store_true")
    p.add_argument("--low_mem", action="store_true")
    p.add_argument("--min_abundance", type=float, default=10 ** -4)
    p.add_argument("--no_quantify_unmapped", action="store_true")
    p.add_argument("--output", default="abundances.tsv")
    p.add_argument("--pct_id", type=float, default=0.5)
    p.add_argument("--precise", action="store_true")
    p.add_argument("--rank_renormalize", action="store_true")
    p.add_argument("--read_cutoff", type=int, default=1)
    p.add_argument("--sampleID", default="NONE")
    p.add_argument("--sensitive", action="store_true")
    p.add_argument("--strain_level", action="store_true")
    p.add_argument("--temp_dir", default="AUTO/")
    p.add_argument("--threads", type=int, default=4)
    p.add_argument("--verbose", action="store_true")
    # additions
    p.add_argument("--db_file", default="AUTO")
    p.add_argument("--gate", default="exact", choices=["exact", "none"])
    p.add_argument("--device", type=int, default=0)
    p.add_argument("--select_only", action="store_true", help="stop after database selection")
    return p.parse_args(argv)


def main(argv=None):
    args = metalign_parseargs(argv)
    select.init_ranks(args)
    rank, world = select.ranks()
    select.resolve_data(args)
    if args.temp_dir == "AUTO/":
        args.temp_dir = select.shared_mkdtemp(args.data, rank, world)
    if not args.temp_dir.endswith("/"):
        args.temp_dir += "/"
    if args.sensitive and args.precise:
        sys.exit("You cannot use both --sensitive and --precise.")
    if args.sensitive:                         # metalign.py:70-71 of the reference
        args.cutoff = 0.0
    elif args.precise:
        args.read_cutoff, args.min_abundance = 100, 0.1
    # wiring shared with the mapper, as metalign.py:77-81
    args.db = args.temp_dir + "cmashed_db.fna"
    args.dbinfo = args.temp_dir + "subset_db_info.txt"
    args.dbinfo_out = args.dbinfo
    args.infiles = [args.reads]
    args.cmash_results = "NONE"

    select.select_main(args)
    mapper = None
    if rank != 0:
        return
    if not args.select_only:
        try:
            import map_and_profile as mapper      # the reference's scripts/ directory on PYTHONPATH
        except ImportError:
            # the reference always goes on to mapper.map_main(args) (metalign.py:85): a run that cannot must not look
            # like one that did -- no abundances file was written
            sys.exit("Error: map_and_profile (the reference's alignment/profiling stage, scripts/ of nlapier2/Metalign) is "
                     "not importable, so %s was not written; selection outputs are in %s (use --select_only to stop "
                     "after database selection)" % (args.output, args.temp_dir))
    if mapper is not None:
        mapper.map_main(args)
        if not args.keep_temp_files:
            shutil.rmtree(args.temp_dir, ignore_errors=True)


if __name__ == "__main__":
    main()
