#! /usr/bin/env python
"""Drop-in for scripts/select_db.py of nlapier2/Metalign: same command line, same `select_main(args)` entry
point (called by metalign.py:84 of the reference), same files out (`cmash_query_results.csv`, the subset
FASTA `cmashed_db.fna`, `subset_db_info.txt`).  What changes is behind `run_kmc_steps` and
`run_cmash_and_cutoff`: instead of starting kmc / kmc_tools / kmc_dump / StreamingQueryDNADatabase.py
(select_db.py:50-76) the reads are streamed to the GPU library and the containment table comes back.

The database is the native file `data/cmash_db_n1000_k60.mlgdb` (metalign_b200.dbformat) in place of
cmash_db_n1000_k60.h5 / _30-60-10.bf / _dump.kmc_* (select_db.py:44,69,70).

Extra, optional flags (not in the reference): --db_file, --gate, --device, --k_range, --read_kmer_budget,
--read_kmer_passes.
"""
from __future__ import annotations

import argparse
import gzip
import os
import shutil
import sys
import tempfile

DB_BASENAME = "cmash_db_n1000_k60.mlgdb"
HEADER_LINES = ("Accesion\tLength\tTaxID\tLineage\tTaxID_Lineage\n",          # sic: spelling of the reference, select_db.py:109
                "Unmapped\t0\tUnmapped\t|||||||Unmapped\t|||||||Unmapped\n")


_T0 = None


def _tick(label):
    """MLG_TIMING=1: stage times on stderr (seconds since the module was imported)"""
    if os.environ.get("MLG_TIMING"):
        import time
        global _T0
        now = time.perf_counter()
        if _T0 is None:
            _T0 = now
        sys.stderr.write("[mlg %7.3f s] %s\n" % (now - _T0, label))


def select_parseargs(argv=None):
    p = argparse.ArgumentParser(description="Score every database genome against the reads (containment min-hash, "
                                            "k=30..60) and write the reduced database to align to.")
    p.add_argument("reads", help="reads file (FASTA/FASTQ, optionally .gz)")
    p.add_argument("data", help="data/ directory (database, db_info.txt, organism_files/)")
    p.add_argument("--cmash_results", default="NONE", help="reuse an existing query-results CSV; skips the GPU stage")
    p.add_argument("--cutoff", type=float, default=0.01, help="containment cutoff at the largest k (default 0.01)")
    p.add_argument("--db", default="AUTO", help="where to write the subset FASTA (default temp_dir/cmashed_db.fna)")
    p.add_argument("--db_dir", default="AUTO", help="directory holding the organism files of the full database")
    p.add_argument("--dbinfo_in", default="AUTO", help="db_info file of the full database (default data/db_info.txt)")
    p.add_argument("--dbinfo_out", default="AUTO", help="where to write the subset db_info (default temp_dir/subset_db_info.txt)")
    p.add_argument("--input_type", default="AUTO", choices=["fastq", "fasta", "AUTO"], help="reads format (default: by extension)")
    p.add_argument("--keep_temp_files", action="store_true",
                   help="keep the intermediate files the reference keeps: the KMC databases of the reads (reads_60mers, "
                        "-ci2 -cs3) and of the intersection (60mers_intersection), and the intersection dump")
    p.add_argument("--strain_level", action="store_true", help="keep every strain above the cutoff (default: one per species)")
    p.add_argument("--temp_dir", default="AUTO/", help="directory for intermediate files")
    p.add_argument("--threads", type=int, default=4, help="accepted for compatibility (KMC threads in the reference)")
    # additions
    p.add_argument("--db_file", default="AUTO", help="native database file (default data/%s)" % DB_BASENAME)
    p.add_argument("--gate", default="exact", choices=["exact", "none"], help="smallest-k prefilter model (see DESIGN.md)")
    p.add_argument("--device", type=int, default=0, help="CUDA device")
    p.add_argument("--read_kmer_budget", type=int, default=0,
                   help="with --keep_temp_files: cap in bytes on the GPU table of read k-mers behind reads_60mers (0 = none); "
                        "past it that database is skipped and everything else is still written")
    p.add_argument("--read_kmer_passes", action="store_true",
                   help="with --keep_temp_files: count the k-mers behind reads_60mers in key-range passes over a GPU copy of "
                        "the reads, for read sets whose table would not fit in one GPU; --read_kmer_budget then caps that "
                        "copy plus one pass, and only reads that do not fit themselves skip the database")
    return p.parse_args(argv)


def read_dbinfo(args):
    """taxid -> [[accessions...], length, name lineage, taxid lineage]   (format: data/spec_db_info.txt;
    same structure as select_db.py:27-40 of the reference builds)"""
    table = {}
    with open(args.dbinfo_in, "r") as fh:
        next(fh, None)                                    # column titles
        for raw in fh:
            cols = raw.strip().split("\t")
            accession, taxid = cols[0], cols[2]
            entry = table.get(taxid)
            if entry is None:
                table[taxid] = [[accession], cols[1]] + cols[3:]
            else:
                entry[0].append(accession)
    return table


def taxid_of(organism_name: str) -> str:
    """'taxid_562_1_genomic.fna.gz' -> '562.1'  (naming from utils/ncbi2db.py:170, parsed back at select_db.py:88-89)"""
    return organism_name.split("taxid_")[1].split("_genomic.fna")[0].replace("_", ".")


def run_kmc_steps(args):
    """Replaces kmc + kmc_tools intersect + kmc_dump (select_db.py:43-65): counts the canonical 60-mers of the
    reads that belong to the database sketch; the live query is parked on args for run_cmash_and_cutoff."""
    from . import ingest
    from .api import Context, Database, pinned_array
    ctx = db = query = reader = None
    try:
        # pandas (the CSV tail) takes a good part of a second to import: do it while the GPU works
        import threading
        threading.Thread(target=lambda: __import__("pandas"), daemon=True).start()
        _tick("imports done")
        ctx = Context(args.device)
        _tick("CUDA context")
        # the native reader (its worker count = --threads, KMC's -t in the reference) is set up -- pinned buffers, file
        # mapped, parser threads started -- by a helper thread while this one reads the database file (both are C calls
        # that release the interpreter lock); it then cuts the first batches while the database is still loading, and
        # later fills one pinned buffer set while the previous batch is on its way to the GPU
        box = {}

        def open_reader():
            try:
                # 2 M reads per batch: two buffer sets of ~110 MB of page-locked memory (0.7 ms per MiB to pin: with 4 M reads
                # per batch the reader's set-up outlasted the database load it is meant to hide behind)
                box["reader"] = ingest.PackedBatches(args.reads, args.input_type, reads_per_batch=2_000_000, alloc=pinned_array,
                                                     threads=max(1, int(getattr(args, "threads", 4) or 4)))
            except BaseException as e:  # noqa: BLE001
                box["error"] = e
        th = threading.Thread(target=open_reader)
        th.start()
        try:
            db = Database.load(ctx, args.db_file)
        finally:
            th.join()
            reader = box.get("reader")
        if "error" in box:
            raise box["error"]
        _tick("database loaded, reader started")
        # -ci2 (select_db.py:50); the read k-mer table only for the reads_60mers database --keep_temp_files leaves behind
        query = db.query(ci_min=2, gate=args.gate, count_empty_in_den=True, read_kmers=bool(args.keep_temp_files),
                         read_kmer_budget=args.read_kmer_budget, read_kmer_passes=args.read_kmer_passes)
        for bases, nruns, off, n_reads in reader:
            query.push_packed_nruns(bases, nruns if len(nruns) else None, off, n_reads)
        query.sync()
        _tick("reads pushed and probed")
    except BaseException:
        # a corrupt reads file, a failed push: give the device and pinned memory back before the error travels on
        # (a caller looping over samples would otherwise accumulate them)
        for obj in (reader, query, db, ctx):
            if obj is not None:
                try:
                    obj.close()
                except Exception:  # noqa: BLE001
                    pass
        raise
    reader.close()
    _tick("reader closed")
    args._mlg = (ctx, db, query)


def run_cmash_and_cutoff(args, taxid2info):
    """Replaces the CMash subprocess (select_db.py:68-76), then applies the cutoff and the one-strain-per-species
    rule exactly as select_db.py:80-96 does, reading the CSV back in file order."""
    if args.cmash_results == "NONE":
        from . import cmash_tail, codec
        from ._lib import MLG_ERR_NOMEM, MlgError
        ctx, db, query = args._mlg
        cmash_out = args.temp_dir + "cmash_query_results.csv"
        res = query.finish_sparse()                       # rows for the genomes with a hit: all the CSV can hold
        _tick("containment table")
        cmash_tail.write_results_csv_sparse(cmash_out, db.names, db.ks, res["genomes"], res["ci"], 0.0)      # '-c 0'
        _tick("csv written")
        if args.keep_temp_files:
            # what kmc_dump and the FASTA rewrite leave in the temp dir (select_db.py:58-65): "<k-mer>\t<count>" lines
            # and the ">seq" records CMash is given
            query.dump_intersection(args.temp_dir + "60mers_intersection_dump", args.temp_dir + "60mers_intersection_dump.fa")
            # the two KMC databases of select_db.py:50-56
            query.write_intersection_kmc(args.temp_dir + "60mers_intersection", counter_max=3)
            try:
                query.write_reads_kmc(args.temp_dir + "reads_60mers", min_count=2, counter_max=3)
            except MlgError as e:
                if e.code != MLG_ERR_NOMEM:
                    raise
                sys.stderr.write("select_db: reads_60mers.kmc_* not written: %s\n" % e)
        if not getattr(args, "_mlg_leave_open", False):     # the command-line script exits right after: no point in freeing GBs first
            query.close(); db.close(); ctx.close()
        del args._mlg
        _tick("GPU objects closed")
    else:
        cmash_out = args.cmash_results

    chosen, seen_species = [], set()
    with open(cmash_out, "r") as fh:
        next(fh, None)                                    # ',k=30,k=40,k=50,k=60'
        for raw in fh:
            fields = raw.strip().split(",")
            organism, containment = fields[0], float(fields[-1])
            if not (containment >= args.cutoff):          # '>=' as at select_db.py:86
                continue
            if not args.strain_level:
                species = taxid2info[taxid_of(organism)][3].split("|")[-2]
                if species != "" and species in seen_species:
                    continue
                seen_species.add(species)
            chosen.append(organism)
    return chosen


def _inflate(path):
    with gzip.open(path, "rb") as src:
        return src.read()


def make_db_and_dbinfo(args, organisms_to_include, taxid2info):
    """Same outputs as select_db.py:99-117: the selected organism files inflated and concatenated in selection
    order, and the subset db_info with its two fixed header lines.  The reference starts one `zcat` per genome, one
    after the other (select_db.py:103-105); here a few threads inflate ahead (zlib releases the GIL) while the
    main thread writes the results in order -- same bytes out."""
    from concurrent.futures import ThreadPoolExecutor
    workers = max(1, min(16, int(getattr(args, "threads", 4) or 4)))
    window = 4 * workers                                   # bounded look-ahead: genomes are MBs each
    with open(args.db, "wb") as out, ThreadPoolExecutor(max_workers=workers) as pool:
        pending = []
        it = iter(organisms_to_include)
        for organism in it:
            pending.append(pool.submit(_inflate, args.db_dir + organism))
            if len(pending) >= window:
                out.write(pending.pop(0).result())
        for fut in pending:
            out.write(fut.result())
    with open(args.dbinfo_out, "w") as out:
        out.writelines(HEADER_LINES)
        for organism in organisms_to_include:
            taxid = taxid_of(organism)
            accessions, length, names, taxids = taxid2info[taxid][0], taxid2info[taxid][1], taxid2info[taxid][2], taxid2info[taxid][3]
            for acc in accessions:
                out.write("\t".join((acc, length, taxid, names, taxids)) + "\n")


def _normalise(args):
    """AUTO / NONE resolution, same outcomes as select_db.py:126-153"""
    for name, default in (("db_file", "AUTO"), ("gate", "exact"), ("device", 0), ("read_kmer_budget", 0),
                          ("read_kmer_passes", False)):
        if not hasattr(args, name):
            setattr(args, name, default)       # Namespace handed over by the reference's metalign.py
    if not args.data.endswith("/"):
        args.data += "/"
    if args.db_dir == "AUTO":
        args.db_dir = args.data + "organism_files/"
    if not args.db_dir.endswith("/"):
        args.db_dir += "/"
    if args.temp_dir == "AUTO/":
        args.temp_dir = tempfile.mkdtemp(prefix=args.data)
    if not args.temp_dir.endswith("/"):
        args.temp_dir += "/"
    os.makedirs(args.temp_dir, exist_ok=True)
    if args.dbinfo_in == "AUTO":
        args.dbinfo_in = args.data + "db_info.txt"
    if args.dbinfo_out == "AUTO":
        args.dbinfo_out = args.temp_dir + "subset_db_info.txt"
    if args.db == "AUTO":
        args.db = args.temp_dir + "cmashed_db.fna"
    if args.db_file == "AUTO":
        args.db_file = args.data + DB_BASENAME
    if args.input_type == "AUTO":
        from .ingest import detect_input_type
        args.input_type = detect_input_type(args.reads)


def select_main(args=None):
    if args is None:
        args = select_parseargs()
    elif args.cutoff < 0.0 or args.cutoff > 1.0:
        print("Error: args.cutoff must be between 0 and 1, inclusive.")
        sys.exit()
    _normalise(args)
    _tick("start")
    if args.cmash_results == "NONE":
        # db_info.txt has a line per accession of the full database: parsed beside the GPU stage, needed after it
        import threading
        box = {}

        def load_info():
            try:
                box["info"] = read_dbinfo(args)
            except BaseException as e:  # noqa: BLE001
                box["error"] = e
        th = threading.Thread(target=load_info)
        th.start()
        try:
            run_kmc_steps(args)
        finally:
            th.join()
        if "error" in box:
            raise box["error"]
        taxid2info = box["info"]
    else:
        taxid2info = read_dbinfo(args)
    _tick("db_info read")
    organisms_to_include = run_cmash_and_cutoff(args, taxid2info)
    _tick("selection done")
    make_db_and_dbinfo(args, organisms_to_include, taxid2info)
    _tick("subset files written")
    return organisms_to_include


if __name__ == "__main__":
    select_main(select_parseargs())
