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

Under torchrun (WORLD_SIZE > 1) every rank drives the GPU of its LOCAL_RANK: it reads its own byte range of the reads
file (ingest.share_ranges), the ranks sum their counters in one exchange (dist.reduce_query, each rank's counters clamped
to counter_max so that the intersection counts are those of one GPU), and rank 0 alone writes the files -- the same bytes
as a single-process run.  --threads is then per rank.

A single process, the ranks of a torchrun launch and the samples of a batch (select_many) share one pipeline, whose pieces
are told their rank and world: open_database + open_reader, push_sample, exchange (world > 1), write_gpu_files,
run_cmash_and_cutoff.
"""
from __future__ import annotations

import argparse
import collections
import copy
import gzip
import os
import re
import sys
import tempfile

DB_BASENAME = "cmash_db_n1000_k60.mlgdb"
HEADER_LINES = ("Accesion\tLength\tTaxID\tLineage\tTaxID_Lineage\n",          # sic: spelling of the reference, select_db.py:109
                "Unmapped\t0\tUnmapped\t|||||||Unmapped\t|||||||Unmapped\n")
# the files a run writes (output_paths); the CSV and the subset files always, the others with --keep_temp_files
OUTPUT_NAMES = ("cmash_query_results.csv", "cmashed_db.fna", "subset_db_info.txt", "60mers_intersection_dump",
                "60mers_intersection_dump.fa", "60mers_intersection.kmc_pre", "60mers_intersection.kmc_suf",
                "reads_60mers.kmc_pre", "reads_60mers.kmc_suf")


_T0 = None


def _now():
    import time
    return time.perf_counter()


def _tick(label):
    """MLG_TIMING=1: stage times on stderr (seconds since the module was imported)"""
    if os.environ.get("MLG_TIMING"):
        import time
        global _T0
        now = time.perf_counter()
        if _T0 is None:
            _T0 = now
        sys.stderr.write("[mlg %7.3f s] %s\n" % (now - _T0, label))


def ranks():
    """(rank, world) of a torchrun launch with the process group up, else (0, 1)"""
    if "torch" not in sys.modules:          # a single process need not pay for importing torch
        return 0, 1
    import torch.distributed as tdist
    if tdist.is_available() and tdist.is_initialized():
        return tdist.get_rank(), tdist.get_world_size()
    return 0, 1


def init_ranks(args):
    """under torchrun (WORLD_SIZE > 1): the NCCL process group, --device = LOCAL_RANK, this process bound to the cores of
    its GPU's NUMA node (before any reader thread starts).  Nothing for a single process."""
    if int(os.environ.get("WORLD_SIZE", "1")) <= 1:
        return
    from . import dist as mdist
    _rank, _world, local = mdist.init_from_env("nccl")
    args.device = local
    mdist.bind_to_gpu_numa(local)


def shared_mkdtemp(prefix, rank=0, world=1):
    """tempfile.mkdtemp on rank 0, the same path on every rank"""
    if world == 1:
        return tempfile.mkdtemp(prefix=prefix)
    import torch.distributed as tdist
    box = [tempfile.mkdtemp(prefix=prefix) if rank == 0 else None]
    tdist.broadcast_object_list(box, src=0)
    return box[0]


def _on_rank0(fn, rank, world):
    """fn() on rank 0 alone; its result, or its failure, reaches every rank"""
    if world == 1:
        return fn()
    import torch.distributed as tdist
    box = [None, None]
    if rank == 0:
        try:
            box[0] = fn()
        except Exception as e:  # noqa: BLE001  (the other ranks wait in the broadcast)
            box[1] = e
    tdist.broadcast_object_list(box, src=0)
    if box[1] is not None:
        raise box[1] if rank == 0 else RuntimeError("select_db: rank 0 failed: %s" % box[1])
    return box[0]


def _all_ok(err, device, world):
    """raise if this rank has an error (err) or, collectively when world > 1, any other rank has: this rank's own error
    where it has one"""
    ok = err is None
    if world > 1:
        from . import dist as mdist
        ok = mdist.all_ok(ok, device)
    if not ok:
        raise err if err is not None else RuntimeError("select_db: another rank failed")


def _add_common_flags(p):
    """the flags of select_db.py that are not tied to one reads file, which select_many.py takes as well"""
    p.add_argument("--cutoff", type=float, default=0.01, help="containment cutoff at the largest k (default 0.01)")
    p.add_argument("--db_dir", default="AUTO", help="directory holding the organism files of the full database")
    p.add_argument("--dbinfo_in", default="AUTO", help="db_info file of the full database (default data/db_info.txt)")
    p.add_argument("--keep_temp_files", action="store_true",
                   help="keep the intermediate files the reference keeps: the KMC databases of the reads (reads_60mers, "
                        "-ci2 -cs3) and of the intersection (60mers_intersection), and the intersection dump")
    p.add_argument("--strain_level", action="store_true", help="keep every strain above the cutoff (default: one per species)")
    p.add_argument("--threads", type=int, default=4, help="reader threads (per rank under torchrun; KMC threads in the reference)")
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


def select_parseargs(argv=None):
    p = argparse.ArgumentParser(description="Score every database genome against the reads (containment min-hash, "
                                            "k=30..60) and write the reduced database to align to.")
    p.add_argument("reads", help="reads file (FASTA/FASTQ, optionally .gz)")
    p.add_argument("data", help="data/ directory (database, db_info.txt, organism_files/)")
    p.add_argument("--cmash_results", default="NONE", help="reuse an existing query-results CSV; skips the GPU stage")
    p.add_argument("--db", default="AUTO", help="where to write the subset FASTA (default temp_dir/cmashed_db.fna)")
    p.add_argument("--dbinfo_out", default="AUTO", help="where to write the subset db_info (default temp_dir/subset_db_info.txt)")
    p.add_argument("--input_type", default="AUTO", choices=["fastq", "fasta", "AUTO"], help="reads format (default: by extension)")
    p.add_argument("--temp_dir", default="AUTO/", help="directory for intermediate files")
    _add_common_flags(p)
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


def output_paths(args):
    """the paths of the files a run writes (OUTPUT_NAMES): in args.temp_dir, the subset files where --db and --dbinfo_out
    put them"""
    placed = {"cmashed_db.fna": args.db, "subset_db_info.txt": args.dbinfo_out}
    return [placed.get(name, args.temp_dir + name) for name in OUTPUT_NAMES]


def _remove(paths):
    for path in paths:
        try:
            os.remove(path)
        except OSError:
            pass


def open_reader(args, rank=0, world=1, alloc=None):
    """The native reader of args.reads (its worker count = --threads, KMC's -t in the reference): buffers allocated (pinned
    by default), file mapped, parser threads started -- they cut the first batches at once, and later fill one buffer set
    while the previous batch is on its way to the GPU.  With world > 1 (one reads file split over the ranks, which then
    exchange their counters) only rank's byte range of the file; else the whole file."""
    from . import ingest
    from .api import pinned_array
    # 2 M reads per batch: two buffer sets of ~110 MB of page-locked memory (0.7 ms per MiB to pin: with 4 M reads per batch
    # the reader's set-up outlasted the database load it is meant to hide behind)
    share = ingest.share_ranges(args.reads, world)[rank] if world > 1 else None
    return ingest.PackedBatches(args.reads, args.input_type, reads_per_batch=2_000_000, alloc=alloc or pinned_array,
                                threads=max(1, int(getattr(args, "threads", 4) or 4)), share=share)


def _on_helper(fn):
    """fn() started on a helper thread; the returned join() waits for it and gives (its result, its error)"""
    import threading
    box = {}

    def run():
        try:
            box["value"] = fn()
        except BaseException as e:  # noqa: BLE001
            box["error"] = e
    th = threading.Thread(target=run, daemon=True)
    th.start()

    def join():
        th.join()
        return box.get("value"), box.get("error")
    return join


def _close_all(*objs):
    for obj in objs:
        if obj is not None:
            try:
                obj.close()
            except Exception:  # noqa: BLE001
                pass


def _close_gpu(world, query, db, ctx):
    """the query and the database, the exchanges of dist (world > 1), then the context they live in"""
    _close_all(query, db)
    if world > 1:
        from . import dist as mdist
        mdist.close_exchanges()
    _close_all(ctx)


def open_database(args, beside=None):
    """The part of a run that does not depend on the sample: the context of args.device and the database args.db_file.
    beside() (e.g. opening the reader) runs on a helper thread while this one reads the database file (both are C calls
    that release the interpreter lock).  Returns (ctx, db, what beside() returned); if anything fails, what was opened is
    closed again."""
    from .api import Context, Database
    ctx = db = side = None
    try:
        ctx = Context(args.device)
        _tick("CUDA context")
        join = _on_helper(beside) if beside is not None else (lambda: (None, None))
        try:
            db = Database.load(ctx, args.db_file)
        finally:
            side, side_err = join()
        if side_err is not None:
            raise side_err
        return ctx, db, side
    except BaseException:
        _close_all(side, db, ctx)
        raise


def push_sample(args, db, reader, world=1):
    """The per-sample GPU part up to the counters: a query on db, every batch of the reader pushed and probed.  -ci2
    (select_db.py:50); the read k-mer table only for the reads_60mers database --keep_temp_files leaves behind.  With
    world > 1 (a reader of one rank's byte range, open_reader) the read k-mers are counted in passes, because
    share_read_kmers hands the reads around; else only with --read_kmer_passes.  The query is closed again if a push
    fails."""
    query = db.query(ci_min=2, gate=args.gate, count_empty_in_den=True, read_kmers=bool(args.keep_temp_files),
                     read_kmer_budget=args.read_kmer_budget, read_kmer_passes=args.read_kmer_passes or world > 1)
    try:
        for bases, nruns, off, n_reads in reader:
            query.push_packed_nruns(bases, nruns if len(nruns) else None, off, n_reads)
        query.sync()
    except BaseException:
        query.close()
        raise
    return query


def exchange(args, query, share_info, err, world):
    """Collective, world > 1, after every rank's pushes (err: this rank's failure so far, or None): every rank learns
    whether every other rank got this far, and checks the FASTQ phases of all shares (share_info: this rank's reader's);
    then the ranks hand their reads around for reads_60mers (--keep_temp_files) and sum their counters."""
    import torch.distributed as tdist
    from . import dist as mdist
    from . import ingest
    _all_ok(err, args.device, world)
    infos = [None] * world
    tdist.all_gather_object(infos, share_info)
    ingest.check_share_phases(infos, args.input_type)
    if args.keep_temp_files:
        mdist.share_read_kmers(query, args.device)
    mdist.reduce_query(query, args.device, clamp=3)          # -cs3: the intersection counts of one GPU
    query.sync()


def write_gpu_files(args, db, query, rank, world, stages):
    """The per-sample GPU part after the pushes (and the exchange): the containment table as
    args.temp_dir/cmash_query_results.csv (what the CMash subprocess writes, select_db.py:68-76) and, with
    --keep_temp_files, the intersection dump and the two KMC databases.  Every rank finishes its query (identical on every
    rank after the exchange); rank 0 writes the CSV and the intersection files; with world > 1 a failure on any rank
    raises on every rank, and the ranks join reads_60mers (dist.write_reads_kmc).  On one GPU a read k-mer table over
    --read_kmer_budget only skips reads_60mers, with a warning."""
    from . import cmash_tail
    err = None
    try:
        t0 = _now()
        res = query.finish_sparse()                   # rows for the genomes with a hit: all the CSV can hold
        stages["finish_s"] = _now() - t0
        _tick("containment table")
        if rank == 0:
            cmash_tail.write_results_csv_sparse(args.temp_dir + "cmash_query_results.csv", db.names, db.ks, res["genomes"],
                                                res["ci"], 0.0)          # '-c 0'
            _tick("csv written")
            if args.keep_temp_files:
                # what kmc_dump and the FASTA rewrite leave in the temp dir (select_db.py:58-65): "<k-mer>\t<count>" lines
                # and the ">seq" records CMash is given; then the intersection database of select_db.py:53-56
                query.dump_intersection(args.temp_dir + "60mers_intersection_dump",
                                        args.temp_dir + "60mers_intersection_dump.fa")
                query.write_intersection_kmc(args.temp_dir + "60mers_intersection", counter_max=3)
    except Exception as e:  # noqa: BLE001  (with world > 1 every rank has to take part in the check below)
        err = e
    _all_ok(err, args.device, world)
    if not args.keep_temp_files:
        return
    # the reads database of select_db.py:50-52
    prefix = args.temp_dir + "reads_60mers"
    if world > 1:
        from . import dist as mdist
        mdist.write_reads_kmc(query, prefix, 2, 3, args.device)
        return
    from ._lib import MLG_ERR_NOMEM, MlgError
    try:
        query.write_reads_kmc(prefix, min_count=2, counter_max=3)
    except MlgError as e:
        if e.code != MLG_ERR_NOMEM:
            raise
        sys.stderr.write("select_db: reads_60mers.kmc_* not written: %s\n" % e)


def run_kmc_steps(args, rank, world, stages):
    """Replaces kmc + kmc_tools intersect + kmc_dump (select_db.py:43-65): counts the canonical 60-mers of the
    reads that belong to the database sketch.  Returns (ctx, db, query) after the pushes and, with world > 1, the
    exchange; if anything fails, on any rank, what was opened is closed before the error travels on."""
    t0 = _now()
    ctx = db = query = reader = share_info = err = None
    try:
        # pandas (the CSV tail) takes a good part of a second to import: do it while the GPU works
        import threading
        threading.Thread(target=lambda: __import__("pandas"), daemon=True).start()
        _tick("imports done")
        # the reader is set up while the database loads, and cuts the first batches before the load ends
        ctx, db, reader = open_database(args, beside=lambda: open_reader(args, rank, world))
        _tick("database loaded, reader started")
        stages["open_s"] = _now() - t0
        t0 = _now()
        query = push_sample(args, db, reader, world)
        stages["push_s"] = _now() - t0
        _tick("reads pushed and probed")
        if world > 1:
            share_info = reader.share_info()
    except BaseException as e:  # noqa: BLE001  (with world > 1 every rank has to reach the exchange's check)
        err = e
    try:
        if world > 1:
            t0 = _now()
            exchange(args, query, share_info, err, world)
            stages["exchange_s"] = _now() - t0
            _tick("exchange done")
        elif err is not None:
            raise err
    except BaseException:
        # a corrupt reads file, a failed push: give the device and pinned memory back before the error travels on
        _close_all(reader)
        _close_gpu(world, query, db, ctx)
        raise
    reader.close()
    _tick("reader closed")
    return ctx, db, query


def run_cmash_and_cutoff(args, taxid2info, cmash_out):
    """The cutoff and the one-strain-per-species rule of select_db.py:80-96 on the query-results CSV (written by
    write_gpu_files in place of the CMash subprocess of select_db.py:68-76), then the subset files; returns the selection"""
    chosen = _select(args, taxid2info, cmash_out)
    _tick("selection done")
    make_db_and_dbinfo(args, chosen, taxid2info)
    _tick("subset files written")
    return chosen


def _select(args, taxid2info, cmash_out):
    """the cutoff and the one-strain-per-species rule of select_db.py:80-96 on the CSV"""
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


def resolve_data(args):
    """AUTO resolution of the full database's paths, same outcomes as select_db.py:126-153: data/ with its slash, db_dir
    (data/organism_files/), dbinfo_in (data/db_info.txt) and the native database file"""
    if not args.data.endswith("/"):
        args.data += "/"
    for name, value in (("db_dir", "organism_files/"), ("dbinfo_in", "db_info.txt"), ("db_file", DB_BASENAME)):
        if getattr(args, name) == "AUTO":
            setattr(args, name, args.data + value)
    if not args.db_dir.endswith("/"):
        args.db_dir += "/"


def _normalise(args, rank, world):
    """AUTO / NONE resolution, same outcomes as select_db.py:126-153"""
    for name, default in (("db_file", "AUTO"), ("gate", "exact"), ("device", 0), ("read_kmer_budget", 0),
                          ("read_kmer_passes", False)):
        if not hasattr(args, name):
            setattr(args, name, default)       # Namespace handed over by the reference's metalign.py
    resolve_data(args)
    if args.temp_dir == "AUTO/":
        args.temp_dir = shared_mkdtemp(args.data, rank, world)
    if not args.temp_dir.endswith("/"):
        args.temp_dir += "/"
    os.makedirs(args.temp_dir, exist_ok=True)
    if args.dbinfo_out == "AUTO":
        args.dbinfo_out = args.temp_dir + "subset_db_info.txt"
    if args.db == "AUTO":
        args.db = args.temp_dir + "cmashed_db.fna"
    if args.input_type == "AUTO":
        from .ingest import detect_input_type
        args.input_type = detect_input_type(args.reads)


def select_main(args=None, *, stages=None, leave_open=False):
    """select_db.py; returns the selection.  stages: a dict the run fills with its GPU stages' seconds (open_s, push_s,
    exchange_s, finish_s).  leave_open: a single process that succeeds does not free its context, database and query, for
    a caller that exits right after; a failed run frees them.  Under torchrun a failure on any rank raises on every rank
    and rank 0 removes the run's files (output_paths); a single process leaves what it wrote, as the reference does."""
    if args is None:
        args = select_parseargs()
    elif args.cutoff < 0.0 or args.cutoff > 1.0:
        print("Error: args.cutoff must be between 0 and 1, inclusive.")
        sys.exit()
    init_ranks(args)
    rank, world = ranks()
    _normalise(args, rank, world)
    _tick("start")
    if args.cmash_results != "NONE":
        taxid2info = read_dbinfo(args)
        _tick("db_info read")
        return _on_rank0(lambda: run_cmash_and_cutoff(args, taxid2info, args.cmash_results), rank, world)
    stages = {} if stages is None else stages
    # db_info.txt has a line per accession of the full database: parsed beside the GPU stage, needed after it
    join_info = _on_helper(lambda: read_dbinfo(args))
    try:
        ctx, db, query = run_kmc_steps(args, rank, world, stages)
    finally:
        taxid2info, info_err = join_info()
    try:
        _all_ok(info_err, args.device, world)
        _tick("db_info read")
        write_gpu_files(args, db, query, rank, world, stages)
        if world == 1 and not leave_open:
            _close_gpu(world, query, db, ctx)
            _tick("GPU objects closed")
        cmash_out = args.temp_dir + "cmash_query_results.csv"
        chosen = _on_rank0(lambda: run_cmash_and_cutoff(args, taxid2info, cmash_out), rank, world)
    except BaseException:
        if world > 1 and rank == 0:
            _remove(output_paths(args))
        _close_gpu(world, query, db, ctx)
        raise
    if world > 1:
        _close_gpu(world, query, db, ctx)
    return chosen


# ------------------------------------------------------------------ many samples against one database
SUMMARY_NAME = "samples_summary.tsv"
SUMMARY_HEADER = "sample_id\tstatus\tselected\tseconds\terror\n"
_SAFE_ID = re.compile(r"[A-Za-z0-9][A-Za-z0-9._-]{0,127}\Z")

Sample = collections.namedtuple("Sample", "id reads input_type")
# status "ok" or "failed"; organisms: the selection (None when failed); stages: seconds per stage of this sample
SampleResult = collections.namedtuple("SampleResult", "id status organisms seconds error out_dir stages")


class SampleSheetError(ValueError):
    pass


def read_sample_sheet(path):
    """The samples of a sheet: one line per sample, `sample_id <TAB> reads_path [<TAB> fastq|fasta]` (blank lines and lines
    starting with '#' are skipped).  Without the third column the type comes from the extension (ingest.input_type_of); a
    relative reads path is taken from the sheet's directory.  Raises SampleSheetError naming the line for a wrong number of
    columns, an id that is not a safe directory name, a duplicate id or an unknown type.  Whether the reads files exist is
    not checked here: a missing one fails its own sample."""
    from .ingest import input_type_of
    base = os.path.dirname(os.path.abspath(path))
    samples, first_line = [], {}
    with open(path, "r") as fh:
        for no, raw in enumerate(fh, 1):
            line = raw.rstrip("\r\n")
            if not line.strip() or line.startswith("#"):
                continue
            where = "%s, line %d" % (path, no)
            cols = line.split("\t")
            if len(cols) not in (2, 3) or not cols[1]:
                raise SampleSheetError("%s: expected sample_id<TAB>reads_path[<TAB>fastq|fasta], got %d tab-separated "
                                       "column(s)" % (where, len(cols)))
            sid, reads = cols[0], cols[1]
            if not _SAFE_ID.match(sid) or sid == SUMMARY_NAME:
                raise SampleSheetError("%s: sample id %r is not a safe directory name (letters, digits, '.', '_', '-'; not "
                                       "starting with '.' or '-'; at most 128 characters)" % (where, sid))
            if sid in first_line:
                raise SampleSheetError("%s: duplicate sample id %r (first on line %d)" % (where, sid, first_line[sid]))
            kind = cols[2] if len(cols) == 3 else input_type_of(reads)
            if kind not in ("fastq", "fasta"):
                raise SampleSheetError("%s: unknown reads type %r (fastq or fasta)" % (where, cols[2]) if len(cols) == 3 else
                                       "%s: the type of %r does not follow from its extension: add fastq or fasta as a third "
                                       "column" % (where, reads))
            first_line[sid] = no
            samples.append(Sample(sid, reads if os.path.isabs(reads) else os.path.join(base, reads), kind))
    return samples


def rank_samples(n_samples, rank, world):
    """the indices of the samples rank `rank` of `world` runs: i mod world == rank"""
    return list(range(rank, n_samples, world))


def format_summary(results):
    """samples_summary.tsv: a header, then one line per sample -- id, ok / failed, organisms selected, seconds, error"""
    lines = [SUMMARY_HEADER]
    for r in results:
        err = " ".join(str(r.error or "").split())            # one line, no tabs
        lines.append("%s\t%s\t%d\t%.3f\t%s\n" % (r.id, r.status, len(r.organisms or ()), r.seconds, err))
    return "".join(lines)


def _is_device_error(e):
    from ._lib import MlgError
    return isinstance(e, MlgError) and e.code == -1           # MLG_ERR_CUDA: the device state is unknown


class _NotRun(Exception):
    pass


class SelectSession:
    """One CUDA context, one loaded database, the parsed db_info and one pool of pinned reader buffers, kept for any
    number of samples.  `run(samples, out_dir)` writes each sample's select_db.py files into out_dir/<sample_id>/.

    Two threads: a GPU thread runs the per-sample GPU part (open the reader, push, finish, CSV, intersection and KMC files,
    close the query and reader) sample after sample on the context's streams, and the calling thread applies the cutoff
    and writes the subset FASTA and db_info (make_db_and_dbinfo).  So while sample i's subset files are written, sample
    i + 1's reads are already read and probed; the GPU thread runs at most one sample ahead.  The next sample's reader is
    opened while the current one finishes, in the buffers the closed reader gave back (ingest.BufferPool): pinned memory
    stays at one reader's buffer sets.  Every sample is read whole and queried alone (rank 0 of a world of 1), also
    under torchrun.

    A failing sample (an unreadable, truncated or corrupt reads file, a failed write, any library error but a device
    error) fails alone: its query and reader are closed, its files and directory removed, and the batch goes on.  A
    device error (MLG_ERR_CUDA) ends the batch: the samples not yet run are reported as failed and no later run() starts
    any."""

    def __init__(self, args):
        """args: the flags of select_many (data and db_file resolved as resolve_data resolves them)"""
        from . import ingest
        from .api import pinned_array
        t0 = _now()
        self.args = args
        self.pool = ingest.BufferPool(pinned_array)
        self.stopped = None          # the message of the device error that ended the batch
        self.ctx, self.db, self.taxid2info = open_database(args, beside=lambda: read_dbinfo(args))
        self.open_s = _now() - t0

    def close(self):
        _close_all(self.db, self.ctx)
        self.db = self.ctx = None
        self.pool.clear()

    def _sample_args(self, s, out_dir):
        a = copy.copy(self.args)
        a.reads, a.input_type, a.cmash_results = s.reads, s.input_type, "NONE"
        a.temp_dir = os.path.join(out_dir, s.id) + "/"
        a.db, a.dbinfo_out = a.temp_dir + "cmashed_db.fna", a.temp_dir + "subset_db_info.txt"
        return a

    def _gpu_part(self, a, reader_join, open_next, stages):
        """one sample's GPU part; open_next() is called once this sample's reader is closed"""
        query = reader = None
        t0 = _now()
        try:
            reader, err = reader_join()
            if err is not None:
                raise err
            os.makedirs(a.temp_dir, exist_ok=True)
            query = push_sample(a, self.db, reader)
            reader.close()
            reader = None
            open_next()                              # its parser threads cut the first batches while this sample finishes
            stages["push_s"] = _now() - t0
            t0 = _now()
            write_gpu_files(a, self.db, query, 0, 1, {})
            stages["gpu_files_s"] = _now() - t0
        finally:
            _close_all(reader, query)

    def run(self, samples, out_dir):
        """-> [SampleResult] in the order of `samples`"""
        import queue
        import threading
        sargs = [self._sample_args(s, out_dir) for s in samples]
        handoff = queue.Queue()
        ahead = threading.Semaphore(2)               # the sample whose subset files are being written + one GPU part ahead

        def reader_of(i):
            if i >= len(samples) or self.stopped is not None:
                return lambda: (None, None)
            return _on_helper(lambda: open_reader(sargs[i], alloc=self.pool))

        def gpu_thread():
            # every sample is handed over, with its error if anything failed: the calling thread waits for each one
            join = None
            for i, a in enumerate(sargs):
                nxt, stages, err = [], {}, None
                try:
                    ahead.acquire()
                    if join is None:
                        join = reader_of(i)

                    def open_next():
                        nxt.append(reader_of(i + 1))
                    if self.stopped is not None:
                        _close_all(join()[0])
                        err = _NotRun("not run: " + self.stopped)
                    else:
                        self._gpu_part(a, join, open_next, stages)
                except BaseException as e:  # noqa: BLE001
                    err = err or e
                    if _is_device_error(e):
                        self.stopped = "the batch stopped after a device error on sample %s: %s" % (samples[i].id, e)
                join = nxt[0] if nxt else None       # None: the next sample opens its reader itself
                handoff.put((i, stages, err))

        th = threading.Thread(target=gpu_thread, daemon=True)
        th.start()
        results = []
        for _ in samples:
            i, stages, err = handoff.get()
            a = sargs[i]
            chosen = None
            if err is None:
                t0 = _now()
                try:
                    chosen = run_cmash_and_cutoff(a, self.taxid2info, a.temp_dir + "cmash_query_results.csv")
                except Exception as e:  # noqa: BLE001
                    err = e
                stages["subset_s"] = _now() - t0
            ahead.release()
            seconds = sum(stages.values())
            if err is not None:
                _remove(output_paths(a))
                try:
                    os.rmdir(a.temp_dir)
                except OSError:
                    pass                             # not empty: files that are not this run's stay
                msg = str(err) if isinstance(err, _NotRun) else "%s: %s" % (type(err).__name__, err)
                results.append(SampleResult(samples[i].id, "failed", None, seconds, msg, a.temp_dir, stages))
            else:
                results.append(SampleResult(samples[i].id, "ok", chosen, seconds, "", a.temp_dir, stages))
        th.join()
        return results


def select_many_parseargs(argv=None):
    p = argparse.ArgumentParser(description="select_db.py for many samples against one database: one CUDA context and one "
                                            "loaded database per GPU, each sample's files in out_dir/<sample_id>/.")
    p.add_argument("sample_sheet", help="one line per sample: sample_id<TAB>reads_path[<TAB>fastq|fasta]")
    p.add_argument("data", help="data/ directory (database, db_info.txt, organism_files/)")
    p.add_argument("--out_dir", default="AUTO", help="where the sample directories and %s go (default: a new temporary "
                                                     "directory under data/)" % SUMMARY_NAME)
    _add_common_flags(p)
    return p.parse_args(argv)


def normalise_many(args, rank=0, world=1):
    """the AUTO defaults of select_many's flags, as _normalise resolves them for select_db; out_dir created"""
    resolve_data(args)
    if args.out_dir == "AUTO":
        args.out_dir = shared_mkdtemp(args.data, rank, world)
    os.makedirs(args.out_dir, exist_ok=True)


def select_many(sample_sheet, args, stages=None):
    """select_db.py for every sample of a sample sheet (read_sample_sheet) against one database: each sample's files in
    args.out_dir/<sample_id>/ -- byte for byte what `select_db.py <reads> <data> --temp_dir out_dir/<sample_id>/` with the
    same flags writes -- and out_dir/samples_summary.tsv (format_summary).  Returns a SampleResult per sample in sheet
    order; a caller can map and profile each ok sample from its out_dir.  stages: a dict this rank fills with the seconds
    it took to open the context and the database (open_s).

    The sheet is checked before any GPU work.  Under torchrun (WORLD_SIZE > 1) rank r runs the samples i with
    i mod world == r on its LOCAL_RANK GPU (its own context and database, no exchange); every rank gets every result, and
    rank 0 writes the summary."""
    if args.cutoff < 0.0 or args.cutoff > 1.0:
        raise ValueError("cutoff must be between 0 and 1, inclusive")
    samples = read_sample_sheet(sample_sheet)
    init_ranks(args)
    rank, world = ranks()
    normalise_many(args, rank, world)
    mine = [samples[i] for i in rank_samples(len(samples), rank, world)]
    session = None
    try:
        session = SelectSession(args)
        if stages is not None:
            stages["open_s"] = session.open_s
        results = session.run(mine, args.out_dir)
    except Exception as e:  # noqa: BLE001  (no context or database: none of this rank's samples runs)
        msg = "not run: the database could not be opened on this GPU: %s: %s" % (type(e).__name__, e)
        results = [SampleResult(s.id, "failed", None, 0.0, msg, os.path.join(args.out_dir, s.id) + "/", {}) for s in mine]
    finally:
        if session is not None:
            session.close()
    if world > 1:
        from . import dist as mdist
        order = {s.id: i for i, s in enumerate(samples)}
        results = sorted(mdist.all_gather_rows(results), key=lambda r: order[r.id])
    if rank == 0:
        with open(os.path.join(args.out_dir, SUMMARY_NAME), "w") as f:
            f.write(format_summary(results))
    return results


if __name__ == "__main__":
    select_main(select_parseargs())
