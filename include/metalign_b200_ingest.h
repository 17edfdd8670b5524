/* metalign_b200_ingest -- host-side read ingest for the database-selection path.
 *
 * In the reference this job belongs to KMC: `kmc -k60 -fq|-fa ... <reads>` (scripts/select_db.py:46-52) opens the
 * reads file (FASTQ or single-line FASTA, optionally gzip) and extracts the sequences itself.  Here a small
 * multi-threaded reader turns the file into the packed batches mlg_query_push_packed_nruns() takes:
 *   - 2-bit packed bases, reads back to back at base granularity (A=0 C=1 G=2 T=3, lower case folded);
 *   - every other symbol is an N: packed as A and listed as a (start, length) run in batch base coordinates;
 *   - read offsets in bases.
 * Record rules (same as KMC's -fq / -fa):
 *   fastq  4-line records, the sequence is line 2 of each record
 *   fasta  every non-empty line that does not start with '>' or ';' is one record
 * A trailing '\r' is stripped; a file need not end with a newline.
 *
 * Pipeline: a plain file is mapped and `threads` threads find the sequence lines (two passes: count the newlines of every
 * part, then cut); a gzip file is inflated by one thread (an in-house DEFLATE decoder with CRC check; MLGI_ZLIB=1 = zlib), a BGZF one (bgzip: independent members) by `threads`
 * threads at a time; `threads` workers then pack a batch in parallel into the caller's (pinned) buffers, 32 bases at a time
 * with AVX2 where the CPU has it.  No CUDA dependency: this library only fills host memory.  The file must not be
 * truncated while it is being read (it is mapped).
 */
#ifndef METALIGN_B200_INGEST_H
#define METALIGN_B200_INGEST_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLGI_FASTQ 0
#define MLGI_FASTA 1

typedef struct mlgi_reader mlgi_reader;

const char* mlgi_last_error(void);
/* threads <= 0: all hardware threads */
int mlgi_open(const char* path, int input_type, int threads, mlgi_reader** out);
/* Next batch: at most max_reads reads and max_bases bases (a single read longer than max_bases is an error).
 *   bases      cap_bases_bytes >= max_bases / 4 + 32; the used part (rounded up to 16 bytes) is written in full
 *   nruns      cap_runs (start, length) pairs of uint32; max_bases must be < 2^32
 *   off        max_reads + 1 entries
 * Returns 1 with *n_reads > 0, 0 at end of input (nothing written), < 0 on error; 2 = like 1, but the batch has more
 * than cap_runs N runs: *n_runs says how many, nruns was not written, and mlgi_spilled_runs() hands them over. */
int mlgi_next(mlgi_reader* r, uint8_t* bases, uint64_t cap_bases_bytes, uint32_t* nruns, uint64_t cap_runs, uint64_t* off,
              uint64_t max_reads, uint64_t max_bases, uint64_t* n_reads, uint64_t* n_runs);
int mlgi_spilled_runs(mlgi_reader* r, uint32_t* nruns, uint64_t cap_runs);
/* A share of a reads file for one of several readers (one per GPU): like mlgi_open, but only the records of the byte range
 * [begin, end) of the file on disk.  A line belongs to the share that holds its first byte and is read to its end.
 *   plain file   the range is a range of the file's bytes
 *   BGZF         the share takes the members whose compressed start is in the range, and the lines that start in their
 *                text (inflating the following members as far as its last line runs)
 *   other gzip   one DEFLATE stream cannot be split: the share with begin = 0 reads the whole file (and says so on stderr
 *                when end is before the end of the file), every other share is empty
 * FASTA shares start at the first line start in the range.  A FASTQ share also needs the line number mod 4 of its first
 * line: it takes the first line that starts with '@' and whose line two after starts with '+' (exact for 4-line FASTQ).
 * Shares of consecutive ranges that cover the file deliver, joined in order, the reads of mlgi_open -- if every share's
 * phase equals the sum of the earlier shares' newline counts mod 4 (mlgi_share_info); otherwise the file is not 4-line
 * FASTQ and must be read whole. */
int mlgi_open_share(const char* path, int input_type, int threads, uint64_t begin, uint64_t end, mlgi_reader** out);
/* after mlgi_next returned 0: text offset of the share's first line, its number of '\n', and the phase it took (-1: the
 * share is empty, -2: no record start near it) */
int mlgi_share_info(mlgi_reader* r, uint64_t* first, uint64_t* newlines, int* phase);
/* totals so far: reads and bases delivered, compressed/raw bytes consumed from the file */
int mlgi_stats(mlgi_reader* r, uint64_t* reads, uint64_t* bases, uint64_t* text_bytes);
void mlgi_close(mlgi_reader* r);

/* Whole files, for the sketch builder (mlg_db_builder_add_fasta): each file of paths[] inflated whole and raw (headers and
 * newlines kept), in the order given.  `threads` workers (<= 0: all hardware threads) inflate one file each -- BGZF members,
 * other gzip streams with every member's CRC-32 and length checked, plain files with read(2) -- and run a few files ahead
 * of the consumer.  A batch does not depend on the number of workers. */
typedef struct mlgi_files mlgi_files;
int mlgi_files_open(const char* const* paths, uint32_t nfiles, int threads, mlgi_files** out);
/* Next batch: the next consecutive files, at most max_files of them, as many as fit in buf[0, cap); file i of the batch is
 * buf[file_off[i], file_off[i + 1]), file_off has max_files + 1 entries.  Returns 1 with *n_files > 0, 0 at the end, -3
 * when a file cannot be read or inflated (the message names it), 2 when the next file alone is larger than cap: nothing was
 * taken, *need (if not null) is its size, and a call with a buffer of that size delivers it. */
int mlgi_files_next(mlgi_files* r, uint8_t* buf, uint64_t cap, uint64_t* file_off, uint32_t max_files, uint32_t* n_files, uint64_t* need);
void mlgi_files_close(mlgi_files* r);

/* KMC k-mer databases (<prefix>.kmc_pre / .kmc_suf, both layouts) -- the artefacts scripts/select_db.py:44,50-56 of the
 * reference hands between kmc, kmc_tools and kmc_dump.  keys: total x (hi, lo) 2k-bit integers, first base most significant
 * (the key form of include/metalign_b200.h), in file order; k <= 63.  UNPINNED against files made by a real kmc. */
typedef struct mlgi_kmcdb mlgi_kmcdb;
int mlgi_kmc_open(const char* prefix, mlgi_kmcdb** out);
int mlgi_kmc_info(mlgi_kmcdb* d, uint32_t* k, uint64_t* total, uint32_t* counter_size, uint32_t* min_count, uint64_t* max_count,
                  int* canonical, uint32_t* version);
int mlgi_kmc_read(mlgi_kmcdb* d, uint64_t* keys, uint32_t* counts_or_null);
void mlgi_kmc_close(mlgi_kmcdb* d);

#ifdef __cplusplus
}
#endif
#endif
