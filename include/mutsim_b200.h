/*
 * mutsim_b200.h — C ABI of libmutsim_b200.so, the B200 (sm_100a) implementation of
 * Mutation-Simulator's mutation-injection hot path.
 *
 * The reference (mkpython3/Mutation-Simulator 3.0.2) is pure Python and has no
 * FFI of its own; the boundary it exposes for this path is the class API
 *   Mutator(args, fasta, sim).mutate()        mutation_simulator/mutator.py:79,105
 *   ITMutator(args, fasta, sim).mutate()      mutation_simulator/it_mutator.py:25,215
 * Each entry point below names the reference code it replaces.  The Python side
 * (mutation_simulator_b200/) binds these with ctypes and mirrors the reference's
 * classes on top; INTEGRATION.md shows the stub a maintainer of the reference
 * would add.
 *
 * Conventions: plain pointers and sizes only; every call returns an int status
 * (0 = MS_OK) and leaves a message retrievable with ms_last_error(); HOST
 * pointers are caller-owned; device memory is owned by the context until
 * ms_destroy(); all work is ordered on the context's CUDA stream; calls that
 * return sizes or copy to the host synchronise that stream.
 * There is no CPU fallback: without a CUDA device ms_create() fails.
 *
 * Mutation type codes (reference dict order, rmt.py:443-450 and :91-94):
 *   0 SN  1 IN  2 DE  3 IV  4 DU  5 TL  6 TLI  (7 IT: interchromosomal segment)
 */
#ifndef MUTSIM_B200_H
#define MUTSIM_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ms_ctx ms_ctx;

enum {
    MS_OK = 0,
    MS_ERR_CUDA = 1,        /* a CUDA runtime call failed (message has file:line) */
    MS_ERR_ARG = 2,         /* invalid argument */
    MS_ERR_STATE = 3,       /* call order violated (e.g. apply before a genome is resident) */
    MS_ERR_SAMPLE = 4,      /* k > population or k < 0: what random.sample raises as ValueError (util.py:104) */
    MS_ERR_OVERLAP = 5,     /* records overlap / run past a contig end */
    MS_ERR_LIMIT = 6,       /* size limit of this build exceeded (contig >= 2^31 bases, body >= 2^32 bytes) */
    MS_ERR_INTERNAL = 7
};

/* 32-byte splice descriptor (mutation_simulator_b200/csrc/ms_records.h, `Rec`). */
typedef struct {
    uint32_t pos, cons, prod, out;
    int64_t src;
    uint8_t kind, type, ref, alt;
    uint32_t contig;
} ms_rec;

/* One RMT range with mutations (rmt.py:166-189 RangeDefinition + :79-163 MutationSettings). */
typedef struct {
    uint32_t contig;       /* local contig index */
    uint32_t start, stop;  /* 0-based inclusive */
    uint32_t k;            /* int(((stop-start)+1)*sum(rates)) — computed by the caller in float64, mutator.py:225 */
    int64_t limit;         /* exclusive end an SV may reach: contig length or start of the next None range */
    double cdf[7];         /* cumulative mut_chances, canonical type order */
    int32_t minlen[7];
    int32_t maxlen[7];
} ms_range;

typedef struct {
    int64_t n_candidates, n_accepted, n_records, lit_bytes, fasta_bytes, vcf_bytes, kernel_launches;
    int64_t counts[8];           /* records per mutation type */
    float stage_ms[16];          /* CUDA-event time of each pipeline stage of the last call (see ms_stage_name) */
} ms_stats;

/* ---- lifecycle --------------------------------------------------------- */
int ms_create(int device, ms_ctx** ctx);
int ms_destroy(ms_ctx* ctx);
const char* ms_last_error(const ms_ctx* ctx);   /* ctx may be NULL: error of the last failed ms_create */
int ms_abi_version(void);
/* Run on an existing CUDA stream (e.g. torch's current stream) instead of the context's own. */
int ms_set_stream(ms_ctx* ctx, void* cuda_stream);
int ms_synchronize(ms_ctx* ctx);

/* ---- genome ------------------------------------------------------------
 * Replaces the per-base pyfaidx access of the walk (mutator.py:119,133-139,423;
 * util.py:77-91 load_fasta).  `bases` = all contigs concatenated, upper-cased
 * (util.py:87), no line breaks; bpl = bases per line of each input record
 * (pyfaidx lenc, mutator.py:133-134); headers = full deflines without '>'
 * (long_name, mutator.py:135-136); names = first token (VCF CHROM, mutator.py:341);
 * gid = index of the contig in the whole FASTA — the RNG key, so that results do
 * not depend on how contigs are partitioned over GPUs (NULL: 0..n-1).
 * hdr_off / name_off have n_contigs+1 entries. */
int ms_genome_upload(ms_ctx* ctx, const uint8_t* bases, int64_t total_bases, int32_t n_contigs,
                     const int64_t* contig_len, const int32_t* bpl, const uint32_t* gid,
                     const uint8_t* headers, const int64_t* hdr_off,
                     const uint8_t* names, const int64_t* name_off);
/* Same, from a DEVICE pointer (bases already resident, e.g. produced by ms_genome_synth). */
int ms_genome_adopt(ms_ctx* ctx, const uint8_t* d_bases, int64_t total_bases, int32_t n_contigs,
                    const int64_t* contig_len, const int32_t* bpl, const uint32_t* gid,
                    const uint8_t* headers, const int64_t* hdr_off,
                    const uint8_t* names, const int64_t* name_off);
/* Synthetic iid-ACGT genome with N runs generated on the device (benchmarks; SURVEY.md §8d).  Base j of contig gid is a
 * function of (seed, gid, j) only, so any partition of the contigs over GPUs synthesises the same genome. */
int ms_genome_synth(ms_ctx* ctx, uint64_t seed, int32_t n_contigs, const int64_t* contig_len,
                    const int32_t* bpl, const uint32_t* gid, double n_fraction, int64_t telomere_n,
                    const uint8_t* headers, const int64_t* hdr_off,
                    const uint8_t* names, const int64_t* name_off);
int ms_genome_download(ms_ctx* ctx, uint8_t* bases, int64_t cap);
/* Make the mutated genome of the last ms_apply the resident genome (headers / line breaks stripped on the device):
 * what __main__.py:88-95 does by re-loading the just-written *_ms.fa before ITMutator runs.  Contig lengths become
 * the mutated lengths; bpl follows pyfaidx's rule for the re-loaded file (a contig shorter than one line gets
 * bpl = its length).  Records and ranges are cleared. */
int ms_genome_adopt_output(ms_ctx* ctx);
/* ---- FASTA ingest on the device ------------------------------------------
 * Replaces util.py:77-91 (load_fasta -> pyfaidx.Fasta: build the index, serve upper-cased bases) for regularly wrapped
 * files.  ms_fasta_ingest_fd reads the open file through two pinned staging buffers into device memory (pread of one
 * chunk overlapping the H2D copy of the previous) and finds records and their line layout there; *regular = 0 means the
 * file needs the host parser (CRLF, text before the first record, lines or deflines over 1 MiB).  ms_fasta_index
 * returns what pyfaidx stores per record (.fai: length, offset of the first base, bases and bytes per line) and the
 * deflines (without '>'), packed, hdr_off having n_records + 1 entries; hdr_blob may be NULL to query sizes.
 * ms_fasta_commit strips line breaks, upper-cases (util.py:87) and verifies every line against the index in one pass,
 * making the bases the resident genome (headers / names / gid as for ms_genome_upload); *regular = 0 if the bytes do
 * not fit the index (ragged or blank lines) — nothing is resident then.  ms_genome_read copies a slice of the resident
 * bases to the host (the lazy per-record views of the Python Fasta object). */
int ms_fasta_ingest_fd(ms_ctx* ctx, int fd, int64_t nbytes, int32_t* n_records, int32_t* regular);
/* The same for a SUBSET of the file: the image is the concatenation of the byte ranges [off[r], off[r] + len[r]), each
 * made of whole records ('>' ... up to the next record).  With one process per GPU every rank finds the record starts
 * of its 1/N slice of the file, the ranks exchange them, and each then reads only the records of its own contigs
 * (mutator.py:111 iterates contigs independently) — ingest time and host traffic shrink with the GPU count instead of
 * every rank reading the whole file.  seq_off of ms_fasta_index is then relative to the image, not the file. */
int ms_fasta_ingest_ranges(ms_ctx* ctx, int fd, int32_t n_ranges, const int64_t* off, const int64_t* len,
                           int32_t* n_records, int32_t* regular);
int ms_fasta_index(ms_ctx* ctx, int64_t* hdr_off, int64_t* seq_off, int64_t* length, int32_t* lenc, int32_t* lenb,
                   uint8_t* hdr_blob, int64_t blob_cap);
int ms_fasta_commit(ms_ctx* ctx, const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off,
                    const uint8_t* names, const int64_t* name_off, int32_t* regular);
int ms_genome_read(ms_ctx* ctx, int64_t off, int64_t n, uint8_t* dst);
/* Keep only the listed contigs of the resident genome (in the given order; their gid — the RNG key — is unchanged).
 * With several GPUs every rank ingests the file and keeps its share (mutator.py:111 iterates contigs independently). */
int ms_genome_subset(ms_ctx* ctx, const int32_t* ids, int32_t n);
/* Contig table only: the bases follow with ms_mutate_streamed. */
int ms_genome_declare(ms_ctx* ctx, int64_t total_bases, int32_t n_contigs, const int64_t* contig_len,
                      const int32_t* bpl, const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off,
                      const uint8_t* names, const int64_t* name_off);
/* Reserve `extra_bytes` of staging space behind the genome for bases of contigs that live on another GPU
 * (interchromosomal partners, it_mutator.py:133-137).  Call before ms_genome_upload (a genome that is already resident
 * is moved into a buffer with the extra space).  The region starts at
 * genome index total_bases + 64 (ms_device_ptr(4) gives the base pointer); K_RAW records may point into it,
 * so a peer's ncclSend or ms_peer_pull can land directly where the splice kernel gathers from. */
int ms_genome_reserve(ms_ctx* ctx, int64_t extra_bytes);
/* Peer windows: with one process per GPU the partner contig of an interchromosomal pair (it_mutator.py:91-102 picks
 * the pairs, :133-142 swaps the odd intervals) may live in another process.  The owner exports its resident genome
 * buffer (a 64-byte CUDA IPC handle; valid until the owner uploads, reserves or destroys), the reader maps it and gets
 * `rel_off` = (mapped base - its own genome pointer): a K_RAW record whose src = rel_off + the interval's index in the
 * owner's genome makes the splice kernel gather those bases in place over NVLink — no staging copy, no collective.
 * ms_peer_pull instead copies intervals (src relative like above) into the staging region of ms_genome_reserve
 * (dst = genome index >= total_bases + 64) on the context's stream.  The caller orders the two processes: export after
 * the owner's genome is final, close every window before the owner frees it. */
int ms_genome_export(ms_ctx* ctx, uint8_t* handle64, int64_t* nbytes);
int ms_peer_open(ms_ctx* ctx, const uint8_t* handle64, int64_t nbytes, int64_t* rel_off);
int ms_peer_pull(ms_ctx* ctx, int32_t n, const int64_t* src, const int64_t* dst, const int64_t* nbytes);
int ms_peer_close(ms_ctx* ctx);

/* ---- fresh sampling ----------------------------------------------------
 * Replaces Mutator.__get_mutations / __get_mut_positions / __get_stop_position /
 * __link_tls (mutator.py:144-316) and util.sample_with_minimum_distance
 * (util.py:94-109) for all ranges of all contigs at once.
 * block[7] = SimulationSettings.mut_block (rmt.py:326-345), min_dist = min(block)
 * (mutator.py:161), p_ti = titv*(1/(titv+1)) (mutator.py:436). */
int ms_set_ranges(ms_ctx* ctx, const ms_range* ranges, int32_t n_ranges, const int32_t* block,
                  int32_t min_dist, double p_ti);
int ms_sample(ms_ctx* ctx, uint64_t seed);

/* ---- replay ------------------------------------------------------------
 * Loads an explicit mutation table (what Mutator.__mutate_sequence receives as
 * `muts`, mutator.py:318) as splice descriptors sorted by (contig, pos). */
int ms_load_records(ms_ctx* ctx, const ms_rec* recs, int64_t n_recs, const uint8_t* lit, int64_t lit_bytes);
/* Parse VCF text (header lines skipped) into the context's record table and literal pool: what records_from_vcf
 * (mutation_simulator_b200/records.py:119-191) + ms_load_records do, parsed on the device, for the regular shape of
 * the lines VcfWriter.write emits (the reference's vcf_writer.py:118-126, and this package's VCF body): lines end in
 * '\n' (no '\r' or other line breaks), >= 8 tab-separated fields, CHROM one of the resident contigs' names (lines of
 * other contigs are dropped when skip_unknown is 1), POS ASCII digits, INFO '.' or exactly
 * SVTYPE=<type>;END=<digits>;SVLEN=<digits>, every contig's lines in one block with increasing POS (blocks in any
 * contig order), every record inside its contig.  The text is copied to the device in chunks.
 * *regular = 0: nothing was loaded (the context is unchanged) and the caller must use the host parser.  *regular = 1:
 * the table is byte-identical to records_from_vcf's, with literal offsets in file order; the checks of
 * ms_load_records ran with its error codes, and *n_recs holds the number of records. */
int ms_load_vcf(ms_ctx* ctx, const uint8_t* text, int64_t nbytes, int32_t skip_unknown,
                int32_t* regular, int64_t* n_recs);

/* ---- apply -------------------------------------------------------------
 * Replaces Mutator.__mutate_sequence (mutator.py:318-426) with FastaWriter
 * (fasta_writer.py:40-65) and VcfWriter.write (vcf_writer.py:118-126): builds the
 * complete output FASTA image and the VCF body (no header) in device memory. */
int ms_apply(ms_ctx* ctx, int64_t* fasta_bytes, int64_t* vcf_bytes);
/* ms_apply for ONE PART of the output when several GPUs hold the same genome and the same record table (sampling is
 * keyed by (seed, contig id, position), so every GPU that runs ms_sample with the same seed draws the same table):
 * part `part` of `n_parts` produces the 16 KiB tiles [T*part/n, T*(part+1)/n) of the FASTA image (T = all tiles) and the
 * VCF lines of records [M*part/n, M*(part+1)/n).  This is the chunking of a contig that is larger than one GPU's share
 * — mutator.py:332 walks a contig serially and README.md:441 benchmarks a single 1 Gbp contig; here the cut points are
 * tile boundaries of the OUTPUT, and the rejection carry (mutator.py:184-213), the running length delta and the TLI
 * sources (mutator.py:401-406) that cross a cut need no exchange because only the byte-moving stages are sharded.
 * window[6] = { fasta_bytes, vcf_bytes (whole outputs), fasta_lo, fasta_hi, vcf_lo, vcf_hi (byte ranges this part
 * wrote; the buffers returned by ms_download / ms_download_to_fd are valid inside them only) }. */
int ms_apply_window(ms_ctx* ctx, int32_t part, int32_t n_parts, int64_t* window);
/* Mutator.mutate() (mutator.py:105-142) for a genome in HOST memory in one call: = ms_genome_upload + ms_sample +
 * ms_apply + ms_download of both outputs, with the copies overlapped with the kernels.  Contigs are grouped
 * (>= group_min_bases per group, 0 = 48 Mbp); the upload of group g+1, the splice of group g and the download of group g-1 run
 * concurrently on three streams (PCIe is full duplex).  Everything that does not need bases — positions, types,
 * lengths, conflict resolution, TL links, the output layout — runs while the first group is still in flight.
 * Needs ms_genome_declare + ms_set_ranges first; `bases` as for ms_genome_upload (any case); pinned host buffers
 * give the overlap, pageable ones still work.  Results are byte-identical to the unstreamed calls. */
int ms_mutate_streamed(ms_ctx* ctx, uint64_t seed, const uint8_t* bases, uint8_t* fasta, int64_t fasta_cap,
                       uint8_t* vcf, int64_t vcf_cap, int64_t* fasta_bytes, int64_t* vcf_bytes,
                       int64_t group_min_bases);
/* which: 0 FASTA image, 1 VCF body, 2 records (ms_rec[]), 3 literal pool, 4 resident genome, 5 BGZF output of the
 * last ms_bgzf_compress */
int ms_download(ms_ctx* ctx, int which, void* dst, int64_t cap, int64_t* nbytes);
int ms_device_ptr(ms_ctx* ctx, int which, void** dptr, int64_t* nbytes);
/* Stream bytes [src_off, src_off+nbytes) of an output buffer into an open file at file_off: D2H through two pinned
 * staging buffers with the pwrite of one chunk overlapping the copy of the next.  Replaces the per-base
 * file.write() calls of FastaWriter.write (fasta_writer.py:49-58) / VcfWriter.write (vcf_writer.py:118-126) for a whole
 * file (or, with several GPUs, one contig's slice of it). */
int ms_download_to_fd(ms_ctx* ctx, int which, int64_t src_off, int64_t nbytes, int fd, int64_t file_off);
int ms_contig_out_len(ms_ctx* ctx, int64_t* out_len /* n_contigs */);
/* Per-contig slices of the last ms_apply outputs, for assembling one file from several GPUs:
 * fasta_off[c]..fasta_off[c+1] = header + body (+ separator) bytes of contig c in the FASTA image,
 * vcf_off[c]..vcf_off[c+1] = its VCF lines; sep[c] = 1 if the slice ends with the '\n' that closes a partial
 * last line (fasta_writer.py:44-45); partial[c] = 1 if the last line is partial.  Arrays have n_contigs+1 /
 * n_contigs entries. */
int ms_contig_layout(ms_ctx* ctx, int64_t* fasta_off, int64_t* vcf_off, uint8_t* sep, uint8_t* partial);
/* Number of records (applied mutations) of each contig after ms_sample / ms_load_records + ms_apply. */
int ms_contig_records(ms_ctx* ctx, int64_t* n_records /* n_contigs */);

/* ---- interchromosomal translocations ------------------------------------
 * Replaces ITMutator.__get_breakpoints (it_mutator.py:94-118): for each pair p,
 * n[p] breakpoints on each member, sample_with_minimum_distance(1, len, n, 1).
 * bp_a/bp_b receive sum(n) sorted positions each (pair-major). */
int ms_it_breakpoints(ms_ctx* ctx, uint64_t seed, int32_t n_pairs, const uint32_t* contig_a,
                      const uint32_t* contig_b, const uint32_t* n, uint32_t* bp_a, uint32_t* bp_b);
/* util.sample_with_minimum_distance (util.py:94-109) for many ranges at once, independent of the resident
 * genome: range i = (gid[i], start[i], stop[i], k[i]); out receives sum(k) sorted positions, range-major.
 * The stream is keyed by (seed, gid, start), so any GPU computes the same positions. */
int ms_sample_positions(ms_ctx* ctx, uint64_t seed, int32_t n, const uint32_t* gid, const uint32_t* start,
                        const uint32_t* stop, const uint32_t* k, int32_t min_dist, uint32_t* out);

/* 64-bit content hash of byte ranges [start[i], end[i]) of an output buffer (`which` as for ms_download), computed on
 * the device: sum over the range's bytes of mix(byte, offset within the range) mod 2^64 — order-free, so any launch
 * geometry gives the same value.  bench.py uses it to check that the N-GPU outputs are the 1-GPU outputs without
 * moving them off the devices (SURVEY.md §4.5: results must not depend on the GPU count). */
int ms_hash_ranges(ms_ctx* ctx, int which, int32_t n, const int64_t* start, const int64_t* end, uint64_t* out);

/* ---- BGZF output ---------------------------------------------------------
 * Compresses segments of buffer `which` (0 FASTA image, 1 VCF body) into BGZF members on the device; the members,
 * back to back in segment order, become buffer 5 (ms_download, ms_download_to_fd, ms_device_ptr, ms_hash_ranges).
 * Segment s is bytes [src_off[s], src_off[s] + nbytes[s]) of the buffer, followed by one '\n' when add_nl[s] is 1
 * (add_nl may be NULL), and starts at byte file_off[s] of the uncompressed file.  Members never span two segments
 * and are cut at multiples of 16 KiB of the file, so a member is a pure function of the file's bytes and of where
 * the segments begin: pass one segment per contig (ms_contig_layout) and several GPUs write the same file as one.
 * Each member is a literal-only dynamic-Huffman deflate block, or a stored block when that is smaller (a member is
 * at most its input + 31 bytes).  seg_zbytes[s] receives segment s's compressed size; the caller appends the 28-byte
 * BGZF end-of-file member. */
int ms_bgzf_compress(ms_ctx* ctx, int which, int32_t n_seg, const int64_t* src_off, const int64_t* nbytes,
                     const int64_t* file_off, const uint8_t* add_nl, int64_t* seg_zbytes, int64_t* total_zbytes);
/* The same encoder on the host for small data (the VCF header): src[0..n) as members of 16 KiB each into dst.
 * dst = NULL queries an upper bound of the size.  ctx may be NULL (no device is used). */
int ms_bgzf_compress_host(ms_ctx* ctx, const uint8_t* src, int64_t n, uint8_t* dst, int64_t cap, int64_t* zbytes);

/* ---- introspection ------------------------------------------------------ */
int ms_get_stats(ms_ctx* ctx, ms_stats* out);
const char* ms_stage_name(int stage);
/* Debug/validation taps used by the parity tests: candidates after K1..K3. */
int ms_debug_candidates(ms_ctx* ctx, int64_t cap, int64_t* gpos, uint8_t* type, uint32_t* len, uint8_t* accept,
                        int64_t* n);

#ifdef __cplusplus
}
#endif
#endif /* MUTSIM_B200_H */
