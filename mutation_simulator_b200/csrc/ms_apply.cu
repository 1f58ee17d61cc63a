// ms_apply.cu — K5 (plan: delta scan, layout, block index), K6 (splice + SNP +
// line wrap -> FASTA image), K7 (VCF lines).  Replaces Mutator.__mutate_sequence
// (mutator.py:318-426), FastaWriter (fasta_writer.py:40-65) and VcfWriter.write
// (vcf_writer.py:118-126).
#include <algorithm>
#include <climits>
#include "ms_common.cuh"
#include "ms_scan.cuh"
#include "ms_splice_core.h"
#define MS_TILE_RAND_OOL 1
#include "ms_tile_core.h"
#include "ms_vcf_core.h"
#include "ms_sample_core.h"

namespace ms {

// Random-insert bytes are rare (0.5 % of the output); calling Philox out of line keeps it from inflating the
// register count (and lowering the occupancy) of the kernels that consume them.
__device__ __noinline__ uint8_t rand_base_ool(Seed seed, uint32_t gid, uint32_t pos, uint32_t j) {
    return rand_insert_base(seed, gid, pos, j);
}

__device__ inline void raise_error(Totals* t, int64_t code, int64_t arg) {
    if (atomicCAS((unsigned long long*)&t->error, 0ull, (unsigned long long)code) == 0ull) t->error_arg = arg;
}

// ---- record ranges per contig -------------------------------------------------------
__global__ void k_rec_bounds(const Rec* recs, int64_t n_recs, Contig* contigs, int32_t n_contigs) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > n_contigs) return;
    int64_t lo = 0, hi = n_recs;  // first record with contig >= c
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (recs[mid].contig < (uint32_t)c) lo = mid + 1; else hi = mid;
    }
    if (c < n_contigs) contigs[c].rec_lo = lo;
    if (c > 0) contigs[c - 1].rec_hi = lo;
}

// ---- layout of the output file image ---------------------------------------------------
// One CTA walks the contigs in FASTA order (they are few: 24 .. 200k) carrying the
// running file offset and piece count.
__global__ void __launch_bounds__(SCAN_THREADS)
k_contig_layout(Contig* contigs, int32_t n_contigs, const int64_t* S, int64_t* piece_lo, int64_t tile_bytes,
                Totals* tot, int64_t n_recs, const int64_t* V, const uint32_t* N) {
    __shared__ int64_t sm1[2 * SCAN_THREADS / 32];
    int64_t carry = 0;
    for (int base = 0; base < n_contigs; base += SCAN_THREADS) {
        const int c = base + threadIdx.x;
        int64_t v = 0;
        if (c < n_contigs) {
            Contig& k = contigs[c];
            const int64_t delta = S[k.rec_hi] - S[k.rec_lo];
            const int64_t out_len = k.len + delta;
            if (out_len < 0) raise_error(tot, MS_ERR_OVERLAP, c);
            k.out_len = out_len;
            const int64_t bpl = k.bpl;
            k.body_bytes = out_len + out_len / bpl;
            if (k.body_bytes >= (int64_t)0xFFFFFFF0ll || out_len >= (int64_t)0xFFFFFFF0ll) raise_error(tot, MS_ERR_LIMIT, c);
            k.sep = (out_len % bpl != 0 && c != n_contigs - 1) ? 1u : 0u;
            v = (int64_t)k.hdr_len + 2 + k.body_bytes + k.sep;
        }
        int64_t total;
        const int64_t ex = block_excl_scan(v, (int64_t)0, SumOp(), total, sm1);
        if (c < n_contigs) {
            Contig& k = contigs[c];
            k.hdr_off = carry + ex;
            k.body_off = k.hdr_off + k.hdr_len + 2;
        }
        carry += total;
    }
    __syncthreads();
    int64_t pcarry = 0;
    for (int base = 0; base < n_contigs; base += SCAN_THREADS) {
        const int c = base + threadIdx.x;
        int64_t np = 0;
        if (c < n_contigs) {
            const Contig& k = contigs[c];
            if (k.body_bytes > 0) np = (k.body_off + k.body_bytes - 1) / tile_bytes - k.body_off / tile_bytes + 1;
        }
        int64_t total;
        int64_t ex = block_excl_scan(np, (int64_t)0, SumOp(), total, sm1);
        if (c < n_contigs) { contigs[c].piece_lo = pcarry + ex; piece_lo[c] = pcarry + ex; }
        pcarry += total;
    }
    if (threadIdx.x == 0) {
        piece_lo[n_contigs] = pcarry;
        tot->fasta_bytes = carry;
        tot->n_blk = (int64_t)N[n_recs];          // (field reused: number of SvRecs)
        tot->n_pieces = pcarry;
        tot->vcf_bytes = V[n_recs];
        tot->n_recs = n_recs;
    }
}

// The same layout for large contig tables (many-small-contig genomes): two device-wide scans instead of one CTA
// walking 200 k contigs (3.6 ms on C5).
__global__ void k_layout_totals(const int64_t* t1, const int64_t* t2, int64_t* piece_lo, int32_t n_contigs, Totals* tot, int64_t n_recs,
                                const int64_t* V, const uint32_t* N) {
    piece_lo[n_contigs] = *t2;
    tot->fasta_bytes = *t1; tot->n_blk = (int64_t)N[n_recs]; tot->n_pieces = *t2;
    tot->vcf_bytes = V[n_recs]; tot->n_recs = n_recs;
}

static int layout_by_scan(ms_ctx* c, Contig* d_contigs, const int64_t* S, const int64_t* V, const uint32_t* N, int64_t M, Totals* d_tot) {
    const int32_t n = c->n_contigs;
    int64_t* d_piece_lo = c->piece_lo.as<int64_t>();
    const int64_t tile_bytes = c->tile_bytes;
    MS_CUDA(c, c->scan_tmp2.ensure(64));
    int64_t* d_t1 = c->scan_tmp2.as<int64_t>();
    int64_t* d_t2 = d_t1 + 1;
    {
        auto in = [=] __device__(int64_t i) -> int64_t {
            Contig& k = d_contigs[i];
            const int64_t out_len = k.len + (S[k.rec_hi] - S[k.rec_lo]);
            if (out_len < 0) raise_error(d_tot, MS_ERR_OVERLAP, i);
            const int64_t bpl = k.bpl;
            const int64_t body = out_len + out_len / bpl;
            if (body >= (int64_t)0xFFFFFFF0ll) raise_error(d_tot, MS_ERR_LIMIT, i);
            const uint32_t sep = (out_len % bpl != 0 && i != n - 1) ? 1u : 0u;
            k.out_len = out_len; k.body_bytes = body; k.sep = sep;
            return (int64_t)k.hdr_len + 2 + body + sep;
        };
        auto out = [=] __device__(int64_t i, int64_t ex, int64_t) {
            Contig& k = d_contigs[i];
            k.hdr_off = ex; k.body_off = ex + k.hdr_len + 2;
        };
        int64_t* tot1 = nullptr;
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, (int64_t)n, (int64_t)0, SumOp(), c->scan_tmp, &tot1)));
        MS_CUDA(c, cudaMemcpyAsync(d_t1, tot1, sizeof(int64_t), cudaMemcpyDeviceToDevice, c->stream));
    }
    {
        auto in = [=] __device__(int64_t i) -> int64_t {
            const Contig& k = d_contigs[i];
            return k.body_bytes > 0 ? (k.body_off + k.body_bytes - 1) / tile_bytes - k.body_off / tile_bytes + 1 : 0;
        };
        auto out = [=] __device__(int64_t i, int64_t ex, int64_t) { d_contigs[i].piece_lo = ex; d_piece_lo[i] = ex; };
        int64_t* tot2 = nullptr;
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, (int64_t)n, (int64_t)0, SumOp(), c->scan_tmp, &tot2)));
        MS_CUDA(c, cudaMemcpyAsync(d_t2, tot2, sizeof(int64_t), cudaMemcpyDeviceToDevice, c->stream));
    }
    k_layout_totals<<<1, 1, 0, c->stream>>>(d_t1, d_t2, d_piece_lo, n, d_tot, M, V, N);
    MS_LAUNCH_CHECK(c);
    return MS_OK;
}

// ---- out positions, validation, and the two record streams the splice kernel reads -----------------------------
// S[i] = sum of length deltas before record i, N[i] = number of non-SNP records before i (both over all contigs).
// Record i lands in slot N[i] of the SvRec stream or slot i - N[i] of the Snp8 stream; a contig's entries are
// [N[rec_lo], N[rec_hi]) resp. [rec_lo - N[rec_lo], rec_hi - N[rec_hi]).  The record table itself is only read.
__device__ __forceinline__ void rec_out_one(const Rec* recs, int64_t i, const Contig* contigs, const int64_t* S, const uint32_t* N, SvRec* sv,
                                            Snp8* snp, Totals* tot, unsigned int* hist) {
    const Rec r = recs[i];
    {   // one shared-memory atomic per (warp, type): three quarters of a warp's lanes hold the same type
        const uint32_t t = r.type < 8 ? r.type : 8u;
        const uint32_t peers = __match_any_sync(__activemask(), t);
        if (t < 8u && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[t], (unsigned)__popc(peers));
    }
    const Contig& k = contigs[r.contig];
    const int64_t out = (int64_t)r.pos + (S[i] - S[k.rec_lo]);
    if ((int64_t)r.pos + r.cons > k.len) raise_error(tot, MS_ERR_OVERLAP, i);
    if (i > k.rec_lo) {
        const Rec p = recs[i - 1];
        if ((int64_t)r.pos < (int64_t)p.pos + p.cons || r.pos == p.pos) raise_error(tot, MS_ERR_OVERLAP, i);
    }
    const uint32_t nsv = N[i];
    if (r.kind == K_SNP) snp[i - (int64_t)nsv] = Snp8{(uint32_t)out, (uint32_t)r.alt};
    else sv[nsv] = SvRec{(uint32_t)out, r.prod, r.pos + r.cons, r.pos, r.src, (uint32_t)r.kind, 0u};
}

// Rec.out is not needed on the device any more (the streams carry it); it is filled in when the records are handed out
// (ms_download / ms_device_ptr of the record table).
__global__ void __launch_bounds__(256) k_fill_out(Rec* recs, int64_t n_recs, const Contig* contigs, const int64_t* S) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_recs) return;
    const Contig& k = contigs[recs[i].contig];
    recs[i].out = (uint32_t)((int64_t)recs[i].pos + (S[i] - S[k.rec_lo]));
}

int fill_record_out(ms_ctx* c) {
    if (c->rec_out_valid || c->n_recs <= 0) return MS_OK;
    k_fill_out<<<(unsigned)ceil_div(c->n_recs, 256), 256, 0, c->stream>>>(c->recs.as<Rec>(), c->n_recs, c->contigs.as<Contig>(), c->svec.as<int64_t>());
    MS_LAUNCH_CHECK(c);
    c->rec_out_valid = true;
    return MS_OK;
}



__global__ void __launch_bounds__(256)
k_rec_out(const Rec* recs, int64_t n_recs, const Contig* contigs, const int64_t* S, const uint32_t* N, SvRec* sv, Snp8* snp, Totals* tot) {
    __shared__ unsigned int hist[8];          // records per mutation type (ms_get_stats), counted on the way
    if (threadIdx.x < 8) hist[threadIdx.x] = 0u;
    __syncthreads();
    // grid-stride: a few thousand CTAs flush their counts at the end instead of one CTA per 256 records (163 k CTAs
    // x 8 atomics on the same eight words were 40 % of this kernel's stall samples, profiles/r3f)
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < n_recs; i0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = i0 + threadIdx.x;
        if (i < n_recs) rec_out_one(recs, i, contigs, S, N, sv, snp, tot, hist);
    }
    __syncthreads();
    if (threadIdx.x < 8 && hist[threadIdx.x]) atomicAdd((unsigned long long*)&tot->counts[threadIdx.x], (unsigned long long)hist[threadIdx.x]);
}

// ---- K6: splice + SNP + line wrap -----------------------------------------------------
// One CTA per piece (= 16 KiB tile of the output file image intersected with one contig body).
//
// Run-centric splice over the two record streams of the plan pass.  SNPs move nothing, so between two consecutive
// SvRecs the output is one shifted copy of the input ("run", ~290 bases at human-like rates).  A CTA assembles the
// mutated bases of its tile in shared memory:
//   segs one thread per SvRec of the tile: its raw payload (tandem duplication, interchromosomal segment) and its
//        trailing run become copy segments — the SvRec stream IS the run list, no pass over the SNP records
//   S1   every segment is a shifted copy staged-input -> tile, 16 bytes per lane, half a warp per segment
//   S2   one thread per Snp8 scatters the substituted base; one thread per SvRec queues the payloads that have to be
//        generated (random inserts, inversions, translocation inserts) as byte jobs for warps
//   S3   line breaks are inserted while the tile is written out, 16 aligned bytes per lane
// The tile's contiguous input span arrives by ONE bulk copy (TMA) issued before anything else.
constexpr int SPLICE_THREADS = 256;
struct SegC { int64_t src; uint32_t dst; uint32_t n; };   // copy n bytes genome[src..] -> tile[dst..]; jobs: n | kind << 24

// bytes [o, o+16) of the 32-byte window (a, b)
__device__ __forceinline__ uint4 shift16(const uint4 a, const uint4 b, uint32_t o) {
    const bool s2 = (o & 8u) != 0u, s1 = (o & 4u) != 0u;
    const uint32_t t0 = s2 ? a.z : a.x, t1 = s2 ? a.w : a.y, t2 = s2 ? b.x : a.z, t3 = s2 ? b.y : a.w,
                   t4 = s2 ? b.z : b.x, t5 = s2 ? b.w : b.y;
    const uint32_t u0 = s1 ? t1 : t0, u1 = s1 ? t2 : t1, u2 = s1 ? t3 : t2, u3 = s1 ? t4 : t3, u4 = s1 ? t5 : t4;
    const uint32_t bs = (o & 3u) * 8u;
    return make_uint4(__funnelshift_r(u0, u1, bs), __funnelshift_r(u1, u2, bs), __funnelshift_r(u2, u3, bs),
                      __funnelshift_r(u3, u4, bs));
}

constexpr int SP_SEG_CAP = 320;
constexpr int SP_JOB_CAP = 192;
constexpr uint32_t SP_DIRECT = 0xFFFFFFFFu;        // segment did not fit the staging buffer: copied straight from global
constexpr uint32_t SP_SEG_SPLIT = 2048;

__global__ void __launch_bounds__(256)
k_piece_desc(const Contig* contigs, int32_t n_contigs, const int64_t* piece_lo, int64_t n_pieces, const SvRec* sv, const Snp8* snp,
             const uint32_t* N, const Totals* tot, PieceDesc* out) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pieces) return;
    if (tot->error) {   // k_rec_out rejected the records (overlap / out of bounds): every piece becomes empty, the
        PieceDesc z{};  // splice kernel then touches nothing and ms_apply reports the error
        z.bpl = 60u;
        out[p] = z;
        return;
    }
    int lo = 0, hi = n_contigs;  // last c with piece_lo[c] <= p
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (piece_lo[mid] <= p) lo = mid; else hi = mid;
    }
    const Contig k = contigs[lo];
    const int64_t tile_i = (k.body_off >> TL_TILE_SHIFT) + (p - k.piece_lo);
    int64_t f_lo = tile_i << TL_TILE_SHIFT, f_hi = f_lo + TL_TILE;
    if (f_lo < k.body_off) f_lo = k.body_off;
    if (f_hi > k.body_off + k.body_bytes) f_hi = k.body_off + k.body_bytes;
    const int64_t n_lo = (int64_t)N[k.rec_lo], n_hi = (int64_t)N[k.rec_hi];
    out[p] = tile_describe(k, (uint32_t)lo, f_lo, f_hi, sv, n_lo, n_hi, snp, k.rec_lo - n_lo, k.rec_hi - n_hi);
}

// ---- TMA (bulk async copy) + mbarrier, raw PTX -----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion is signalled on `bar`
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_global, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst_smem)),
                 "l"(src_global), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// `bytes` (a multiple of 16) from a 16-byte aligned global address into L2, no destination
__device__ __forceinline__ void bulk_prefetch_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// byte x of a clipped generated payload; s0 as prepared in S2 (RC: last source index, RAND: the cached 2-bit bases
// shifted to the first byte, RANDL (insert reaching past its 32 cached bases): pos << 32 | first byte index)
constexpr uint32_t K_RANDL = 7;
__device__ __forceinline__ uint8_t payload_at(const SpliceView& v, uint32_t kind, int64_t s0, uint32_t x, uint32_t gid) {
    switch (kind) {
        case K_LIT:   return v.lit[s0 + x];
        case K_CONV:  return v.conv[v.genome[s0 + x]];
        case K_RAND:  return cached_insert_base(s0, x);
        case K_RANDL: return rand_base_ool(v.seed, gid, (uint32_t)((uint64_t)s0 >> 32), (uint32_t)s0 + x);
        default:      return v.comp[v.conv[v.genome[s0 - (int64_t)x]]];
    }
}

// 8 lanes per segment (the average run is ~270 bytes = 17 chunks: 16 lanes left a third of them idle and paid the
// per-segment fixed cost twice as often, profiles/r2m).  ql = lane within the quarter-warp; n == 0 makes it idle.
// The ragged ends go in 12 slots — <= 3 bytes and <= 3 words up to the first aligned chunk, <= 3 words and <= 3
// bytes after the last — each read as one unaligned word through a funnel shift.
__device__ __forceinline__ void quarter_copy_stage_to_tile(uint8_t* tile, const uint8_t* stage, uint32_t so, uint32_t d0, uint32_t n, int ql) {
    const uint32_t d1 = d0 + n;
    const uint32_t a0 = (d0 + 15u) & ~15u, a1 = d1 & ~15u;
    if (a0 >= a1) {                                   // no aligned chunk inside: at most 30 bytes
        for (uint32_t x = d0 + ql; x < d1; x += 8u) tile[x] = stage[so + (x - d0)];
        return;
    }
    const uint32_t h4 = (d0 + 3u) & ~3u;              // (<= a0) head: bytes [d0, h4), words [h4, a0)
    const uint32_t t4 = a1 + ((d1 - a1) & ~3u);       // tail: words [a1, t4), bytes [t4, d1)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int slot = ql + 8 * r;                  // 0-2 head bytes, 3-5 head words, 6-8 tail words, 9-11 tail bytes
        if (slot < 12) {
            const uint32_t k = (uint32_t)slot % 3u;
            const bool word = slot >= 3 && slot < 9;
            const uint32_t x = slot < 3 ? d0 + k : slot < 6 ? h4 + 4u * k : slot < 9 ? a1 + 4u * k : t4 + k;
            const uint32_t lim = slot < 3 ? h4 : slot < 6 ? a0 : slot < 9 ? t4 : d1;
            if (x < lim) {
                const uint32_t s = so + (x - d0);
                const uint32_t* w = reinterpret_cast<const uint32_t*>(stage + (s & ~3u));
                const uint32_t v = __funnelshift_r(w[0], w[1], (s & 3u) * 8u);
                if (word) *reinterpret_cast<uint32_t*>(tile + x) = v; else tile[x] = (uint8_t)v;
            }
        }
    }
    for (uint32_t c = a0 + 16u * ql; c < a1; c += 128u) {
        const uint32_t s = so + (c - d0);
        const uint4* w = reinterpret_cast<const uint4*>(stage + (s & ~15u));
        *reinterpret_cast<uint4*>(tile + c) = shift16(w[0], w[1], s & 15u);
    }
}

__device__ __forceinline__ void warp_copy_to_tile(uint8_t* tile, const uint8_t* __restrict__ genome, const SegC sg, int lane) {
    const uint32_t d0 = sg.dst, d1 = sg.dst + sg.n;
    const uint32_t a0 = (d0 + 15u) & ~15u, a1 = d1 & ~15u;
    if (a0 >= a1) {   // no aligned 16-byte chunk inside: at most 30 bytes
        const uint32_t x = d0 + lane;
        if (x < d1) tile[x] = __ldg(genome + sg.src + lane);
        return;
    }
    {   // <= 15 head bytes on lanes 0..15, <= 15 tail bytes on lanes 16..31
        const uint32_t x = lane < 16 ? d0 + lane : a1 + (lane - 16);
        if (x < (lane < 16 ? a0 : d1)) tile[x] = __ldg(genome + sg.src + (x - d0));
    }
    for (uint32_t c = a0 + 16u * lane; c < a1; c += 512u) {
        const int64_t s = sg.src + (int64_t)(c - d0);
        const uint4* w = reinterpret_cast<const uint4*>(genome + (s & ~(int64_t)15));
        const uint4 wa = __ldg(w), wb = __ldg(w + 1);
        *reinterpret_cast<uint4*>(tile + c) = shift16(wa, wb, (uint32_t)(s & 15));
    }
}

constexpr int SP_DYN = TL_TILE + 64 + TL_STAGE_CAP + 32;       // [tile | stage]

__global__ void __launch_bounds__(SPLICE_THREADS, 5)
k_splice(SpliceView v, const Contig* contigs, const PieceDesc* pieces, const SvRec* sv_stream, const Snp8* snp_stream,
         const Tables* tables, uint8_t* fasta, int64_t n_pieces) {
    __shared__ Contig sc;
    __shared__ __align__(16) PieceDesc sd;
    extern __shared__ __align__(16) uint8_t sp_dyn[];
    uint8_t* const tile = sp_dyn;
    uint8_t* const stage = sp_dyn + TL_TILE + 64;
    __shared__ SegC segs[SP_SEG_CAP];
    __shared__ uint32_t seg_stage[SP_SEG_CAP];     // offset of the segment's input in `stage`, or SP_DIRECT
    SegC* const jobs = reinterpret_cast<SegC*>(stage);   // payload jobs are queued after S1, when the staging buffer is dead
    __shared__ __align__(8) uint64_t bar;
    __shared__ int n_segs, n_jobs, fallback;
    __shared__ uint8_t s_conv[256], s_comp[256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t p = blockIdx.x;
    if (warp == 0) {
        reinterpret_cast<uint32_t*>(&sd)[lane] = __ldg(reinterpret_cast<const uint32_t*>(pieces + p) + lane);
        if (lane == 0) { n_segs = 0; n_jobs = 0; fallback = 0; mbar_init(&bar, 1u); }
        __syncwarp();
        // the tile's whole input span as ONE TMA bulk copy, issued before anything else so that it overlaps the
        // segment pass below (S1 waits for it)
        if (lane == 0 && !(sd.flags & PD_FALLBACK)) {
            const uint32_t nb = sd.in_bytes;
            if (nb) tma_load_1d(stage, v.genome + sd.in_lo, nb, &bar);
            mbar_arrive_expect_tx(&bar, nb);
        }
    } else if (warp == 1) {
        // software wave prefetch: the descriptor of the tile that runs in this SM slot two waves from now, and the input
        // span + records of the one a wave from now (its descriptor was requested a wave ago), go to L2
        constexpr int64_t W = 148 * 5;
        if (lane == 0 && p + 2 * W < n_pieces) prefetch_l2(pieces + p + 2 * W);
        if (lane < 3 && p + W < n_pieces) {
            const PieceDesc* nx = pieces + p + W;
            if (lane == 0) {
                const uint32_t nb = __ldg(&nx->in_bytes);
                const int64_t lo = __ldg(&nx->in_lo);
                // not for a span in a peer's HBM (interchromosomal partner on another GPU): the TMA copy of such a span
                // runs at NVLink speed, but an L2 prefetch of a peer address completes one at a time, ≈ 1.6 µs each
                // (measured: 41 ms instead of 1.1 ms for the 26 k remote tiles of C4, profiles/r2w_*)
                if (nb && lo >= 0 && lo < v.local_cap) bulk_prefetch_l2(v.genome + lo, nb);
            } else if (lane == 1) {
                const uint32_t nsv = __ldg(&nx->n_sv);
                if (nsv) bulk_prefetch_l2(sv_stream + __ldg(&nx->sv_lo), 32u * nsv);
            } else {
                const uint32_t nsnp = __ldg(&nx->n_snp);
                if (nsnp) bulk_prefetch_l2(snp_stream + (__ldg(&nx->snp_lo) & ~(int64_t)1), 8u * ((nsnp + 2u) & ~1u));
            }
        }
    }
    s_conv[tid] = tables->conv[tid];
    s_comp[tid] = tables->comp[tid];
    __syncthreads();
    const PieceDesc& k = sd;
    v.conv = s_conv;
    v.comp = s_comp;
    const int64_t f_lo = k.f_lo, f_hi = k.f_hi;
    if (f_hi <= f_lo) return;
    const int64_t g0 = f_lo & ~(int64_t)15;
    const int ngroups = (int)((f_hi - g0 + 15) >> 4);
    const uint32_t bpl = k.bpl, w1 = bpl + 1u;
    const uint32_t b_lo = k.b_lo, b_hi = k.b_hi;   // mutated bases [b_lo, b_hi) live in this tile
    const uint32_t virt = (k.flags & PD_GOV_VIRTUAL) ? 1u : 0u;
    const int n_sv = (int)k.n_sv;                  // slot 0 = the governing record (virtual: the start of the contig)
    const SvRec* const sv = sv_stream + k.sv_lo;   // slot j >= virt is sv[j - virt]
    bool use_fallback = (k.flags & PD_FALLBACK) != 0u;

    if (!use_fallback) {
        // ---- segs: copy segments of every run (raw payload + trailing shifted copy), clipped to the tile
        for (int j = tid; j < n_sv; j += SPLICE_THREADS) {
            uint32_t o = 0u, pr = 0u, kind = K_NONE;
            int64_t run_src = k.goff, psrc = 0;   // source of the base right after the payload
            if (j >= (int)virt) {
                const uint4 a = __ldg(reinterpret_cast<const uint4*>(sv + (j - virt)));        // out, prod, run_in, pos
                const uint4 b = __ldg(reinterpret_cast<const uint4*>(sv + (j - virt)) + 1);    // src, kind
                o = a.x; pr = a.y; kind = b.z;
                run_src = k.goff + (int64_t)a.z;
                psrc = (int64_t)(((uint64_t)b.y << 32) | b.x);
            }
            uint32_t end = j + 1 < n_sv ? __ldg(&sv[j + 1 - virt].out) : b_hi;
            if (end > b_hi) end = b_hi;
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                uint32_t lo, hi;
                int64_t src;
                if (part == 0) {  // raw payload [o, o+pr)
                    if (kind != K_RAW || pr == 0u) continue;
                    lo = o > b_lo ? o : b_lo;
                    hi = o + pr < end ? o + pr : end;
                    src = psrc + (int64_t)(lo - o);
                } else {          // trailing run [o+pr, end)
                    lo = o + pr > b_lo ? o + pr : b_lo;
                    hi = end;
                    src = run_src + (int64_t)(lo - (o + pr));
                }
                while (lo < hi) {
                    const uint32_t n = hi - lo < SP_SEG_SPLIT ? hi - lo : SP_SEG_SPLIT;
                    const int slot = atomicAdd(&n_segs, 1);
                    if (slot < SP_SEG_CAP) {
                        segs[slot] = SegC{src, lo - b_lo, n};
                        // staged iff the segment's source lies inside the span the prologue's TMA copy brings in
                        const int64_t rel = src - k.in_lo;
                        seg_stage[slot] = (rel >= 0 && rel + (int64_t)n <= (int64_t)k.in_bytes) ? (uint32_t)rel : SP_DIRECT;
                    } else {
                        fallback = 1;
                    }
                    lo += n; src += n;
                }
            }
        }
        // one warp waits on the mbarrier (the TMA copy of the input span); the others park at the CTA barrier instead of
        // spinning on try_wait (8 spinning warps were 11.6 % of all issued instructions, profiles/r1h).  The same barrier
        // publishes the segment list.
        if (warp == 0) mbar_wait(&bar, 0u);
        __syncthreads();
        use_fallback = fallback != 0;
    }

    if (!use_fallback) {
        const int ns = n_segs;
        // ---- S1: shifted copies shared -> shared, a quarter of a warp per segment
        {
            const int quarter = lane >> 3, ql = lane & 7;
            bool any_direct = false;
            for (int s0 = 4 * warp; s0 < ns; s0 += 4 * (SPLICE_THREADS / 32)) {
                const int sidx = s0 + quarter;
                uint32_t so = 0u, d0 = 0u, n = 0u;
                if (sidx < ns) {
                    const uint32_t off = seg_stage[sidx];
                    if (off == SP_DIRECT) any_direct = true;
                    else { const SegC sg = segs[sidx]; so = off; d0 = sg.dst; n = sg.n; }
                }
                quarter_copy_stage_to_tile(tile, stage, so, d0, n, ql);
            }
            if (__any_sync(0xffffffffu, any_direct)) {   // segments that did not fit the staging buffer (rare)
                for (int s0 = 4 * warp; s0 < ns; s0 += 4 * (SPLICE_THREADS / 32))
                    for (int h = 0; h < 4; ++h)
                        if (s0 + h < ns && seg_stage[s0 + h] == SP_DIRECT) warp_copy_to_tile(tile, v.genome, segs[s0 + h], lane);
            }
        }
        __syncthreads();
        // ---- S2: SNP bases (one thread per Snp8 of the tile) ...
        {
            const Snp8* snp = snp_stream + k.snp_lo;
            for (uint32_t i = tid; i < k.n_snp; i += SPLICE_THREADS) {
                const uint2 s = __ldg(reinterpret_cast<const uint2*>(snp + i));
                tile[s.x - b_lo] = (uint8_t)s.y;
            }
        }
        // ... and generated payloads (one thread per SvRec; short ones written on the spot, the others queued)
        for (int j = tid + (int)virt; j < n_sv; j += SPLICE_THREADS) {
            const uint4 a = __ldg(reinterpret_cast<const uint4*>(sv + (j - virt)));
            const uint4 b = __ldg(reinterpret_cast<const uint4*>(sv + (j - virt)) + 1);
            const uint32_t o = a.x, pr = a.y, kind = b.z;
            uint32_t pkind = kind;
            if (pr > 0u && kind != K_RAW) {
                const uint32_t lo = o > b_lo ? o : b_lo, hi = o + pr < b_hi ? o + pr : b_hi;
                if (lo < hi) {
                    const int64_t src = (int64_t)(((uint64_t)b.y << 32) | b.x);
                    const uint32_t rel = lo - o, n = hi - lo;
                    // RC walks backwards; a random insert is addressed by (position, first byte index)
                    int64_t s0;
                    if (kind == K_RC) s0 = src + (int64_t)(pr - 1u - rel);
                    else if (kind != K_RAND) s0 = src + rel;
                    else if (rel + n <= 32u) s0 = (int64_t)((uint64_t)src >> (2u * rel));
                    else { s0 = (int64_t)(((uint64_t)a.w << 32) | rel); pkind = K_RANDL; }
                    if (n <= 3u) {
                        for (uint32_t x = 0; x < n; ++x) {
                            const uint8_t ch = payload_at(v, pkind, s0, x, k.gid);
                            tile[lo - b_lo + x] = ch;
                        }
                    } else {
                        const int slot = atomicAdd(&n_jobs, 1);
                        if (slot < SP_JOB_CAP) jobs[slot] = SegC{s0, lo - b_lo, n | (pkind << 24)};
                        else {
                            for (uint32_t x = 0; x < n; ++x) {
                                const uint8_t ch = payload_at(v, pkind, s0, x, k.gid);
                                tile[lo - b_lo + x] = ch;
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();
        const int nj = n_jobs < SP_JOB_CAP ? n_jobs : SP_JOB_CAP;
        for (int jb = warp; jb < nj; jb += SPLICE_THREADS / 32) {
            const SegC job = jobs[jb];
            const uint32_t n = job.n & 0xFFFFFFu, kind = job.n >> 24;
            uint8_t* d = tile + job.dst;
            if (kind == K_RC) {
                const uint8_t* g = v.genome + job.src;
                for (uint32_t x = lane; x < n; x += 32u) d[x] = s_comp[s_conv[g[-(int)x]]];
            } else if (kind == K_CONV) {
                const uint8_t* g = v.genome + job.src;
                for (uint32_t x = lane; x < n; x += 32u) d[x] = s_conv[g[x]];
            } else if (kind == K_RAND || kind == K_RANDL) {
                for (uint32_t x = lane; x < n; x += 32u) d[x] = payload_at(v, kind, job.src, x, k.gid);
            } else {
                const uint8_t* g = v.lit + job.src;
                for (uint32_t x = lane; x < n; x += 32u) d[x] = g[x];
            }
        }
        __syncthreads();
        // ---- S3: insert line breaks, write the file image
        // line / column of a thread's groups advance by a constant per iteration: one division per thread
        const int g_first = (int)((f_lo - g0 + 15) >> 4);                 // first full group
        const int g_end = (int)((f_hi - g0) >> 4);                        // one past the last full group
        if (bpl >= 16u && g_end > g_first) {
            const uint32_t step_q = 16u * SPLICE_THREADS;
            const uint32_t step_line = step_q / w1, step_col = step_q - step_line * w1;
            int gi = g_first + tid;
            uint32_t q0 = (uint32_t)(g0 - k.body_off) + ((uint32_t)gi << 4);
            uint32_t line = q0 / w1, col = q0 - line * w1;
            uint8_t* out = fasta + g0 + ((int64_t)gi << 4);
            for (; gi < g_end; gi += SPLICE_THREADS) {
                const uint32_t j = bpl - col;                             // lane of the line break (if < 16)
                const uint32_t so = (q0 - line) - b_lo;                   // tile offset of the group's first base
                const uint32_t* w = reinterpret_cast<const uint32_t*>(tile + (so & ~3u));
                const uint32_t bs = (so & 3u) * 8u;
                const uint32_t u0 = w[0], u1 = w[1], u2 = w[2], u3 = w[3], u4 = w[4];
                uint4 y = make_uint4(__funnelshift_r(u0, u1, bs), __funnelshift_r(u1, u2, bs), __funnelshift_r(u2, u3, bs),
                                     __funnelshift_r(u3, u4, bs));
                if (j < 16u) {
                    // one PRMT per word: word w = prmt(x_w, other, sel) with
                    //   w <  jw : sel 0x3210 (untouched)
                    //   w == jw : other = '\n', byte t becomes '\n', bytes above it take x_w[t..]
                    //   w >  jw : other = x_{w-1}, sel 0x2107 (shifted up by one byte)
                    const uint32_t jw = j >> 2, t = j & 3u;
                    const uint32_t selnl = (uint32_t)(0x4210241021402104ull >> (16u * t)) & 0xFFFFu;
                    const uint32_t x0 = y.x, x1 = y.y, x2 = y.z, x3 = y.w;
                    y.x = __byte_perm(x0, 0x0Au, jw == 0u ? selnl : 0x3210u);
                    y.y = __byte_perm(x1, jw == 1u ? 0x0Au : x0, jw > 1u ? 0x3210u : (jw == 1u ? selnl : 0x2107u));
                    y.z = __byte_perm(x2, jw == 2u ? 0x0Au : x1, jw > 2u ? 0x3210u : (jw == 2u ? selnl : 0x2107u));
                    y.w = __byte_perm(x3, jw == 3u ? 0x0Au : x2, jw == 3u ? selnl : 0x2107u);
                }
                __stcs(reinterpret_cast<uint4*>(out), y);
                out += step_q;
                q0 += step_q;
                line += step_line; col += step_col;
                if (col >= w1) { col -= w1; ++line; }
            }
        }
        // edge bytes of the piece (and everything when lines are shorter than a group)
        {
            const int64_t e0 = bpl >= 16u ? g0 + ((int64_t)g_first << 4) : f_lo;   // [f_lo, e0) and [e1, f_hi) go byte-wise
            const int64_t e1 = bpl >= 16u ? (g_end > g_first ? g0 + ((int64_t)g_end << 4) : e0) : f_lo;
            const int64_t n_head = (e0 < f_hi ? e0 : f_hi) - f_lo;
            const int64_t n_tail = f_hi - (e1 > f_lo ? e1 : f_lo);
            for (int64_t y = tid; y < n_head + (n_tail > 0 ? n_tail : 0); y += SPLICE_THREADS) {
                const int64_t x = y < n_head ? f_lo + y : e1 + (y - n_head);
                if (x >= f_hi) continue;
                const uint32_t q = (uint32_t)(x - k.body_off);
                const uint32_t ln = q / w1;
                fasta[x] = (q - ln * w1 == bpl) ? (uint8_t)'\n' : tile[(q - ln) - b_lo];
            }
        }
    } else {
        // ---- fallback for tiles with more runs than the staging lists hold: generic per-byte path
        if (tid == 0) sc = contigs[k.cidx];
        __syncthreads();
        for (int gi = tid; gi < ngroups; gi += SPLICE_THREADS) {
            const int64_t g = g0 + ((int64_t)gi << 4);
            const int64_t a = g < f_lo ? f_lo : g;
            const int64_t b = g + 16 > f_hi ? f_hi : g + 16;
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            group_slow(v, sc, (uint32_t)(a - k.body_off), (int)(b - a), (int)(a - g), w);
            for (int64_t x = a; x < b; ++x) {
                const int ln = (int)(x - g);
                fasta[x] = (uint8_t)(w[ln >> 2] >> (8 * (ln & 3)));
            }
        }
    }
}

// ">header\n" of every contig and the "\n" that closes a partial last line
// (fasta_writer.py:40-47).
// Only bytes inside the file window [w_lo, w_hi) are written (ms_apply_window: another GPU owns the rest).
__global__ void k_headers(const Contig* contigs, int32_t n_contigs, const uint8_t* headers, uint8_t* fasta, int64_t w_lo, int64_t w_hi) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_contigs) return;
    const Contig& k = contigs[c];
    const int64_t h0 = k.hdr_off;
    if (h0 + k.hdr_len + 2 > w_lo && h0 < w_hi) {
        auto put = [&](int64_t x, uint8_t ch) { if (x >= w_lo && x < w_hi) fasta[x] = ch; };
        put(h0, '>');
        for (int i = 0; i < k.hdr_len; ++i) put(h0 + 1 + i, headers[k.hdr_src + i]);
        put(h0 + 1 + k.hdr_len, '\n');
    }
    const int64_t s = k.body_off + k.body_bytes;
    if (k.sep && s >= w_lo && s < w_hi) fasta[s] = '\n';
}

// ---- K7: VCF lines -----------------------------------------------------------------
// One CTA formats 256 consecutive records.  Their lines are contiguous in the output,
// so they are assembled in shared memory (placed at the same offset mod 16 as the
// destination) and written out with aligned 16-byte stores; a CTA whose lines exceed
// the staging buffer (long REF/ALT strings) writes straight to global memory.
//
// Emission is data driven: every record type runs the same instruction stream over a
// table of up to four sequence segments (REF, ALT1..3), so a warp does not serialise
// over the type switch of vcf_emit(); segments longer than one byte are queued as
// copy jobs and moved by whole warps afterwards (profiles/r1b: the per-byte REF/ALT
// loops ran on 1.5 lanes and were half of all instructions).
constexpr int VCF_THREADS = 256;
constexpr int VCF_SMEM = 13 * 1024;
#ifndef MS_VCF_INLINE
#define MS_VCF_INLINE 3
#endif
constexpr uint32_t VCF_INLINE_MAX = MS_VCF_INLINE;   // REF / ALT pieces up to this long are written by the record's own thread
constexpr int VCF_MAX_JOBS = 192;
enum SegMode : uint32_t { SM_IMM = 0, SM_RAW = 1, SM_CONV = 2, SM_RC = 3, SM_LIT = 4, SM_RAND = 5, SM_RANDL = 6 };   // RAND: src = cached 2-bit bases (<= 32); RANDL: src = gid << 32 | pos
struct Seg { int64_t src; uint32_t len; uint32_t mode; };
struct CopyJob { int64_t src; uint32_t dst; uint32_t len_mode; };   // len | mode << 29

__device__ __forceinline__ uint8_t seg_byte(const VcfView& v, uint32_t mode, int64_t src, uint32_t len, uint32_t i) {
    switch (mode) {
        case SM_IMM:  return (uint8_t)src;
        case SM_RAW:  return v.genome[src + i];
        case SM_CONV: return v.conv[v.genome[src + i]];
        case SM_RC:   return v.comp[v.conv[v.genome[src + (int64_t)(len - 1 - i)]]];
        case SM_RAND: return cached_insert_base(src, i);
        case SM_RANDL: return rand_base_ool(v.seed, (uint32_t)((uint64_t)src >> 32), (uint32_t)src, i);
        default:      return v.lit[src + i];
    }
}

__device__ __forceinline__ uint8_t* put_u32(uint8_t* p, uint32_t v) {
    const uint32_t n = ndigits(v);
    uint8_t* e = p + n;
    uint8_t* q = e;
    while (v >= 100u) {   // two digits per division
        const uint32_t d = v / 100u, r = v - d * 100u, t = (r * 205u) >> 11;   // t = r / 10 for r < 100
        *--q = (uint8_t)('0' + (r - t * 10u));
        *--q = (uint8_t)('0' + t);
        v = d;
    }
    if (v >= 10u) { const uint32_t t = (v * 205u) >> 11; *--q = (uint8_t)('0' + (v - t * 10u)); *--q = (uint8_t)('0' + t); }
    else *--q = (uint8_t)('0' + v);
    return e;
}

__device__ __forceinline__ uint8_t* put_lit(uint8_t* p, const char* t, int n) {
    for (int i = 0; i < n; ++i) p[i] = (uint8_t)t[i];
    return p + n;
}

// Segment table of one record: mutator.py:334-421 (REF/ALT per type).
__device__ __forceinline__ void vcf_segments(const VcfView& v, const Contig& c, const Rec& r, Seg sg[4], uint32_t& pos1, uint32_t& end,
                                             uint32_t& svlen, uint32_t& svt) {
    const int64_t g0 = c.goff;
    const uint32_t p = r.pos;
    const Seg none{0, 0u, SM_IMM};
    sg[0] = sg[1] = sg[2] = sg[3] = none;
    const uint32_t pmode = r.kind == K_LIT ? SM_LIT : r.kind == K_RAW ? SM_RAW : r.kind == K_CONV ? SM_CONV
                         : r.kind == K_RAND ? (r.prod <= 32u ? SM_RAND : SM_RANDL) : SM_RC;
    switch (r.type) {
        case T_SN:
            pos1 = p + 1u; end = 0u; svlen = 0u; svt = 0u;
            sg[0] = Seg{(int64_t)r.ref, 1u, SM_IMM}; sg[1] = Seg{(int64_t)r.alt, 1u, SM_IMM};
            break;
        case T_IN: case T_TLI: {
            pos1 = p > 0u ? p : 1u; end = pos1; svlen = r.prod; svt = r.type == T_IN ? 1u : 6u;
            const Seg anchor{g0 + (p > 0u ? (int64_t)p - 1 : 0), 1u, SM_CONV};
            const Seg pay{pmode == SM_RANDL ? (int64_t)(((uint64_t)c.gid << 32) | p) : r.src, r.prod, pmode};
            sg[0] = anchor;
            if (p > 0u) { sg[1] = anchor; sg[2] = pay; } else { sg[1] = pay; sg[2] = anchor; }
        } break;
        case T_DE: case T_TL: {
            pos1 = p > 0u ? p : 1u; end = p > 0u ? p + r.cons : r.cons + 1u; svlen = r.cons; svt = r.type == T_DE ? 2u : 5u;
            if (p > 0u) {
                sg[0] = Seg{g0 + (int64_t)p - 1, r.cons + 1u, SM_CONV};
                sg[1] = Seg{g0 + (int64_t)p - 1, 1u, SM_CONV};
            } else {
                uint32_t rl = r.cons + 1u;
                if ((int64_t)rl > c.len) rl = (uint32_t)c.len;
                sg[0] = Seg{g0, rl, SM_CONV};
                sg[1] = Seg{g0 + (int64_t)rl - 1, 1u, SM_CONV};
            }
        } break;
        case T_IV:
            pos1 = p + 1u; end = p + r.cons; svlen = 0u; svt = 3u;
            sg[0] = Seg{g0 + (int64_t)p, r.cons, SM_CONV}; sg[1] = Seg{g0 + (int64_t)p, r.cons, SM_RC};
            break;
        default:  // T_DU
            pos1 = p + 1u; end = p + r.prod; svlen = r.prod; svt = 4u;
            sg[0] = sg[1] = sg[2] = Seg{g0 + (int64_t)p, r.prod, SM_RAW};
            break;
    }
}

template <bool STAGED>
__device__ __forceinline__ void vcf_emit_uniform(const VcfView& v, const Contig& c, const Rec& r, uint8_t* line0, uint8_t* p,
                                                 CopyJob* jobs, int* n_jobs) {
    Seg sg[4];
    uint32_t pos1, end, svlen, svt;
    vcf_segments(v, c, r, sg, pos1, end, svlen, svt);
    for (int i = 0; i < c.name_len; ++i) p[i] = v.names[c.name_src + i];
    p += c.name_len;
    *p++ = '\t';
    p = put_u32(p, pos1);
    p = put_lit(p, "\t.\t", 3);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (q == 1) *p++ = '\t';
        const Seg g = sg[q];
        if (g.len <= VCF_INLINE_MAX) {
            for (uint32_t i = 0; i < g.len; ++i) *p++ = seg_byte(v, g.mode, g.src, g.len, i);
        } else {
            const int slot = atomicAdd(n_jobs, 1);
            if (slot < VCF_MAX_JOBS) jobs[slot] = CopyJob{g.src, (uint32_t)(p - line0), g.len | (g.mode << 29)};
            else for (uint32_t i = 0; i < g.len; ++i) p[i] = seg_byte(v, g.mode, g.src, g.len, i);   // queue full (never at sane densities)
            p += g.len;
        }
    }
    p = put_lit(p, "\t.\t.\t", 5);
    if (svt == 0u) {
        *p++ = '.';
    } else {
        const char* names = "INS\0\0\0\0\0DEL\0\0\0\0\0INV\0\0\0\0\0DUP\0\0\0\0\0DEL:ME\0\0INS:ME\0\0";
        const char* nm = names + 8 * (svt - 1u);
        p = put_lit(p, "SVTYPE=", 7);
        const int nn = svt >= 5u ? 6 : 3;
        p = put_lit(p, nm, nn);
        p = put_lit(p, ";END=", 5);
        p = put_u32(p, end);
        p = put_lit(p, ";SVLEN=", 7);
        p = put_u32(p, svlen);
    }
    put_lit(p, "\tGT\t1\n", 6);
}

__global__ void __launch_bounds__(VCF_THREADS, 8)
k_vcf_write(VcfView v, const Rec* recs, int64_t rec_lo, int64_t n_recs, const Contig* contigs, const Tables* tables, const int64_t* V,
            uint8_t* vcf) {
    __shared__ uint8_t s_conv[256], s_comp[256];
    __shared__ int n_jobs, n_sv;
    __shared__ uint8_t sv_list[VCF_THREADS];
    __shared__ CopyJob jobs[VCF_MAX_JOBS];
    extern __shared__ __align__(16) uint8_t buf[];
    __shared__ __align__(16) Rec s_rec[VCF_THREADS];          // this CTA's records and line offsets, brought in by two
    __shared__ __align__(16) int64_t s_V[VCF_THREADS + 2];    // TMA bulk copies issued before anything else
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x;
    // records [rec_lo, n_recs); CTAs start at an even record so that the TMA source of the offsets is 16-byte aligned
    const int64_t i0 = (rec_lo & ~(int64_t)1) + (int64_t)blockIdx.x * VCF_THREADS;
    const int64_t i1 = i0 + VCF_THREADS < n_recs ? i0 + VCF_THREADS : n_recs;
    const int skip = i0 < rec_lo ? 1 : 0;     // record i0 belongs to an earlier launch
    if (tid == 0) {
        n_jobs = 0; n_sv = 0;
        mbar_init(&bar, 1u);
        const uint32_t nr = (uint32_t)(i1 - i0) * (uint32_t)sizeof(Rec);
        const uint32_t nv = ((uint32_t)(i1 - i0 + 1) * 8u + 15u) & ~15u;     // the offsets array has slack behind V[n_recs]
        tma_load_1d(s_rec, recs + i0, nr, &bar);
        tma_load_1d(s_V, V + i0, nv, &bar);
        mbar_arrive_expect_tx(&bar, nr + nv);
    }
    s_conv[tid] = tables->conv[tid];
    s_comp[tid] = tables->comp[tid];
    v.conv = s_conv; v.comp = s_comp;
    if (tid < 32) mbar_wait(&bar, 0u);
    __syncthreads();
    const int64_t base = s_V[skip], end = s_V[i1 - i0];
    const uint32_t shift = (uint32_t)(base & 15);
    const bool staged = (end - base) + shift <= VCF_SMEM;
    uint8_t* line0 = staged ? buf + shift : vcf + base;   // byte 0 of this CTA's lines
    const int64_t i = i0 + tid;
    // pass 1: SNP lines (three quarters of all records) in lock step; everything else is queued
    bool is_sv = false;
    if (i < i1 && tid >= skip) {
        const int64_t a = s_V[tid], b = s_V[tid + 1];
        if (b > a) {
            const uint4 hi = reinterpret_cast<const uint4*>(s_rec + tid)[1];   // src, kind/type/ref/alt, contig
            const uint32_t type = (hi.z >> 8) & 0xffu;
            if (type == T_SN) {
                const uint32_t pos = s_rec[tid].pos;
                const Contig& c = contigs[hi.w];
                uint8_t* p = staged ? buf + shift + (a - base) : vcf + a;
                for (int q = 0; q < c.name_len; ++q) p[q] = v.names[c.name_src + q];
                p += c.name_len;
                *p++ = '\t';
                p = put_u32(p, pos + 1u);
                p[0] = '\t'; p[1] = '.'; p[2] = '\t'; p[3] = (uint8_t)(hi.z >> 16); p[4] = '\t'; p[5] = (uint8_t)(hi.z >> 24);
                p[6] = '\t'; p[7] = '.'; p[8] = '\t'; p[9] = '.'; p[10] = '\t'; p[11] = '.'; p[12] = '\t'; p[13] = 'G'; p[14] = 'T';
                p[15] = '\t'; p[16] = '1'; p[17] = '\n';
            } else {
                is_sv = true;
            }
        }
    }
    {
        const uint32_t m = __ballot_sync(0xffffffffu, is_sv);
        const int lane = tid & 31;
        if (m) {
            int b0 = 0;
            const int leader = __ffs(m) - 1;
            if (lane == leader) b0 = atomicAdd(&n_sv, __popc(m));
            b0 = __shfl_sync(0xffffffffu, b0, leader);
            if (is_sv) sv_list[b0 + __popc(m & ((1u << lane) - 1u))] = (uint8_t)tid;
        }
    }
    __syncthreads();
    // pass 2: the remaining record types, densely packed over the threads
    for (int e = tid; e < n_sv; e += VCF_THREADS) {
        const int64_t a = s_V[sv_list[e]];
        const Rec r = s_rec[sv_list[e]];
        if (staged) vcf_emit_uniform<true>(v, contigs[r.contig], r, line0, buf + shift + (a - base), jobs, &n_jobs);
        else vcf_emit_uniform<false>(v, contigs[r.contig], r, line0, vcf + a, jobs, &n_jobs);
    }
    __syncthreads();
    // pass 3: copy jobs.  Most are 4-50 bytes (a deleted stretch, a duplicated or inverted one, an insert): a quarter
    // of a warp per job, so that one pass over the dispatch code serves four of them; jobs longer than 64 bytes take a
    // whole warp, those longer than 2 KiB all warps together.
    const int nj = n_jobs < VCF_MAX_JOBS ? n_jobs : VCF_MAX_JOBS;
    const int warp = tid >> 5, lane = tid & 31;
    bool any_big = false, any_mid = false;
    {
        const int quarter = lane >> 3, ql = lane & 7;
        for (int j0 = 4 * warp; j0 < nj; j0 += 4 * (VCF_THREADS / 32)) {
            const int jb = j0 + quarter;
            if (jb >= nj) continue;
            const CopyJob job = jobs[jb];
            const uint32_t len = job.len_mode & 0x1FFFFFFFu, mode = job.len_mode >> 29;
            if (len > 64u) { if (len > 2048u) any_big = true; else any_mid = true; continue; }
            uint8_t* d = line0 + job.dst;
            if (mode == SM_RAND || mode == SM_RANDL) {
                for (uint32_t x = ql; x < len; x += 8u) d[x] = seg_byte(v, mode, job.src, len, x);
            } else {
                const bool conv = mode == SM_CONV || mode == SM_RC, rc = mode == SM_RC;
                // the lane's first source byte and its stride: forwards, or backwards from the end for a reverse complement
                const uint8_t* g = (mode == SM_LIT ? v.lit : v.genome) + job.src + (rc ? (int64_t)len - 1 - ql : (int64_t)ql);
                const int step = rc ? -8 : 8;
                uint8_t* dq = d + ql;
                for (int left = (int)len - ql; left > 0; left -= 8, g += step, dq += 8) {
                    uint32_t ch = *g;
                    if (conv) { ch = s_conv[ch]; if (rc) ch = s_comp[ch]; }
                    *dq = (uint8_t)ch;
                }
            }
        }
    }
    if (__any_sync(0xffffffffu, any_mid)) {
        for (int j0 = 4 * warp; j0 < nj; j0 += 4 * (VCF_THREADS / 32)) {
            for (int h = 0; h < 4 && j0 + h < nj; ++h) {
                const CopyJob job = jobs[j0 + h];
                const uint32_t len = job.len_mode & 0x1FFFFFFFu, mode = job.len_mode >> 29;
                if (len <= 64u || len > 2048u) continue;
                uint8_t* d = line0 + job.dst;
                for (uint32_t x = lane; x < len; x += 32u) d[x] = seg_byte(v, mode, job.src, len, x);
            }
        }
    }
    if (__syncthreads_or(any_big)) {
        for (int jb = 0; jb < nj; ++jb) {
            const CopyJob job = jobs[jb];
            const uint32_t len = job.len_mode & 0x1FFFFFFFu, mode = job.len_mode >> 29;
            if (len <= 2048u) continue;
            uint8_t* d = line0 + job.dst;
            for (uint32_t x = tid; x < len; x += VCF_THREADS) d[x] = seg_byte(v, mode, job.src, len, x);
        }
    }
    if (!staged) return;
    __syncthreads();
    // (32-bit offsets from `base`: the staged lines are at most VCF_SMEM bytes)
    const uint32_t total = (uint32_t)(end - base);
    uint32_t al = (16u - shift) & 15u;               // first 16-aligned destination offset
    if (al > total) al = total;
    const uint32_t ah = al + ((total - al) & ~15u);
    uint8_t* const out = vcf + base;
    const uint8_t* const in = buf + shift;
    if ((uint32_t)tid < al) out[tid] = in[tid];
    for (uint32_t x = al + 16u * (uint32_t)tid; x < ah; x += 16u * VCF_THREADS)
        *reinterpret_cast<uint4*>(out + x) = *reinterpret_cast<const uint4*>(in + x);
    if (ah + (uint32_t)tid < total) out[ah + tid] = in[ah + tid];
}

// delta (prod - cons) and VCF line size of every record, computed once (the scan reads 8 bytes per record)
__global__ void __launch_bounds__(256)
k_rec_sizes(VcfView v, const Rec* recs, int64_t n, const Contig* contigs, int32_t* delta, uint32_t* vsize) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Rec r = recs[i];
    delta[i] = (int32_t)r.prod - (int32_t)r.cons;
    vsize[i] = vcf_line_size(v, contigs[r.contig], r) | (r.kind != K_SNP ? VSIZE_SV : 0u);   // bit 31: the record moves bases (SvRec)
}

// Down-sweep of the plan scan, written out for its fixed types: a thread owns 8 consecutive records, reads their
// (delta, size) words with 16-byte loads, keeps them as 32-bit values (the generic k_scan_down held eight I64x3 per
// thread: 77 registers, 3 CTAs per SM, 0.55 ms for 1.1 GB) and writes S / V / N with 16-byte stores.
__global__ void __launch_bounds__(SCAN_THREADS)
k_plan_down(const int32_t* __restrict__ delta, const uint32_t* __restrict__ vsize, int64_t n, const I64x3* __restrict__ tile_prefix,
            int64_t* __restrict__ S, int64_t* __restrict__ V, uint32_t* __restrict__ N) {
    __shared__ I64x3 sm[2 * SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    static_assert(SCAN_ITEMS == 8, "two 16-byte loads per array");
    int32_t d[8];
    uint32_t vs[8];
    const bool full = base + 8 <= n;
    if (full) {
        const int4 d0 = __ldg(reinterpret_cast<const int4*>(delta + base)), d1 = __ldg(reinterpret_cast<const int4*>(delta + base) + 1);
        const uint4 v0 = __ldg(reinterpret_cast<const uint4*>(vsize + base)), v1 = __ldg(reinterpret_cast<const uint4*>(vsize + base) + 1);
        d[0] = d0.x; d[1] = d0.y; d[2] = d0.z; d[3] = d0.w; d[4] = d1.x; d[5] = d1.y; d[6] = d1.z; d[7] = d1.w;
        vs[0] = v0.x; vs[1] = v0.y; vs[2] = v0.z; vs[3] = v0.w; vs[4] = v1.x; vs[5] = v1.y; vs[6] = v1.z; vs[7] = v1.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) { const bool ok = base + j < n; d[j] = ok ? delta[base + j] : 0; vs[j] = ok ? vsize[base + j] : 0u; }
    }
    I64x3 acc{0, 0, 0};
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc.a += d[j]; acc.b += (int64_t)(vs[j] & ~VSIZE_SV); acc.c += (int64_t)(vs[j] >> 31); }
    I64x3 total;
    const I64x3 ex = block_excl_scan(acc, I64x3{0, 0, 0}, SumOp(), total, sm);
    I64x3 run = tile_prefix[blockIdx.x] + ex;
    if (full) {
        longlong2* const s2 = reinterpret_cast<longlong2*>(S + base);
        longlong2* const v2 = reinterpret_cast<longlong2*>(V + base);
        uint32_t nn[8];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            longlong2 a, b;
            a.x = run.a; b.x = run.b; nn[j] = (uint32_t)run.c;
            run.a += d[j]; run.b += (int64_t)(vs[j] & ~VSIZE_SV); run.c += (int64_t)(vs[j] >> 31);
            a.y = run.a; b.y = run.b; nn[j + 1] = (uint32_t)run.c;
            run.a += d[j + 1]; run.b += (int64_t)(vs[j + 1] & ~VSIZE_SV); run.c += (int64_t)(vs[j + 1] >> 31);
            s2[j >> 1] = a;
            v2[j >> 1] = b;
        }
        reinterpret_cast<uint4*>(N + base)[0] = make_uint4(nn[0], nn[1], nn[2], nn[3]);
        reinterpret_cast<uint4*>(N + base)[1] = make_uint4(nn[4], nn[5], nn[6], nn[7]);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (base + j < n) { S[base + j] = run.a; V[base + j] = run.b; N[base + j] = (uint32_t)run.c; }
            run.a += d[j]; run.b += (int64_t)(vs[j] & ~VSIZE_SV); run.c += (int64_t)(vs[j] >> 31);
        }
    }
}

__global__ void k_store_total3(const I64x3* total, int64_t* S_end, int64_t* V_end, uint32_t* N_end) {
    *S_end = total->a;
    *V_end = total->b;
    *N_end = (uint32_t)total->c;
}

// ---- image -> bases (chained RMT -> IT without the file round trip) ---------------------------------------------
// new_off[c] = index of contig c's first base in the new genome; 16 bases per thread.
__global__ void __launch_bounds__(256)
k_strip_image(const uint8_t* image, const Contig* contigs, int32_t n_contigs, const int64_t* new_off, int64_t total, uint8_t* out) {
    const int64_t g0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (g0 >= total) return;
    int lo = 0, hi = n_contigs;   // last c with new_off[c] <= g0
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (new_off[mid] <= g0) lo = mid; else hi = mid; }
    int c = lo;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    for (int t = 0; t < 16 && g0 + t < total; ++t) {
        const int64_t g = g0 + t;
        while (c + 1 < n_contigs && new_off[c + 1] <= g) ++c;
        const Contig& k = contigs[c];
        const int64_t b = g - new_off[c];
        const uint8_t ch = image[k.body_off + b + b / k.bpl];
        w[t >> 2] |= (uint32_t)ch << (8 * (t & 3));
    }
    if (g0 + 16 <= total) *reinterpret_cast<uint4*>(out + g0) = make_uint4(w[0], w[1], w[2], w[3]);
    else for (int t = 0; g0 + t < total; ++t) out[g0 + t] = (uint8_t)(w[t >> 2] >> (8 * (t & 3)));
}

int adopt_output(ms_ctx* c) {
    if (c->n_contigs <= 0 || !c->fasta.p || c->fasta_bytes <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_genome_adopt_output: no applied output");
    cudaStream_t st = c->stream;
    MS_CUDA(c, cudaMemcpyAsync(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    std::vector<int64_t> off((size_t)c->n_contigs + 1);
    int64_t total = 0;
    for (int i = 0; i < c->n_contigs; ++i) { off[i] = total; total += c->h_contigs[i].out_len; }
    off[c->n_contigs] = total;
    MS_CUDA(c, c->scan_tmp2.ensure((size_t)(c->n_contigs + 1) * 8));
    MS_CUDA(c, cudaMemcpyAsync(c->scan_tmp2.p, off.data(), (size_t)(c->n_contigs + 1) * 8, cudaMemcpyHostToDevice, st));
    DevBuf fresh;
    MS_CUDA(c, fresh.ensure((size_t)total + 64 + (size_t)c->foreign_cap + 64));
    if (total > 0) {
        k_strip_image<<<(unsigned)ceil_div(ceil_div(total, 16), 256), 256, 0, st>>>(c->fasta.as<uint8_t>(), c->contigs.as<Contig>(), c->n_contigs,
                                                                                    c->scan_tmp2.as<int64_t>(), total, fresh.as<uint8_t>());
        MS_LAUNCH_CHECK(c);
    }
    MS_CUDA(c, cudaMemsetAsync(fresh.as<uint8_t>() + total, 'N', 64, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    c->genome.release();
    c->genome = fresh;
    for (int i = 0; i < c->n_contigs; ++i) {
        Contig& k = c->h_contigs[i];
        const int64_t L = k.out_len;
        if (L > 0 && L < k.bpl) k.bpl = (int32_t)L;        // pyfaidx lenc of a record shorter than one line
        k.goff = off[i]; k.len = L; k.out_len = L;
        k.rec_lo = k.rec_hi = 0;
    }
    c->total_bases = total;
    MS_CUDA(c, cudaMemcpyAsync(c->contigs.p, c->h_contigs.data(), sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyHostToDevice, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    c->n_recs = 0; c->lit_bytes = 0; c->n_ranges = 0; c->sizes_valid = false; c->counts_valid = false;
    c->fasta_bytes = 0; c->vcf_bytes = 0;
    chain_invalidate(c);
    genotype_clear(c);
    return MS_OK;
}

// ---- host orchestration --------------------------------------------------------------
// plan: per-record output offsets (S) and VCF offsets (V), contig layout, output buffers.
// vcf_sizes = false (streamed run: bases not resident yet) plans the FASTA only; vcf_stage() sizes the VCF later.
static int plan_stage(ms_ctx* c, bool vcf_sizes) {
    const int64_t M = c->n_recs;
    Contig* d_contigs = c->contigs.as<Contig>();
    Totals* d_tot = c->totals.as<Totals>();
    cudaStream_t st = c->stream;

    chain_invalidate(c);
    stage_begin(c, ST_PLAN);
    MS_CUDA(c, cudaMemsetAsync(d_tot, 0, sizeof(Totals), st));
    MS_CUDA(c, c->svec.ensure((size_t)(M + 1) * sizeof(int64_t)));
    MS_CUDA(c, c->vcf_off.ensure((size_t)(M + 1) * sizeof(int64_t)));
    MS_CUDA(c, c->nvec.ensure((size_t)(M + 1) * sizeof(uint32_t)));
    MS_CUDA(c, c->piece_lo.ensure((size_t)(c->n_contigs + 1) * sizeof(int64_t)));
    MS_CUDA(c, c->recs.ensure(32));  // M == 0: keep pointers valid
    Rec* d_recs = c->recs.as<Rec>();
    int64_t* S = c->svec.as<int64_t>();
    int64_t* V = c->vcf_off.as<int64_t>();
    uint32_t* N = c->nvec.as<uint32_t>();

    k_rec_bounds<<<(unsigned)ceil_div(c->n_contigs + 1, 128), 128, 0, st>>>(d_recs, M, d_contigs, c->n_contigs);
    MS_LAUNCH_CHECK(c);

    const Tables* d_tab = c->tables.as<Tables>();
    VcfView vv{c->genome.as<uint8_t>(), c->lit.as<uint8_t>(), c->names.as<uint8_t>(), d_tab->conv, d_tab->comp, c->seed_last};
    {
        int32_t* d_delta;
        uint32_t* d_vsize;
        if (c->sizes_valid) {   // ms_sample already produced them while building the records
            d_delta = c->keep.as<int32_t>();
            d_vsize = c->cand_val.as<uint32_t>();
        } else {
            MS_CUDA(c, c->lvec.ensure((size_t)(M + 1) * 4));
            MS_CUDA(c, c->vvec.ensure((size_t)(M + 1) * 4));
            d_delta = c->lvec.as<int32_t>();
            d_vsize = c->vvec.as<uint32_t>();
        }
        if (M > 0 && !c->sizes_valid) {
            if (!vcf_sizes) MS_FAIL(c, MS_ERR_INTERNAL, "plan without bases needs sizes from the sampler");
            k_rec_sizes<<<(unsigned)ceil_div(M, 256), 256, 0, st>>>(vv, d_recs, M, d_contigs, d_delta, d_vsize);
            MS_LAUNCH_CHECK(c);
        }
        // one pass: output shift (S), VCF offset (V) and SvRec-stream slot (N) of every record
        auto in = [=] __device__(int64_t i) -> I64x3 {      // 8 bytes per record: the records themselves are not touched
            const uint32_t vs = d_vsize[i];
            return I64x3{(int64_t)d_delta[i], (int64_t)(vs & ~VSIZE_SV), (int64_t)(vs >> 31)};
        };
        I64x3* tile_prefix = nullptr;
        int64_t nt = 0;
        MS_CUDA(c, (scan_tile_sums<I64x3>(c, in, M, I64x3{0, 0, 0}, SumOp(), c->scan_tmp, &tile_prefix, &nt)));
        if (nt > 0) {
            k_plan_down<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(d_delta, d_vsize, M, tile_prefix, S, V, N);
            MS_LAUNCH_CHECK(c);
        }
        I64x3* d_total = tile_prefix + nt;
        k_store_total3<<<1, 1, 0, st>>>(d_total, S + M, V + M, N + M);
        MS_LAUNCH_CHECK(c);
    }
    if (c->n_contigs <= 2048) {
        k_contig_layout<<<1, SCAN_THREADS, 0, st>>>(d_contigs, c->n_contigs, S, c->piece_lo.as<int64_t>(), (int64_t)c->tile_bytes, d_tot, M, V, N);
        MS_LAUNCH_CHECK(c);
    } else {
        int rc = layout_by_scan(c, d_contigs, S, V, N, M, d_tot);
        if (rc) return rc;
    }
    MS_CUDA(c, cudaMemcpyAsync(c->h_totals, d_tot, sizeof(Totals), cudaMemcpyDeviceToHost, st));
    stage_end(c, ST_PLAN);
    MS_CUDA(c, cudaStreamSynchronize(st));
    Totals t = *c->h_totals;
    if (t.error) MS_FAIL(c, (int)t.error, "ms_apply: layout failed (code %lld at contig %lld)", (long long)t.error, (long long)t.error_arg);
    c->fasta_bytes = t.fasta_bytes; c->vcf_bytes = t.vcf_bytes; c->n_sv = t.n_blk; c->n_pieces = t.n_pieces;

    MS_CUDA(c, c->fasta.ensure((size_t)t.fasta_bytes + 64));
    MS_CUDA(c, c->vcf.ensure((size_t)t.vcf_bytes + 64));
    MS_CUDA(c, c->piece_desc.ensure((size_t)(t.n_pieces + 1) * sizeof(PieceDesc)));
    MS_CUDA(c, c->sv_stream.ensure((size_t)(c->n_sv + 4) * sizeof(SvRec)));
    MS_CUDA(c, c->snp_stream.ensure((size_t)(M - c->n_sv + 4) * sizeof(Snp8)));
    return MS_OK;
}

// index: record output positions, the SvRec / Snp8 streams, per-tile descriptors
static int index_stage(ms_ctx* c) {
    const int64_t M = c->n_recs;
    Contig* d_contigs = c->contigs.as<Contig>();
    Rec* d_recs = c->recs.as<Rec>();
    Totals* d_tot = c->totals.as<Totals>();
    const int64_t* S = c->svec.as<int64_t>();
    const uint32_t* N = c->nvec.as<uint32_t>();
    cudaStream_t st = c->stream;
    stage_begin(c, ST_INDEX);
    if (M > 0) {
        k_rec_out<<<(unsigned)std::min<int64_t>(ceil_div(M, 256), (int64_t)NUM_SMS_B200 * 32), 256, 0, st>>>(d_recs, M, d_contigs, S, N, c->sv_stream.as<SvRec>(), c->snp_stream.as<Snp8>(), d_tot);
        MS_LAUNCH_CHECK(c);
    }
    if (c->n_pieces > 0) {
        k_piece_desc<<<(unsigned)ceil_div(c->n_pieces, 256), 256, 0, st>>>(d_contigs, c->n_contigs, c->piece_lo.as<int64_t>(), c->n_pieces,
                                                                          c->sv_stream.as<SvRec>(), c->snp_stream.as<Snp8>(), N, d_tot,
                                                                          c->piece_desc.as<PieceDesc>());
        MS_LAUNCH_CHECK(c);
    }
    c->rec_out_valid = false;
    stage_end(c, ST_INDEX);
    return MS_OK;
}

// splice: tiles [piece_lo, piece_lo + n_pieces) and the headers of contigs [ctg_lo, ctg_lo + n_ctg)
static int splice_launch(ms_ctx* c, int64_t piece_lo, int64_t n_pieces, int32_t ctg_lo, int32_t n_ctg, int64_t w_lo = 0,
                         int64_t w_hi = INT64_MAX) {
    if (c->tile_bytes != TL_TILE) MS_FAIL(c, MS_ERR_INTERNAL, "tile_bytes must equal %d", TL_TILE);
    const Tables* d_tab = c->tables.as<Tables>();
    Contig* d_contigs = c->contigs.as<Contig>();
    cudaStream_t st = c->stream;
    SpliceView sv{c->genome.as<uint8_t>(), c->lit.as<uint8_t>(), c->recs.as<Rec>(), c->svec.as<int64_t>(), d_tab->conv, d_tab->comp, c->seed_last};
    sv.local_cap = (int64_t)c->genome.cap;
    if (n_pieces > 0) {
        if (!c->splice_attr_set) {   // per context: the attribute is per device, and a process may hold contexts on several
            MS_CUDA(c, cudaFuncSetAttribute(k_splice, cudaFuncAttributeMaxDynamicSharedMemorySize, SP_DYN));
            c->splice_attr_set = true;
        }
        k_splice<<<(unsigned)n_pieces, SPLICE_THREADS, SP_DYN, st>>>(sv, d_contigs, c->piece_desc.as<PieceDesc>() + piece_lo,
                                                                   c->sv_stream.as<SvRec>(), c->snp_stream.as<Snp8>(), d_tab,
                                                                   c->fasta.as<uint8_t>(), n_pieces);
        MS_LAUNCH_CHECK(c);
    }
    if (n_ctg > 0) {
        k_headers<<<(unsigned)ceil_div(n_ctg, 128), 128, 0, st>>>(d_contigs + ctg_lo, n_ctg, c->headers.as<uint8_t>(), c->fasta.as<uint8_t>(),
                                                                   w_lo, w_hi);
        MS_LAUNCH_CHECK(c);
    }
    return MS_OK;
}

// VCF lines of records [r0, r1) (V already holds their offsets)
static int vcf_launch(ms_ctx* c, int64_t r0, int64_t r1, cudaStream_t st) {
    const Tables* d_tab = c->tables.as<Tables>();
    VcfView vv{c->genome.as<uint8_t>(), c->lit.as<uint8_t>(), c->names.as<uint8_t>(), d_tab->conv, d_tab->comp, c->seed_last};
    if (r1 > r0) {
        if (!c->vcf_attr_set) {
            MS_CUDA(c, cudaFuncSetAttribute(k_vcf_write, cudaFuncAttributeMaxDynamicSharedMemorySize, VCF_SMEM + 32));
            c->vcf_attr_set = true;
        }
        k_vcf_write<<<(unsigned)ceil_div(r1 - (r0 & ~(int64_t)1), VCF_THREADS), VCF_THREADS, VCF_SMEM + 32, st>>>(
            vv, c->recs.as<Rec>(), r0, r1, c->contigs.as<Contig>(), d_tab, c->vcf_off.as<int64_t>(), c->vcf.as<uint8_t>());
        MS_LAUNCH_CHECK(c);
    }
    return MS_OK;
}

static int finish_apply(ms_ctx* c) {
    MS_CUDA(c, cudaMemcpyAsync(c->h_totals, c->totals.p, sizeof(Totals), cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    const Totals t = *c->h_totals;
    if (t.error) MS_FAIL(c, (int)t.error, "ms_apply: records invalid (code %lld at record %lld): overlapping or out of bounds",
                         (long long)t.error, (long long)t.error_arg);
    c->last_totals.fasta_bytes = c->fasta_bytes;
    c->last_totals.vcf_bytes = c->vcf_bytes;
    c->last_totals.n_recs = c->n_recs;
    for (int k = 0; k < 8; ++k) c->last_totals.counts[k] = t.counts[k];     // counted by k_rec_out
    c->counts_valid = true;
    return MS_OK;
}

int apply_pipeline(ms_ctx* c) {
    if (c->n_contigs <= 0 || !c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_apply: no genome resident");
    int rc = plan_stage(c, true);
    if (rc) return rc;
    if ((rc = index_stage(c))) return rc;
    stage_begin(c, ST_SPLICE);
    if ((rc = splice_launch(c, 0, c->n_pieces, 0, c->n_contigs))) return rc;
    stage_end(c, ST_SPLICE);
    stage_begin(c, ST_VCF);
    if ((rc = vcf_launch(c, 0, c->n_recs, c->stream))) return rc;
    stage_end(c, ST_VCF);
    if ((rc = finish_apply(c))) return rc;
    c->chain_ready = true;
    c->apply_full = true;
    return MS_OK;
}

// ---- tile-sharded apply: one genome, several GPUs ------------------------------------------------------------------
// Every rank holds the whole genome and the whole record table (sampling is keyed by position, so all ranks draw the
// same table); the layout of the output is therefore identical everywhere and the work of producing it can be cut at
// ANY tile / record boundary: part p of n writes tiles [T*p/n, T*(p+1)/n) of the FASTA image and the VCF lines of
// records [M*p/n, M*(p+1)/n).  This is how a contig larger than one GPU's share (the reference's own benchmark is
// one 1 Gbp contig, README.md:441) is spread over the box: chunks are cut at 16 KiB tile boundaries of the output;
// the rejection carry, the delta prefix and TLI sources that cross a cut need no exchange because the (cheap)
// candidate table is replicated and only the byte-moving stages are sharded.
int apply_window(ms_ctx* c, int part, int n_parts, int64_t* win) {
    if (c->n_contigs <= 0 || !c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_apply_window: no genome resident");
    if (n_parts < 1 || part < 0 || part >= n_parts) MS_FAIL(c, MS_ERR_ARG, "ms_apply_window: part %d of %d", part, n_parts);
    int rc = plan_stage(c, true);
    if (rc) return rc;
    if ((rc = index_stage(c))) return rc;
    MS_CUDA(c, cudaMemcpyAsync(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    const int64_t tile = c->tile_bytes;
    const int64_t n_tiles = ceil_div(c->fasta_bytes, tile);
    const int64_t t_lo = n_tiles * part / n_parts, t_hi = n_tiles * (part + 1) / n_parts;
    const int64_t w_lo = t_lo * tile, w_hi = std::min(t_hi * tile, c->fasta_bytes);
    // pieces are ordered by (contig, tile) = by file offset: first piece whose tile is >= T
    auto first_piece = [&](int64_t T) -> int64_t {
        for (int i = 0; i < c->n_contigs; ++i) {
            const Contig& k = c->h_contigs[i];
            if (k.body_bytes <= 0) continue;
            const int64_t ft = k.body_off / tile, lt = (k.body_off + k.body_bytes - 1) / tile;
            if (lt >= T) return k.piece_lo + std::max<int64_t>(0, T - ft);
        }
        return c->n_pieces;
    };
    const int64_t p_lo = first_piece(t_lo), p_hi = first_piece(t_hi);
    const int64_t M = c->n_recs;
    const int64_t r_lo = M * part / n_parts, r_hi = M * (part + 1) / n_parts;
    stage_begin(c, ST_SPLICE);
    if ((rc = splice_launch(c, p_lo, p_hi - p_lo, 0, c->n_contigs, w_lo, w_hi))) return rc;
    stage_end(c, ST_SPLICE);
    stage_begin(c, ST_VCF);
    if ((rc = vcf_launch(c, r_lo, r_hi, c->stream))) return rc;
    stage_end(c, ST_VCF);
    int64_t v[2] = {0, 0};
    if (M > 0) {
        MS_CUDA(c, cudaMemcpyAsync(&v[0], c->vcf_off.as<int64_t>() + r_lo, 8, cudaMemcpyDeviceToHost, c->stream));
        MS_CUDA(c, cudaMemcpyAsync(&v[1], c->vcf_off.as<int64_t>() + r_hi, 8, cudaMemcpyDeviceToHost, c->stream));
    }
    if ((rc = finish_apply(c))) return rc;
    c->chain_ready = true;
    win[0] = c->fasta_bytes; win[1] = c->vcf_bytes; win[2] = w_lo; win[3] = w_hi; win[4] = v[0]; win[5] = v[1];
    return MS_OK;
}

// ---- streamed run: host genome in, host FASTA + VCF out, copies overlapped with the kernels --------------------
// upper-case genome bytes [lo, hi) (util.py:87 sequence_always_upper); byte-exact at both ends so that neighbouring
// groups never touch each other's bytes
__global__ void __launch_bounds__(256) k_upper_range(uint8_t* g, int64_t lo, int64_t hi) {
    const int64_t w = (lo >> 4) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t b0 = w << 4;
    if (b0 >= hi) return;
    if (b0 >= lo && b0 + 16 <= hi) {
        uint4 v = *reinterpret_cast<uint4*>(g + b0);
        uint32_t* x = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t lo7 = x[k] & 0x7F7F7F7Fu;
            const uint32_t is_lower = ((lo7 + 0x1F1F1F1Fu) & ~(lo7 + 0x05050505u) & ~x[k]) & 0x80808080u;
            x[k] &= ~(is_lower >> 2);
        }
        *reinterpret_cast<uint4*>(g + b0) = v;
    } else {
        for (int64_t b = b0 > lo ? b0 : lo; b < b0 + 16 && b < hi; ++b) {
            const uint8_t ch = g[b];
            if (ch >= 'a' && ch <= 'z') g[b] = ch - 32;
        }
    }
}

// ref/alt of the SNP records [lo, hi): the part of record building that needs the bases (mutator.py:429-455)
__global__ void __launch_bounds__(256)
k_snp_fill(Rec* recs, int64_t lo, int64_t hi, const Contig* contigs, const uint8_t* genome, const Tables* tab, Seed seed, double p_ti,
           Snp8* snp, const uint32_t* N) {
    const int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    const uint32_t kind_type = reinterpret_cast<const uint32_t*>(recs + i)[6];   // kind | type<<8 | ref<<16 | alt<<24
    if ((kind_type & 0xFFu) != K_SNP) return;
    const uint32_t pos = recs[i].pos;
    const Contig& ct = contigs[recs[i].contig];
    const uint8_t ref = tab->conv[genome[ct.goff + pos]];
    const uint8_t alt = draw_snp(seed, ct.gid, pos, ref, p_ti, tab->trans);
    reinterpret_cast<uint32_t*>(recs + i)[6] = (kind_type & 0xFFFFu) | ((uint32_t)ref << 16) | ((uint32_t)alt << 24);
    snp[i - (int64_t)N[i]].alt = (uint32_t)alt;      // the record's slot in the Snp8 stream
}

// VCF bytes written up to the end of a contig group: vend[1] = vend[0] + this group's bytes
__global__ void k_store_vend(const I64x2* total, int64_t* vend, int64_t* V_end, Totals* tot) {
    const int64_t e = vend[0] + (total ? total->b : 0);
    vend[1] = e; *V_end = e; tot->vcf_bytes = e;
}

int mutate_streamed(ms_ctx* c, uint64_t seed, const uint8_t* h_bases, uint8_t* h_fasta, int64_t fasta_cap, uint8_t* h_vcf,
                    int64_t vcf_cap, int64_t* fasta_bytes, int64_t* vcf_bytes, int64_t group_min) {
    if (c->n_contigs <= 0 || !c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_mutate_streamed: declare a genome first");
    if (c->n_ranges < 0) MS_FAIL(c, MS_ERR_STATE, "ms_mutate_streamed: set ranges first");
    if (!c->s_up) {
        MS_CUDA(c, cudaStreamCreateWithFlags(&c->s_up, cudaStreamNonBlocking));
        MS_CUDA(c, cudaStreamCreateWithFlags(&c->s_down, cudaStreamNonBlocking));
        MS_CUDA(c, cudaStreamCreateWithFlags(&c->s_vcf, cudaStreamNonBlocking));
    }
    // contig groups of >= GROUP_MIN bases: the unit of upload / splice / download
    const int64_t GROUP_MIN = group_min > 0 ? group_min : (48ll << 20);
    std::vector<int32_t> g_lo;   // first contig of each group (+ sentinel)
    {
        int64_t acc = 0;
        for (int i = 0; i < c->n_contigs; ++i) {
            if (acc == 0) g_lo.push_back(i);
            acc += c->h_contigs[i].len;
            if (acc >= GROUP_MIN) acc = 0;
        }
        g_lo.push_back(c->n_contigs);
    }
    const int G = (int)g_lo.size() - 1;
    while ((int)c->ev_up.size() < G) {
        cudaEvent_t a, b, d;
        MS_CUDA(c, cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        MS_CUDA(c, cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        MS_CUDA(c, cudaEventCreateWithFlags(&d, cudaEventDisableTiming));
        c->ev_up.push_back(a); c->ev_done.push_back(b); c->ev_sized.push_back(d);
    }
    uint8_t* d_genome = c->genome.as<uint8_t>();
    auto goff_of = [&](int32_t ctg) { return ctg < c->n_contigs ? c->h_contigs[ctg].goff : c->total_bases; };

    // uploads: queued now, run while the sampler works on the compute stream
    MS_CUDA(c, cudaEventRecord(c->ev_done[0], c->stream));          // the previous call's readers of the genome are done
    MS_CUDA(c, cudaStreamWaitEvent(c->s_up, c->ev_done[0], 0));
    for (int g = 0; g < G; ++g) {
        const int64_t lo = goff_of(g_lo[g]), hi = goff_of(g_lo[g + 1]);
        if (hi > lo) {
            MS_CUDA(c, cudaMemcpyAsync(d_genome + lo, h_bases + lo, (size_t)(hi - lo), cudaMemcpyHostToDevice, c->s_up));
            const int64_t words = ((hi + 15) >> 4) - (lo >> 4);
            k_upper_range<<<(unsigned)ceil_div(words, 256), 256, 0, c->s_up>>>(d_genome, lo, hi);
            MS_LAUNCH_CHECK(c);
        }
        MS_CUDA(c, cudaEventRecord(c->ev_up[g], c->s_up));
    }

    int rc = sample_pipeline(c, seed, true);      // positions, types, lengths, conflicts, TL links: no bases needed
    if (rc) return rc;
    if ((rc = plan_stage(c, false))) return rc;   // FASTA layout only (VCF sizes depend on bases)
    if (c->fasta_bytes > fasta_cap) MS_FAIL(c, MS_ERR_ARG, "FASTA buffer too small: need %lld bytes", (long long)c->fasta_bytes);
    if ((rc = index_stage(c))) return rc;
    // contig table with rec / piece / file offsets for the per-group launches
    MS_CUDA(c, cudaMemcpyAsync(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<int64_t> h_piece_lo((size_t)c->n_contigs + 1);
    MS_CUDA(c, cudaMemcpy(h_piece_lo.data(), c->piece_lo.p, (size_t)(c->n_contigs + 1) * 8, cudaMemcpyDeviceToHost));

    const Tables* d_tab = c->tables.as<Tables>();
    // c->vcf was sized by the plan from base-independent line sizes (an upper bound); the real offsets are computed
    // group by group as the bases arrive (a SNP or inversion with REF == ALT is not written, vcf_writer.py:123)
    const int64_t M = c->n_recs;
    MS_CUDA(c, c->vend.ensure((size_t)(G + 1) * 8));
    if ((int)c->h_vend_cap < G + 1) {
        if (c->h_vend) cudaFreeHost(c->h_vend);
        MS_CUDA(c, cudaHostAlloc(&c->h_vend, (size_t)(G + 1) * 8 * 2, cudaHostAllocDefault));
        c->h_vend_cap = 2 * (G + 1);
    }
    int64_t* d_vend = c->vend.as<int64_t>();
    MS_CUDA(c, cudaMemsetAsync(d_vend, 0, 8, c->stream));
    c->h_vend[0] = 0;
    int32_t* d_delta = c->keep.as<int32_t>();
    uint32_t* d_vsize = c->cand_val.as<uint32_t>();
    int64_t* V = c->vcf_off.as<int64_t>();
    VcfView vv{d_genome, c->lit.as<uint8_t>(), c->names.as<uint8_t>(), d_tab->conv, d_tab->comp, c->seed_last};
    std::vector<int64_t> g_r0(G), g_r1(G);

    // VCF lines of group g: wait for its sizes, then write and download its byte range
    auto flush_vcf = [&](int g) -> int {
        MS_CUDA(c, cudaEventSynchronize(c->ev_sized[g]));
        const int64_t lo = c->h_vend[g], hi = c->h_vend[g + 1];
        if (hi > vcf_cap) MS_FAIL(c, MS_ERR_ARG, "VCF buffer too small: need more than %lld bytes", (long long)vcf_cap);
        if (hi == lo) return MS_OK;
        MS_CUDA(c, cudaStreamWaitEvent(c->s_vcf, c->ev_sized[g], 0));
        int r = vcf_launch(c, g_r0[g], g_r1[g], c->s_vcf);
        if (r) return r;
        MS_CUDA(c, cudaMemcpyAsync(h_vcf + lo, c->vcf.as<uint8_t>() + lo, (size_t)(hi - lo), cudaMemcpyDeviceToHost, c->s_vcf));
        return MS_OK;
    };

    stage_begin(c, ST_SPLICE);
    for (int g = 0; g < G; ++g) {
        const int32_t c0 = g_lo[g], c1 = g_lo[g + 1];
        const int64_t r0 = c->h_contigs[c0].rec_lo, r1 = c->h_contigs[c1 - 1].rec_hi;
        g_r0[g] = r0; g_r1[g] = r1;
        MS_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_up[g], 0));
        if (r1 > r0) {
            k_snp_fill<<<(unsigned)ceil_div(r1 - r0, 256), 256, 0, c->stream>>>(c->recs.as<Rec>(), r0, r1, c->contigs.as<Contig>(), d_genome, d_tab,
                                                                             c->seed_last, c->p_ti, c->snp_stream.as<Snp8>(), c->nvec.as<uint32_t>());
            MS_LAUNCH_CHECK(c);
        }
        if ((rc = splice_launch(c, h_piece_lo[c0], h_piece_lo[c1] - h_piece_lo[c0], c0, c1 - c0))) return rc;
        MS_CUDA(c, cudaEventRecord(c->ev_done[g], c->stream));
        const int64_t f0 = c->h_contigs[c0].hdr_off, f1 = c1 < c->n_contigs ? c->h_contigs[c1].hdr_off : c->fasta_bytes;
        MS_CUDA(c, cudaStreamWaitEvent(c->s_down, c->ev_done[g], 0));
        MS_CUDA(c, cudaMemcpyAsync(h_fasta + f0, c->fasta.as<uint8_t>() + f0, (size_t)(f1 - f0), cudaMemcpyDeviceToHost, c->s_down));
        // sizes and offsets of this group's VCF lines
        I64x2* d_total = nullptr;
        if (r1 > r0) {
            k_rec_sizes<<<(unsigned)ceil_div(r1 - r0, 256), 256, 0, c->stream>>>(vv, c->recs.as<Rec>() + r0, r1 - r0, c->contigs.as<Contig>(),
                                                                              d_delta + r0, d_vsize + r0);
            MS_LAUNCH_CHECK(c);
            const int64_t* carry = d_vend + g;
            auto in = [=] __device__(int64_t i) -> I64x2 { return I64x2{0, (int64_t)(d_vsize[r0 + i] & ~VSIZE_SV)}; };
            auto out = [=] __device__(int64_t i, I64x2 ex, I64x2) { V[r0 + i] = ex.b + *carry; };
            MS_CUDA(c, (device_scan<I64x2>(c, in, out, r1 - r0, I64x2{0, 0}, SumOp(), c->scan_tmp, &d_total)));
        }
        k_store_vend<<<1, 1, 0, c->stream>>>(d_total, d_vend + g, V + r1, c->totals.as<Totals>());
        MS_LAUNCH_CHECK(c);
        MS_CUDA(c, cudaMemcpyAsync(c->h_vend + g + 1, d_vend + g + 1, 8, cudaMemcpyDeviceToHost, c->stream));
        MS_CUDA(c, cudaEventRecord(c->ev_sized[g], c->stream));
        if (g >= 1 && (rc = flush_vcf(g - 1))) return rc;
    }
    if ((rc = flush_vcf(G - 1))) return rc;
    stage_end(c, ST_SPLICE);
    c->vcf_bytes = c->h_vend[G];
    (void)M;
    rc = finish_apply(c);
    MS_CUDA(c, cudaStreamSynchronize(c->s_vcf));
    MS_CUDA(c, cudaStreamSynchronize(c->s_down));
    if (rc) return rc;
    c->sizes_valid = false;
    if (fasta_bytes) *fasta_bytes = c->fasta_bytes;
    if (vcf_bytes) *vcf_bytes = c->vcf_bytes;
    return MS_OK;
}

}  // namespace ms
