// ms_bgzf.cu — BGZF encoder for the FASTA image and the VCF body (ms_bgzf_compress).
//
// The segments of an output buffer are cut into blocks on a grid of 16 KiB cells of the uncompressed FILE (a block
// never spans two segments, i.e. two contigs), one CTA encodes one block into a member (ms_bgzf_core.h) in its own
// scratch slot, and a second kernel packs the members back to back.  Members depend only on the block's bytes.
#include <algorithm>
#include "ms_bgzf_core.h"
#include "ms_common.cuh"

namespace ms {
namespace {

using namespace bgzf;

constexpr int THREADS = 256;
constexpr int CHUNK = CELL / THREADS;     // input bytes per thread (64)
constexpr int SKEW = CHUNK + 4;           // shared-memory stride of a thread's chunk (17 words: a warp's bytes hit 32 banks)

struct Block {
    int64_t src;      // offset in the source buffer
    int32_t n;        // bytes taken from the buffer
    int32_t nl;       // 1: a '\n' follows them (the separator a partial last line gets in the assembled file)
};

// The block's m bytes are right-aligned in a virtual 16 KiB cell (left-padded with pad = CELL - m zeros): thread t
// owns cell bytes [64 t, 64 t + 64).  Leading zeros leave a CRC register that starts at 0 unchanged, so the chunks'
// raw CRCs combine in a fixed-shape tree whatever m is.
__global__ void __launch_bounds__(THREADS) k_bgzf_encode(const uint8_t* __restrict__ buf, const Block* __restrict__ blocks,
                                                         uint8_t* __restrict__ slots, int32_t* __restrict__ zsize) {
    __shared__ __align__(16) uint8_t s_in[THREADS * SKEW];
    __shared__ uint32_t s_words[WORDS];            // per-warp histograms first, then the deflate bit stream
    __shared__ BlockCode s_bc;
    __shared__ uint32_t s_crc_tab[256];
    __shared__ uint32_t s_shift[6];                // x^(8 * 64 * 2^k): appends 2^k chunks of zeros
    __shared__ uint32_t s_warp[THREADS / 32];
    __shared__ uint32_t s_crc;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const Block B = blocks[blockIdx.x];
    const int m = B.n + B.nl;
    const int pad = CELL - m;

    s_crc_tab[tid] = crc_table_entry((uint32_t)tid);
    if (tid < 6) s_shift[tid] = crc_shift_op((uint64_t)CHUNK << tid);
    for (int i = tid; i < (THREADS / 32) * 256; i += THREADS) s_words[i] = 0;
    const uint8_t* src = buf + B.src;
    for (int i = tid; i < B.n; i += THREADS) {
        const int p = pad + i;
        s_in[(p / CHUNK) * SKEW + p % CHUNK] = src[i];
    }
    if (B.nl && tid == 0) { const int p = pad + B.n; s_in[(p / CHUNK) * SKEW + p % CHUNK] = '\n'; }
    __syncthreads();

    // histogram (one sub-histogram per warp) and the raw CRC of this thread's bytes
    const int c0 = tid * CHUNK;
    const int a = max(c0, pad) - c0;               // first owned byte within the chunk
    const uint8_t* mine = s_in + tid * SKEW;
    uint32_t* hist = s_words + warp * 256;
    uint32_t raw = 0;
    for (int j = a; j < CHUNK; ++j) {
        const uint32_t v = mine[j];
        atomicAdd(&hist[v], 1u);
        raw = s_crc_tab[(raw ^ v) & 0xff] ^ (raw >> 8);
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const uint32_t other = __shfl_down_sync(0xffffffffu, raw, 1 << k);
        if ((lane & ((2 << k) - 1)) == 0) raw = gf2_mul(s_shift[k], raw) ^ other;
    }
    if (lane == 0) s_warp[warp] = raw;
    __syncthreads();
    {
        uint32_t f = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) f += s_words[w * 256 + tid];
        s_bc.freq[tid] = f;
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t acc = 0;
        for (int w = 0; w < THREADS / 32; ++w) acc = gf2_mul(s_shift[5], acc) ^ s_warp[w];
        s_crc = crc32_finish(acc, (uint64_t)m);
        plan_block(s_bc, m);
    }
    for (int i = tid; i < WORDS; i += THREADS) s_words[i] = 0;
    __syncthreads();
    const bool stored = s_bc.stored;
    int dbytes = m + 5;
    if (!stored) {
        if (tid == 0) s_warp[0] = write_dyn_header(s_bc, s_words);   // (s_warp is free again)
        uint32_t nb = 0;
        for (int j = a; j < CHUNK; ++j) nb += (uint32_t)code_len(s_bc.lit[mine[j]]);
        // exclusive scan of the bit counts over the CTA
        uint32_t inc = nb;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, k);
            if (lane >= k) inc += y;
        }
        __shared__ uint32_t s_tot[THREADS / 32];
        if (lane == 31) s_tot[warp] = inc;
        __syncthreads();
        const uint32_t hdr = s_warp[0];
        uint32_t base = hdr;
        for (int w = 0; w < warp; ++w) base += s_tot[w];
        uint32_t pos = base + inc - nb;
        // pack: 64-bit accumulator flushed as aligned 32-bit words (the first / last word may be shared)
        uint32_t wi = pos >> 5;
        int nacc = (int)(pos & 31);
        uint64_t acc = 0;
        for (int j = a; j < CHUNK; ++j) {
            const uint32_t c = s_bc.lit[mine[j]];
            acc |= (uint64_t)(c & 0xFFFFu) << nacc;
            nacc += code_len(c);
            if (nacc >= 32) { atomicOr(&s_words[wi++], (uint32_t)acc); acc >>= 32; nacc -= 32; }
        }
        if (nacc > 0) atomicOr(&s_words[wi], (uint32_t)acc);
        __syncthreads();
        if (tid == 0) {
            uint32_t end = hdr;
            for (int w = 0; w < THREADS / 32; ++w) end += s_tot[w];
            const uint32_t e = s_bc.lit[256];
            or_bits(s_words, end, e & 0xFFFFu, code_len(e));
            s_warp[1] = (end + (uint32_t)code_len(e) + 7) / 8;
        }
        __syncthreads();
        dbytes = (int)s_warp[1];
    }
    const int total = HDR + dbytes + FTR;
    uint8_t* out = slots + (int64_t)blockIdx.x * SLOT;
    const uint8_t* wb = reinterpret_cast<const uint8_t*>(s_words);
    const uint32_t crc = s_crc;
    for (int i = tid; i < total; i += THREADS) {
        uint8_t v;
        if (i < HDR) v = member_header_byte(i, total);
        else if (i < HDR + dbytes) {
            const int j = i - HDR;
            if (!stored) v = wb[j];
            else if (j < 5) v = stored_head_byte(j, m);
            else { const int p = pad + j - 5; v = s_in[(p / CHUNK) * SKEW + p % CHUNK]; }
        } else {
            const int k = i - HDR - dbytes;
            v = k < 4 ? (uint8_t)(crc >> (8 * k)) : (uint8_t)((uint32_t)m >> (8 * (k - 4)));
        }
        out[i] = v;
    }
    if (tid == 0) zsize[blockIdx.x] = total;
}

__global__ void __launch_bounds__(THREADS) k_bgzf_pack(const uint8_t* __restrict__ slots, const int32_t* __restrict__ zsize,
                                                       const int64_t* __restrict__ zoff, uint8_t* __restrict__ out) {
    const uint8_t* s = slots + (int64_t)blockIdx.x * SLOT;
    uint8_t* d = out + zoff[blockIdx.x];
    const int n = zsize[blockIdx.x];
    for (int i = threadIdx.x; i < n; i += THREADS) d[i] = s[i];
}

}  // namespace

int bgzf_compress(ms_ctx* c, int which, int32_t n_seg, const int64_t* src_off, const int64_t* nbytes, const int64_t* file_off,
                  const uint8_t* add_nl, int64_t* seg_zbytes, int64_t* total_zbytes) {
    const uint8_t* buf = which == 0 ? c->fasta.as<uint8_t>() : c->vcf.as<uint8_t>();
    const int64_t size = which == 0 ? c->fasta_bytes : c->vcf_bytes;
    std::vector<Block> blocks;
    std::vector<int32_t> seg_of;
    for (int32_t s = 0; s < n_seg; ++s) {
        const int64_t nl = add_nl && add_nl[s] ? 1 : 0;
        if (src_off[s] < 0 || nbytes[s] < 0 || file_off[s] < 0 || src_off[s] + nbytes[s] > size)
            MS_FAIL(c, MS_ERR_ARG, "ms_bgzf_compress: segment %d lies outside buffer %d", s, which);
        const int64_t L = nbytes[s] + nl;
        for (int64_t pos = 0; pos < L;) {
            const int64_t f = file_off[s] + pos;
            const int64_t take = std::min(L - pos, (f / CELL + 1) * CELL - f);
            const int64_t nb = std::max<int64_t>(0, std::min(take, nbytes[s] - pos));
            blocks.push_back(Block{src_off[s] + pos, (int32_t)nb, (int32_t)(take - nb)});
            seg_of.push_back(s);
            pos += take;
        }
    }
    const int64_t nblk = (int64_t)blocks.size();
    for (int32_t s = 0; s < n_seg; ++s) seg_zbytes[s] = 0;
    c->bgzf_bytes = 0;
    if (nblk == 0) { *total_zbytes = 0; return MS_OK; }
    if (nblk >= (1ll << 31)) MS_FAIL(c, MS_ERR_LIMIT, "ms_bgzf_compress: %lld blocks", (long long)nblk);
    MS_CUDA(c, c->bgzf_blocks.ensure(sizeof(Block) * (size_t)nblk));
    MS_CUDA(c, c->bgzf_slots.ensure((size_t)SLOT * (size_t)nblk));
    MS_CUDA(c, c->bgzf_zsize.ensure(sizeof(int32_t) * (size_t)nblk + sizeof(int64_t) * (size_t)nblk + 16));
    int32_t* d_zsize = c->bgzf_zsize.as<int32_t>();
    int64_t* d_zoff = reinterpret_cast<int64_t*>(c->bgzf_zsize.as<uint8_t>() + ((sizeof(int32_t) * (size_t)nblk + 15) & ~(size_t)15));
    MS_CUDA(c, cudaMemcpyAsync(c->bgzf_blocks.p, blocks.data(), sizeof(Block) * (size_t)nblk, cudaMemcpyHostToDevice, c->stream));
    k_bgzf_encode<<<(unsigned)nblk, THREADS, 0, c->stream>>>(buf, c->bgzf_blocks.as<Block>(), c->bgzf_slots.as<uint8_t>(), d_zsize);
    MS_LAUNCH_CHECK(c);
    std::vector<int32_t> zs((size_t)nblk);
    std::vector<int64_t> zo((size_t)nblk);
    MS_CUDA(c, cudaMemcpyAsync(zs.data(), d_zsize, sizeof(int32_t) * (size_t)nblk, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    int64_t tot = 0;
    for (int64_t b = 0; b < nblk; ++b) { zo[b] = tot; tot += zs[b]; seg_zbytes[seg_of[b]] += zs[b]; }
    MS_CUDA(c, c->bgzf.ensure((size_t)tot + 16));
    MS_CUDA(c, cudaMemcpyAsync(d_zoff, zo.data(), sizeof(int64_t) * (size_t)nblk, cudaMemcpyHostToDevice, c->stream));
    k_bgzf_pack<<<(unsigned)nblk, THREADS, 0, c->stream>>>(c->bgzf_slots.as<uint8_t>(), d_zsize, d_zoff, c->bgzf.as<uint8_t>());
    MS_LAUNCH_CHECK(c);
    MS_CUDA(c, cudaStreamSynchronize(c->stream));    // zo / blocks are pageable host memory
    c->bgzf_bytes = tot;
    *total_zbytes = tot;
    return MS_OK;
}

}  // namespace ms
