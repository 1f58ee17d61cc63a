// ms_sample.cu — K1..K4: fresh sampling of mutations for all ranges of all contigs.
//
//   K1  positions   util.py:94-109 sample_with_minimum_distance: a uniform k-subset of
//                   range(n), generated IN ORDER: the value span is cut into equal sort
//                   buckets, a hypergeometric split tree gives every bucket its count
//                   (no value is drawn or scattered for that), a scan turns counts into
//                   candidate slots, and each bucket draws its values as a uniform subset
//                   of its span in shared memory (bitmap rank / bitonic sort).
//   K2  type+length mutator.py:166-182, 229-265 (fused into the sort's write-back)
//   K3  rejection   mutator.py:184-213 first-come greedy acceptance, in parallel:
//                   exclusive prefix-max of the blocking reach marks "anchors"
//                   (candidates no earlier one can block); one thread walks the
//                   short chain between two anchors.
//   K4  linking     mutator.py:268-316 TL<->TLI: uniform random injection of the
//                   smaller list into the larger one via a keyed permutation.
//   K4b records     32-byte splice descriptors + SNP ALT (mutator.py:429-463) +
//                   random insert strings (mutator.py:466-471).
#include <algorithm>
#include "ms_common.cuh"
#include "ms_scan.cuh"

namespace ms {

constexpr int BUCKET_TARGET = 384;   // mean keys per sort bucket of a multi-bucket range
constexpr int SORT_CAP = 1024;       // keys one sort CTA can hold: mean + 32 sigma of a bucket's count; beyond raises MS_ERR_INTERNAL
constexpr int SORT_THREADS = 512;

__device__ inline void raise_error_s(Totals* t, int64_t code, int64_t arg) {
    if (atomicCAS((unsigned long long*)&t->error, 0ull, (unsigned long long)code) == 0ull) t->error_arg = arg;
}

// largest r in [0, n) with key[r] <= x   (key ascending, key[0] <= x)
__device__ inline int upper_idx(const int64_t* key, int n, int64_t x) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (key[mid] <= x) lo = mid; else hi = mid;
    }
    return lo;
}

// Everything a sort CTA needs to start, built on the host with the range table (the lookups it replaces were a
// chain of dependent loads and two 64-bit divisions on one thread at the head of every CTA, profiles/r1m).
struct BucketInfo {
    uint32_t ridx;        // its range
    uint32_t vlo;         // smallest value that falls into it
    uint32_t width;       // number of values in its span
    uint32_t nw;          // 32-bit bitmap words its span needs
};

// K1a: per-range sub-key, and the root of the range's bucket tree gets all k samples
__global__ void k_range_keys(const Range* ranges, int32_t n_ranges, const Contig* contigs, Seed seed, uint32_t purpose, Seed* keys,
                             uint32_t* bucket_cnt) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_ranges) return;
    const Range& g = ranges[r];
    const U4 k = draw(seed, contigs[g.contig].gid, purpose, g.start);
    keys[r] = Seed{k.x, k.y};
    bucket_cnt[g.bucket_lo] = g.k;
}

// K1b: bucket counts.  bucket_cnt[first bucket of a node] holds the node's sample count; a split leaves the left
// child's count in that slot and puts the right child's into its own first bucket.
//   k_split_top   the few nodes that span more than SPLIT_LEAF buckets (ranges with > 98 k candidates: at most
//                 ~2 * buckets / SPLIT_LEAF nodes in the whole table), level by level inside ONE CTA;
//   k_split_leaf  one thread per bucket walks from its SPLIT_LEAF-sized ancestor down to itself, drawing the splits
//                 on the way (threads of a warp share most of the path and run it in lock step; no barriers, no
//                 level launches).  Leaf counts go to a second array because the ancestors' slots are still being
//                 read by their other descendants.
constexpr uint32_t SPLIT_LEAF = 256;

__device__ __forceinline__ uint32_t node_split(const Range& g, const BucketInfo* bi, Seed key, uint32_t lo, uint32_t hi, uint32_t mid, uint32_t n_node) {
    const uint32_t v_lo = bi[lo].vlo, v_mid = bi[mid].vlo, v_hi = hi < g.nb ? bi[hi].vlo : g.n;
    return split_left(key, lo, hi, v_hi - v_lo, v_mid - v_lo, n_node);
}

__global__ void __launch_bounds__(1024)
k_split_top(const Range* ranges, const BucketInfo* binfo, const Seed* keys, const uint32_t* big, int32_t n_big, int levels, uint32_t* bucket_cnt) {
    for (int level = 0; level < levels; ++level) {
        const int64_t items = (int64_t)n_big << level;
        for (int64_t idx = threadIdx.x; idx < items; idx += blockDim.x) {
            const uint32_t ridx = big[idx >> level];
            const Range& g = ranges[ridx];
            if ((uint32_t)level >= g.top_levels) continue;
            const uint32_t j = (uint32_t)(idx & (((int64_t)1 << level) - 1));
            uint32_t lo = 0u, hi = g.nb;
            for (int s = level - 1; s >= 0; --s) {
                const uint32_t mid = (lo + hi) >> 1;
                if ((j >> s) & 1u) lo = mid; else hi = mid;
            }
            const uint32_t mid = (lo + hi) >> 1;
            uint32_t* cnt = bucket_cnt + g.bucket_lo;
            const uint32_t n_node = cnt[lo];
            const uint32_t left = node_split(g, binfo + g.bucket_lo, keys[ridx], lo, hi, mid, n_node);
            cnt[lo] = left;
            cnt[mid] = n_node - left;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
k_split_leaf(const Range* ranges, const BucketInfo* binfo, const Seed* keys, int64_t n_buckets, const uint32_t* bucket_cnt, uint32_t* leaf_cnt) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_buckets) return;
    const uint32_t ridx = binfo[b].ridx;
    const Range& g = ranges[ridx];
    const uint32_t bl = (uint32_t)(b - (int64_t)g.bucket_lo);
    uint32_t lo = 0u, hi = g.nb;
    for (uint32_t s = 0; s < g.top_levels; ++s) {
        const uint32_t mid = (lo + hi) >> 1;
        if (bl < mid) hi = mid; else lo = mid;
    }
    uint32_t cnt = bucket_cnt[(int64_t)g.bucket_lo + lo];
    const Seed key = keys[ridx];
    const BucketInfo* bi = binfo + g.bucket_lo;
    while (hi - lo >= 2u) {
        const uint32_t mid = (lo + hi) >> 1;
        const uint32_t left = node_split(g, bi, key, lo, hi, mid, cnt);
        if (bl < mid) { hi = mid; cnt = left; } else { lo = mid; cnt -= left; }
    }
    leaf_cnt[b] = cnt;
}

template <int K, int J>
__device__ __forceinline__ uint32_t bitonic_step(uint32_t v, int tid, uint32_t* sm) {
    uint32_t other;
    if (J >= 32) {
        sm[tid] = v;
        __syncthreads();
        other = sm[tid ^ J];
        __syncthreads();
    } else {
        other = __shfl_xor_sync(0xffffffffu, v, J);
    }
    const bool keep_min = ((tid & J) == 0) == ((tid & K) == 0);
    return keep_min ? min(v, other) : max(v, other);
}

template <int K, int J>
__device__ __forceinline__ uint32_t bitonic_merge(uint32_t v, int tid, uint32_t* sm) {
    if constexpr (J >= 1) {
        v = bitonic_step<K, J>(v, tid, sm);
        v = bitonic_merge<K, J / 2>(v, tid, sm);
    }
    return v;
}

template <int N2, int K = 2>
__device__ __forceinline__ uint32_t bitonic_sorted(uint32_t v, int tid, uint32_t* sm) {
    if constexpr (K <= N2) {
        v = bitonic_merge<K, K / 2>(v, tid, sm);
        v = bitonic_sorted<N2, K * 2>(v, tid, sm);
    }
    return v;
}

constexpr int SMALL_BUCKET = 128;   // buckets of at most this many keys are sorted four per CTA (k_sort_emit_small)

// position, type, length and blocking reach of the candidate that ends up in `slot` (K2)
__device__ __forceinline__ void emit_candidate(const Range& g, const Contig& ct, int64_t slot, uint32_t v, Seed seed,
                                               int32_t min_dist, const int32_t* blk, int positions_only, int64_t* cand_gpos,
                                               uint8_t* cand_type, uint32_t* cand_len, int64_t* cand_reach, uint32_t* cand_contig) {
    const uint32_t rank = (uint32_t)(slot - g.cand_lo);
    const uint32_t pos = g.start + v + (uint32_t)min_dist * rank;   // util.py:106-108
    cand_gpos[slot] = ct.goff + pos;
    if (positions_only) return;
    uint8_t type; uint32_t len;
    draw_type_len(seed, ct.gid, pos, g, type, len);
    int64_t reach = block_reach(type, pos, len, blk);
    if (reach > ct.len) reach = ct.len;
    cand_type[slot] = type;
    cand_len[slot] = len;
    cand_reach[slot] = type == T_DEAD ? 0 : ct.goff + reach;
    cand_contig[slot] = g.contig;           // (its range is not needed again: the later stages only ask for the contig)
}

// The values of one bucket are a uniform c-subset of its span: draw c values; while some coincide, keep the distinct
// ones and draw as many new values as were lost, from streams numbered by (round, j) — WHICH thread redraws does not
// matter, only how many do, so the resulting set is a pure function of the range key and invariant under any
// relabelling of the span's values, i.e. uniform over c-subsets.

// Small buckets (many-small-contig genomes: a 5 kbp contig has ~67 candidates): four buckets per CTA, 128 threads
// each, instead of one mostly idle 512-thread CTA per bucket (C5: 4.0 ms -> see profiles).
__global__ void __launch_bounds__(SORT_THREADS)
k_sort_emit_small(const Range* ranges, const BucketInfo* binfo, const Seed* keys, const Contig* contigs, const int64_t* bucket_off,
                  int64_t n_buckets, Seed seed, int32_t min_dist, const int32_t* block7, int positions_only,
                  int64_t* cand_gpos, uint8_t* cand_type, uint32_t* cand_len, int64_t* cand_reach, uint32_t* cand_contig) {
    constexpr int G = SORT_THREADS / SMALL_BUCKET;
    __shared__ uint32_t sm[SORT_THREADS];
    __shared__ Range g4[G];
    __shared__ BucketInfo bi4[G];
    __shared__ Seed key4[G];
    __shared__ int32_t blk[7];
    __shared__ uint32_t n_redraw[G];
    const int tid = threadIdx.x, grp = tid / SMALL_BUCKET, t = tid % SMALL_BUCKET;
    const int64_t b = (int64_t)blockIdx.x * G + grp;
    int64_t lo = 0;
    int cnt = 0;
    if (b < n_buckets) { lo = bucket_off[b]; cnt = (int)(bucket_off[b + 1] - lo); }
    const bool mine = cnt > 0 && cnt <= SMALL_BUCKET;
    if (t == 0) {
        n_redraw[grp] = 0u;
        if (mine) { bi4[grp] = binfo[b]; g4[grp] = ranges[bi4[grp].ridx]; key4[grp] = keys[bi4[grp].ridx]; }
    }
    if (tid < 7) blk[tid] = block7[tid];
    __syncthreads();
    uint32_t* const my = sm + grp * SMALL_BUCKET;
    const uint32_t bl = mine ? (uint32_t)(b - (int64_t)g4[grp].bucket_lo) : 0u;
    uint32_t v = 0xFFFFFFFFu;
    if (mine && t < cnt) v = bi4[grp].vlo + bucket_value(key4[grp], bl, 0u, (uint32_t)t, bi4[grp].width);
    for (uint32_t round = 1u;; ++round) {
        v = bitonic_sorted<SMALL_BUCKET>(v, t, my);   // CTA-wide barriers inside: every thread takes part
        my[t] = v;
        __syncthreads();
        const bool dup = mine && t > 0 && t < cnt && my[t - 1] == v;
        if (dup) v = bi4[grp].vlo + bucket_value(key4[grp], bl, round, atomicAdd(&n_redraw[grp], 1u), bi4[grp].width);
        const int any = __syncthreads_or(dup);
        if (!any) break;
        if (t == 0) n_redraw[grp] = 0u;               // (ordered before the next round's atomics by the barriers in the sort)
    }
    if (mine && t < cnt)
        emit_candidate(g4[grp], contigs[g4[grp].contig], lo + t, v, seed, min_dist, blk, positions_only, cand_gpos,
                       cand_type, cand_len, cand_reach, cand_contig);
}

// K1c + K2: draw one bucket's values in shared memory, in order, then write position, type, length and reach.
__global__ void __launch_bounds__(SORT_THREADS, 4)
k_sort_emit(const Range* ranges, const BucketInfo* binfo, const Seed* keys, const Contig* contigs, const int64_t* bucket_off,
            Seed seed, int32_t min_dist, const int32_t* block7, int positions_only,
            int64_t* cand_gpos, uint8_t* cand_type, uint32_t* cand_len, int64_t* cand_reach, uint32_t* cand_contig, Totals* tot,
            int skip_small) {
    __shared__ __align__(16) uint32_t sm[SORT_CAP];
    __shared__ int32_t blk[7];
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t n_redraw[2];
    const int tid = threadIdx.x;
    const int64_t b = blockIdx.x;
    const int64_t lo = bucket_off[b], hi = bucket_off[b + 1];
    const int cnt = (int)(hi - lo);
    if (cnt <= 0 || (skip_small && cnt <= SMALL_BUCKET)) return;
    if (cnt > SORT_CAP) { if (tid == 0) raise_error_s(tot, MS_ERR_INTERNAL, 100 + b); return; }
    const BucketInfo bi = binfo[b];                 // one 16-byte broadcast load; no per-CTA lookups
    const Range& g = ranges[bi.ridx];               // fields are read where they are needed (L1 broadcast)
    const Seed key = keys[bi.ridx];
    const uint32_t s_nw = bi.nw, s_vlo = bi.vlo, width = bi.width;
    const uint32_t bl = (uint32_t)(b - (int64_t)g.bucket_lo);
    if (tid < 7) blk[tid] = block7[tid];
    if (tid < 2) n_redraw[tid] = 0u;
    const int n2 = cnt <= 32 ? 32 : 1 << (32 - __clz(cnt - 1));      // next power of two (bitonic paths)
    if (cnt >= 64 && s_nw <= (uint32_t)SORT_CAP) {
        // Dense bucket (span of at most 32 Ki values): one bit per value in a bitmap; a draw that finds its bit set
        // is a coincidence and is redrawn in the next round.  The sorted order is then read off the bitmap —
        // prefix-sum the popcounts, write each value to its rank (~100 instructions per thread instead of the ~360
        // of the 512-key bitonic network).
        const uint32_t vlo = s_vlo, nw = s_nw;
        static_assert(SORT_CAP / 4 <= SORT_THREADS, "one uint4 per thread clears the bitmap");
        if (tid < SORT_CAP / 4) reinterpret_cast<uint4*>(sm)[tid] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
        uint32_t n_draw = (uint32_t)cnt;
        for (uint32_t round = 0u; n_draw > 0u; ++round) {
            for (uint32_t jp = tid; 2u * jp < n_draw; jp += SORT_THREADS) {      // one Philox block per two draws
                const U4 r = bucket_block(key, bl, round, jp);
#pragma unroll
                for (uint32_t h = 0; h < 2u; ++h) {
                    if (2u * jp + h >= n_draw) break;
                    const uint32_t d = bucket_value_of(r, h, width);
                    const uint32_t bit = 1u << (d & 31u);
                    if (atomicOr(&sm[d >> 5], bit) & bit) atomicAdd(&n_redraw[round & 1u], 1u);
                }
            }
            __syncthreads();
            n_draw = n_redraw[round & 1u];
            if (tid == 0) n_redraw[(round + 1u) & 1u] = 0u;
            __syncthreads();
        }
        const uint32_t i0 = 2u * (uint32_t)tid;
        uint32_t w0 = i0 < nw ? sm[i0] : 0u, w1 = i0 + 1u < nw ? sm[i0 + 1u] : 0u;
        const uint32_t mine = (uint32_t)(__popc(w0) + __popc(w1));
        uint32_t incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d); if ((tid & 31) >= d) incl += y; }
        if ((tid & 31) == 31) warp_tot[tid >> 5] = incl;
        __syncthreads();                                   // every thread holds its bitmap words: sm can be overwritten
        // + the totals of the warps before this one: lane l holds warp l's total (16 warps), summed across the warp
        uint32_t rank = incl - mine + __reduce_add_sync(0xffffffffu, (tid & 31) < (tid >> 5) ? warp_tot[tid & 31] : 0u);
        uint32_t vb = vlo + (i0 << 5);
        while (w0) { const int bit = __ffs(w0) - 1; w0 &= w0 - 1u; sm[rank++] = vb + (uint32_t)bit; }
        vb += 32u;
        while (w1) { const int bit = __ffs(w1) - 1; w1 &= w1 - 1u; sm[rank++] = vb + (uint32_t)bit; }
        __syncthreads();
    } else if (n2 <= SORT_THREADS) {
        // one key per thread: strides below 32 are exchanged with shuffles, only the
        // 10 cross-warp phases of a 512-key bitonic network go through shared memory;
        // the network is unrolled at compile time (loop control was 22 % of the kernel, profiles/r1e)
        uint32_t v = tid < cnt ? s_vlo + bucket_value(key, bl, 0u, (uint32_t)tid, width) : 0xFFFFFFFFu;
        for (uint32_t round = 1u;; ++round) {
            switch (n2) {
                case 32:  v = bitonic_sorted<32>(v, tid, sm); break;
                case 64:  v = bitonic_sorted<64>(v, tid, sm); break;
                case 128: v = bitonic_sorted<128>(v, tid, sm); break;
                case 256: v = bitonic_sorted<256>(v, tid, sm); break;
                default:  v = bitonic_sorted<512>(v, tid, sm); break;
            }
            sm[tid] = v;
            __syncthreads();
            const bool dup = tid > 0 && tid < cnt && sm[tid - 1] == v;
            if (dup) v = s_vlo + bucket_value(key, bl, round, atomicAdd(&n_redraw[round & 1u], 1u), width);
            const int any = __syncthreads_or(dup);
            if (!any) break;
            if (tid == 0) n_redraw[(round + 1u) & 1u] = 0u;
        }
    } else {
        for (int i = tid; i < n2; i += SORT_THREADS) sm[i] = i < cnt ? s_vlo + bucket_value(key, bl, 0u, (uint32_t)i, width) : 0xFFFFFFFFu;
        __syncthreads();
        for (uint32_t round = 1u;; ++round) {
            for (int k = 2; k <= n2; k <<= 1) {
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int i = tid; i < n2; i += SORT_THREADS) {
                        const int x = i ^ j;
                        if (x > i) {
                            const uint32_t a = sm[i], c = sm[x];
                            const bool asc = (i & k) == 0;
                            if ((a > c) == asc) { sm[i] = c; sm[x] = a; }
                        }
                    }
                    __syncthreads();
                }
            }
            // (two keys per thread: decide on both before either is replaced)
            const int i0 = tid, i1 = tid + SORT_THREADS;
            const bool d0 = i0 > 0 && i0 < cnt && sm[i0 - 1] == sm[i0];
            const bool d1 = i1 < cnt && sm[i1 - 1] == sm[i1];
            const int any = __syncthreads_or(d0 || d1);
            if (!any) break;
            if (d0) sm[i0] = s_vlo + bucket_value(key, bl, round, atomicAdd(&n_redraw[round & 1u], 1u), width);
            if (d1) sm[i1] = s_vlo + bucket_value(key, bl, round, atomicAdd(&n_redraw[round & 1u], 1u), width);
            if (tid == 0) n_redraw[(round + 1u) & 1u] = 0u;
            __syncthreads();
        }
    }
    const Contig& ct = contigs[g.contig];
    for (int i = tid; i < cnt; i += SORT_THREADS)
        emit_candidate(g, ct, lo + i, sm[i], seed, min_dist, blk, positions_only, cand_gpos, cand_type, cand_len, cand_reach,
                       cand_contig);
}

// K3b: walk the chain that starts at each anchor (mutator.py:184-213).
__global__ void __launch_bounds__(256)
k_resolve(int64_t K, const int64_t* gpos, const int64_t* reach, const uint8_t* type, const uint8_t* anchor, uint8_t* accept) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= K || !anchor[s]) return;
    accept[s] = 1;
    int64_t cur = reach[s];
    for (int64_t t = s + 1; t < K && !anchor[t]; ++t) {
        if (type[t] == T_DEAD) continue;           // inversion that does not fit: dropped, blocks nothing (:199-201)
        if (gpos[t] >= cur) { accept[t] = 1; cur = reach[t]; }
    }
}

// The same without the prefix-max scan, for the usual case of short blocking spans: an earlier candidate can only
// block j if it starts less than `maxspan` before it, so "no earlier candidate reaches past j" is a look-back of
// 0-1 steps (average spacing is 1/rate, spans are a few dozen bases).
__device__ __forceinline__ bool is_anchor_local(int64_t j, const int64_t* gpos, const int64_t* reach, const uint8_t* type, int64_t maxspan) {
    if (type[j] == T_DEAD) return false;
    const int64_t g = gpos[j];
    for (int64_t i = j - 1; i >= 0 && g - gpos[i] < maxspan; --i)
        if (reach[i] > g) return false;
    return true;
}

// Every candidate's anchor test is evaluated once, on registers: a warp covers 28 candidates plus three before them
// (their positions and reaches reach the owners by shuffle: a look-back of up to three candidates needs no memory;
// deeper ones — under 1 % at genome-like densities — go on from memory) and the first one of the next warp, whose flag
// tells lane 30 whether its chain ends right there (as it does for almost every candidate).
constexpr int RESOLVE_OWN = 28, RESOLVE_BACK = 3;
__global__ void __launch_bounds__(256)
k_resolve_local(int64_t K, const int64_t* gpos, const int64_t* reach, const uint8_t* type, int64_t maxspan, uint8_t* accept) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t s = warp * RESOLVE_OWN - RESOLVE_BACK + lane;
    const bool valid = s >= 0 && s < K;
    const int64_t g = valid ? gpos[s] : INT64_MIN / 2;          // (an absent predecessor is infinitely far away)
    const int64_t r = valid ? reach[s] : 0;
    bool anchor = valid && type[s] != T_DEAD;
    bool open = anchor;                                          // look-back not finished yet
#pragma unroll
    for (int d = 1; d <= RESOLVE_BACK; ++d) {
        const int64_t gp = __shfl_up_sync(0xffffffffu, g, d), rp = __shfl_up_sync(0xffffffffu, r, d);
        if (open && lane >= d) {
            if (g - gp >= maxspan) open = false;
            else if (rp > g) { anchor = false; open = false; }
        }
    }
    if (open && lane >= RESOLVE_BACK) {
        for (int64_t i = s - RESOLVE_BACK - 1; i >= 0 && g - gpos[i] < maxspan; --i)
            if (reach[i] > g) { anchor = false; break; }
    }
    const bool next_anchor = __shfl_down_sync(0xffffffffu, anchor, 1) != 0;
    if (lane < RESOLVE_BACK || lane == 31 || !anchor) return;   // the halo lanes own nothing
    accept[s] = 1;
    if (next_anchor || s + 1 >= K) return;
    int64_t cur = r;
    for (int64_t t = s + 1; t < K && (t == s + 1 || !is_anchor_local(t, gpos, reach, type, maxspan)); ++t) {
        if (type[t] == T_DEAD) continue;
        if (gpos[t] >= cur) { accept[t] = 1; cur = reach[t]; }
    }
}

// Compaction of the accepted candidates and of the accepted TL / TLI among them (three lists in one scan), written for
// its types: a thread owns 8 consecutive candidates and reads their accept / type bytes as two 8-byte words (the generic
// scan kernels read them byte by byte and carried eight I64x3 per thread: 80 registers, 0.29 ms).
__device__ __forceinline__ void compact_masks(const uint8_t* accept, const uint8_t* type, int64_t base, int64_t K, uint32_t& m_acc,
                                              uint32_t& m_tl, uint32_t& m_tli) {
    uint64_t a8 = 0ull, t8 = 0ull;
    if (base + 8 <= K) {
        a8 = __ldg(reinterpret_cast<const unsigned long long*>(accept + base));
        t8 = __ldg(reinterpret_cast<const unsigned long long*>(type + base));
    } else {
        for (int j = 0; j < 8 && base + j < K; ++j) { a8 |= (uint64_t)accept[base + j] << (8 * j); t8 |= (uint64_t)type[base + j] << (8 * j); }
    }
    m_acc = m_tl = m_tli = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t a = (uint32_t)(a8 >> (8 * j)) & 0xffu, t = (uint32_t)(t8 >> (8 * j)) & 0xffu;
        if (a) { m_acc |= 1u << j; if (t == T_TL) m_tl |= 1u << j; if (t == T_TLI) m_tli |= 1u << j; }
    }
}

__global__ void __launch_bounds__(SCAN_THREADS)
k_compact_reduce(const uint8_t* accept, const uint8_t* type, int64_t K, I64x3* tile_sums) {
    __shared__ I64x3 sm[2 * SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t ma, mtl, mtli;
    compact_masks(accept, type, base, K, ma, mtl, mtli);
    I64x3 total;
    block_excl_scan(I64x3{__popc(ma), __popc(mtl), __popc(mtli)}, I64x3{0, 0, 0}, SumOp(), total, sm);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS)
k_compact_down(const uint8_t* accept, const uint8_t* type, int64_t K, const I64x3* tile_prefix, uint32_t* acc_list, uint32_t* tl_list,
               uint32_t* tli_list, int32_t* link) {
    __shared__ I64x3 sm[2 * SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t ma, mtl, mtli;
    compact_masks(accept, type, base, K, ma, mtl, mtli);
    I64x3 total;
    const I64x3 ex = block_excl_scan(I64x3{__popc(ma), __popc(mtl), __popc(mtli)}, I64x3{0, 0, 0}, SumOp(), total, sm);
    const I64x3 tp = tile_prefix[blockIdx.x];
    const uint32_t i0 = (uint32_t)base;               // candidate slots fit 31 bits (ms_set_ranges checks)
    // the tile's accepted slots are one contiguous stretch of the list: ranked in shared memory, written coalesced
    // (one 4-byte store per accepted candidate at a 32-byte lane stride was most of this kernel's 0.17 ms)
    __shared__ uint32_t stage[SCAN_TILE];
    uint32_t r = (uint32_t)ex.a;
    while (ma) { const int j = __ffs(ma) - 1; ma &= ma - 1u; stage[r++] = i0 + (uint32_t)j; }
    __syncthreads();
    uint32_t* const a = acc_list + tp.a;
    for (uint32_t x = threadIdx.x; x < (uint32_t)total.a; x += SCAN_THREADS) a[x] = stage[x];
    uint32_t* b = tl_list + tp.b + ex.b;              // (2 % of the candidates: written directly)
    uint32_t* cc = tli_list + tp.c + ex.c;
    // (their link entries start out "unlinked"; k_link overwrites the paired ones: no 4-byte-per-candidate memset)
    while (mtl) { const int j = __ffs(mtl) - 1; mtl &= mtl - 1u; *b++ = i0 + (uint32_t)j; link[i0 + j] = -1; }
    while (mtli) { const int j = __ffs(mtli) - 1; mtli &= mtli - 1u; *cc++ = i0 + (uint32_t)j; link[i0 + j] = -1; }
}

// first TL / TLI list entry of every contig.  One warp per (contig, list): a 32-ary search (each round the lanes probe
// 32 evenly spaced entries) finishes in 4-5 rounds of two dependent loads; the one-thread-per-contig binary search it
// replaces took 50 us on 24 contigs — a fixed cost that did not shrink with the GPU count (SCALE_r01).
__global__ void __launch_bounds__(128)
k_contig_tl_bounds(const Contig* contigs, int32_t n_contigs, const int64_t* gpos, const uint32_t* tl_list, const uint32_t* tli_list,
                   const Totals* tot, int64_t* tl_base, int64_t* tli_base) {
    const int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= 2 * (n_contigs + 1)) return;
    const int c = w >> 1;
    const bool tli = (w & 1) != 0;
    const uint32_t* list = tli ? tli_list : tl_list;
    const int64_t n = tli ? tot->pad[1] : tot->pad[0];
    int64_t* out = tli ? tli_base : tl_base;
    if (c == n_contigs) { if (lane == 0) out[c] = n; return; }
    const int64_t key = contigs[c].goff;
    int64_t lo = 0, hi = n;                       // first entry with gpos >= key lies in [lo, hi]
    while (hi - lo > 0) {
        const int64_t span = hi - lo;
        const int64_t probe = lo + (span * (lane + 1)) / 33;          // 32 probes inside [lo, hi)
        const bool less = probe < hi && gpos[list[probe]] < key;
        const uint32_t m = __ballot_sync(0xffffffffu, less);
        const int k = __popc(m);                  // probes are ascending: the first k are "less"
        const int64_t p_lo = k ? lo + (span * k) / 33 + 1 : lo;
        const int64_t p_hi = k < 32 ? lo + (span * (k + 1)) / 33 : hi;
        if (p_lo == lo && p_hi == hi) {           // span too small for the probes to split it
            if (gpos[list[lo]] < key) lo = lo + 1; else hi = lo;
        } else { lo = p_lo; hi = p_hi < p_lo ? p_lo : p_hi; }
    }
    if (lane == 0) out[c] = lo;
}

// K4: element j of the smaller list is paired with element rho(j) of the larger one,
// rho a keyed permutation of the larger list: a uniform random injection, which is
// what "remove random surplus, shuffle, zip" (mutator.py:277-304) produces.
// link[slot]: -1 unlinked (dropped), -2 kept TL, >= 0 (TLI) candidate slot of its TL.
__device__ __forceinline__ void link_one(int64_t x, const Contig* contigs, const Range* ranges, const uint32_t* cand_contig,
                                         const uint32_t* tl_list, int64_t n_tl, const uint32_t* tli_list, int64_t n_tli,
                                         const int64_t* tl_base, const int64_t* tli_base, Seed seed, int32_t* link);

__global__ void __launch_bounds__(256)
k_link(const Contig* contigs, const Range* ranges, const uint32_t* cand_contig, const uint32_t* tl_list, const uint32_t* tli_list,
       const Totals* tot, const int64_t* tl_base, const int64_t* tli_base, Seed seed, int32_t* link) {
    const int64_t n_tl = tot->pad[0], n_tli = tot->pad[1];
    if (n_tl == 0 || n_tli == 0) return;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n_tl + n_tli; x += (int64_t)gridDim.x * blockDim.x)
        link_one(x, contigs, ranges, cand_contig, tl_list, n_tl, tli_list, n_tli, tl_base, tli_base, seed, link);
}

__device__ __forceinline__ void link_one(int64_t x, const Contig* contigs, const Range* ranges, const uint32_t* cand_contig,
                                         const uint32_t* tl_list, int64_t n_tl, const uint32_t* tli_list, int64_t n_tli,
                                         const int64_t* tl_base, const int64_t* tli_base, Seed seed, int32_t* link) {
    const bool is_tl = x < n_tl;
    const int64_t idx = is_tl ? x : x - n_tl;
    const uint32_t slot = is_tl ? tl_list[idx] : tli_list[idx];
    const uint32_t c = cand_contig[slot];
    const int64_t a = tl_base[c + 1] - tl_base[c], b = tli_base[c + 1] - tli_base[c];
    if (a == 0 || b == 0) return;
    // ties (a == b) are driven from the TL side
    const bool tl_small = a <= b;
    if (is_tl != tl_small) return;
    const int64_t j = idx - (is_tl ? tl_base[c] : tli_base[c]);
    const uint32_t m = (uint32_t)(tl_small ? b : a);
    uint32_t rho;
    if (m == 1) rho = 0;
    else { const Prp p = make_prp(seed, contigs[c].gid, P_TL_PRP, 0, m); rho = prp_apply(p, (uint32_t)j); }
    const uint32_t other = tl_small ? tli_list[tli_base[c] + rho] : tl_list[tl_base[c] + rho];
    const uint32_t tl_slot = is_tl ? slot : other, tli_slot = is_tl ? other : slot;
    link[tl_slot] = -2;
    link[tli_slot] = (int32_t)tl_slot;
}

// K4b: one 32-byte record per accepted candidate, in place of the accepted list (no second compaction: an
// unpaired TL / TLI becomes a dead no-op record), together with its length delta and VCF line size so that the
// plan stage does not have to re-read the records.
}  // namespace ms
#include "ms_vcf_core.h"
namespace ms {

__global__ void __launch_bounds__(256, 8)      // 32 registers: the SNP reference gather needs all 64 warps to hide its latency
k_build_records(const Totals* tot, const uint32_t* acc_slot, const int64_t* gpos, const uint8_t* type, const uint32_t* len,
                const uint32_t* cand_contig, const int32_t* link, const Range* ranges, const Contig* contigs, VcfView vv,
                const Tables* tab, Seed seed, double p_ti, Rec* recs, int32_t* delta, uint32_t* vsize, bool defer_bases) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= tot->n_accepted) return;             // the grid is sized from the candidate count (an upper bound)
    const uint32_t s = acc_slot[e];
    const uint32_t cidx = cand_contig[s];
    const Contig& ct = contigs[cidx];
    const int64_t g = gpos[s];
    const uint32_t pos = (uint32_t)(g - ct.goff);
    const uint8_t t = type[s];
    const uint32_t l = len[s];
    Rec r;
    r.pos = pos; r.out = 0; r.src = 0; r.type = t; r.ref = 0; r.alt = 0; r.contig = cidx;
    // SNP substitution, insert bases and the translocation coin are all Philox(contig, purpose of the type, pos): one
    // block per thread ahead of the switch instead of three copies of the generator run by three lane subsets
    const U4 rnd = draw(seed, ct.gid, t == T_SN ? (uint32_t)P_SNP : t == T_IN ? (uint32_t)P_INSERT : (uint32_t)P_TL_REV, pos);
    switch (t) {
        case T_SN: {
            r.cons = 1; r.prod = 1; r.kind = K_SNP;
            if (!defer_bases) {   // streamed runs fill these per contig group once its bases have arrived (k_snp_fill)
                r.ref = tab->conv[vv.genome[g]];
                r.alt = snp_of_block(rnd, r.ref, p_ti, tab->trans);
            }
        } break;
        case T_IN: r.cons = 0; r.prod = l; r.kind = K_RAND; r.src = (int64_t)u64_of(rnd.x, rnd.y); break;   // = rand_insert_cache(seed, gid, pos)
        case T_DE: r.cons = l; r.prod = 0; r.kind = K_NONE; break;
        case T_IV: r.cons = l; r.prod = l; r.kind = K_RC; r.src = g; break;
        case T_DU: r.cons = 0; r.prod = l; r.kind = K_RAW; r.src = g; break;
        default: {  // T_TL / T_TLI: kept only when linked (link: -1 unlinked, -2 kept TL, >= 0 slot of the TLI's TL)
            const int32_t lk = link[s];
            if (lk == -1) { r.cons = 0; r.prod = 0; r.kind = K_NONE; r.type = T_DEAD; }
            else if (t == T_TL) { r.cons = l; r.prod = 0; r.kind = K_NONE; }
            else {
                const uint32_t tl_len = len[lk];
                r.cons = 0; r.prod = tl_len; r.src = gpos[lk];
                r.kind = ((rnd.x & 1u) != 0 && tl_len >= 2) ? K_RC : K_CONV;              // = draw_tl_reverse(seed, gid, pos, tl_len)
            }
        } break;
    }
    recs[e] = r;
    delta[e] = (int32_t)r.prod - (int32_t)r.cons;
    vsize[e] = (defer_bases ? vcf_line_bound(vv, ct, r) : vcf_line_size(vv, ct, r)) | (r.kind != K_SNP ? VSIZE_SV : 0u);
}

__global__ void __launch_bounds__(256) k_count_types(const Rec* recs, int64_t n, Totals* tot) {
    __shared__ unsigned int h[8];
    if (threadIdx.x < 8) h[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        { const uint8_t t = recs[i].type; if (t < 8) atomicAdd(&h[t], 1u); }
    __syncthreads();
    if (threadIdx.x < 8 && h[threadIdx.x]) atomicAdd((unsigned long long*)&tot->counts[threadIdx.x], (unsigned long long)h[threadIdx.x]);
}

template <class T> __global__ void k_copy_scalar(const T* src, T* dst) { *dst = *src; }
__global__ void k_store_counts(const I64x3* total, Totals* tot) { tot->n_accepted = total->a; tot->pad[0] = total->b; tot->pad[1] = total->c; }

// ---- host orchestration --------------------------------------------------------------
static int draw_and_sort(ms_ctx* c, Seed seed, uint32_t purpose, int32_t min_dist, int positions_only, const Contig* d_ctg) {
    cudaStream_t st = c->stream;
    const int64_t K = c->n_candidates;
    const int32_t R = c->n_ranges;
    const Range* d_ranges = c->ranges.as<Range>();
    // side arrays kept right behind the Range table
    int64_t* d_cand_lo = reinterpret_cast<int64_t*>(c->ranges.as<uint8_t>() + sizeof(Range) * (size_t)R);
    int64_t* d_bucket_lo = d_cand_lo + (R + 1);
    Seed* d_keys = reinterpret_cast<Seed*>(d_bucket_lo + (R + 1));
    int32_t* d_block = reinterpret_cast<int32_t*>(d_keys + R);
    Totals* d_tot = c->totals.as<Totals>();
    const BucketInfo* d_binfo = c->bucket_range.as<BucketInfo>();

    MS_CUDA(c, c->bucket_cnt.ensure((size_t)(c->n_buckets + 1) * 8));   // node counts, then leaf counts
    MS_CUDA(c, c->bucket_off.ensure((size_t)(c->n_buckets + 1) * 8));
    MS_CUDA(c, c->cand_reach.ensure((size_t)K * 8 + 16));   // cand_gpos lives in svec
    MS_CUDA(c, c->svec.ensure((size_t)(K + 1) * 8));
    MS_CUDA(c, c->cand_type.ensure((size_t)K + 16));
    MS_CUDA(c, c->cand_len.ensure((size_t)K * 4 + 16));
    MS_CUDA(c, c->lvec.ensure((size_t)K * 4 + 16));         // cand_contig
    uint32_t* d_cnt = c->bucket_cnt.as<uint32_t>();
    int64_t* d_boff = c->bucket_off.as<int64_t>();

    stage_begin(c, ST_SAMPLE_POS);
    k_range_keys<<<(unsigned)ceil_div(R, 128), 128, 0, st>>>(d_ranges, R, d_ctg, seed, purpose, d_keys, d_cnt);
    MS_LAUNCH_CHECK(c);
    if (c->n_big > 0) {
        k_split_top<<<1, 1024, 0, st>>>(d_ranges, d_binfo, d_keys, c->big_ranges.as<uint32_t>(), c->n_big, c->split_levels, d_cnt);
        MS_LAUNCH_CHECK(c);
    }
    uint32_t* d_leaf = d_cnt + (c->n_buckets + 1);
    k_split_leaf<<<(unsigned)ceil_div(c->n_buckets, 256), 256, 0, st>>>(d_ranges, d_binfo, d_keys, c->n_buckets, d_cnt, d_leaf);
    MS_LAUNCH_CHECK(c);
    {
        const uint32_t* cnt = d_leaf;
        auto in = [=] __device__(int64_t i) -> int64_t { return (int64_t)cnt[i]; };
        auto out = [=] __device__(int64_t i, int64_t ex, int64_t) { d_boff[i] = ex; };
        int64_t* d_total = nullptr;
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, c->n_buckets, (int64_t)0, SumOp(), c->scan_tmp, &d_total)));
        k_copy_scalar<int64_t><<<1, 1, 0, st>>>(d_total, d_boff + c->n_buckets);
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_SAMPLE_POS);

    stage_begin(c, ST_SAMPLE_TYPE);
    const int any_small = c->any_small, any_large = c->any_large;
    if (any_small) {
        k_sort_emit_small<<<(unsigned)ceil_div(c->n_buckets, SORT_THREADS / SMALL_BUCKET), SORT_THREADS, 0, st>>>(
            d_ranges, d_binfo, d_keys, d_ctg, d_boff, c->n_buckets, seed, min_dist, d_block, positions_only,
            c->svec.as<int64_t>(), c->cand_type.as<uint8_t>(), c->cand_len.as<uint32_t>(), c->cand_reach.as<int64_t>(),
            c->lvec.as<uint32_t>());
        MS_LAUNCH_CHECK(c);
    }
    if (any_large) {
        k_sort_emit<<<(unsigned)c->n_buckets, SORT_THREADS, 0, st>>>(d_ranges, d_binfo, d_keys, d_ctg, d_boff, seed, min_dist, d_block,
                                                                     positions_only, c->svec.as<int64_t>(), c->cand_type.as<uint8_t>(),
                                                                     c->cand_len.as<uint32_t>(), c->cand_reach.as<int64_t>(),
                                                                     c->lvec.as<uint32_t>(), d_tot, any_small);
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_SAMPLE_TYPE);
    return MS_OK;
}

int sample_pipeline(ms_ctx* c, uint64_t seed64, bool defer_bases) {
    if (c->n_contigs <= 0 || !c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_sample: no genome resident");
    if (c->n_ranges < 0) MS_FAIL(c, MS_ERR_STATE, "ms_sample: call ms_set_ranges first");
    cudaStream_t st = c->stream;
    const Seed seed = make_seed(seed64);
    const int64_t K = c->n_candidates;
    Totals* d_tot = c->totals.as<Totals>();
    MS_CUDA(c, cudaMemsetAsync(d_tot, 0, sizeof(Totals), st));
    c->last_totals = Totals{};
    c->last_totals.n_candidates = K;
    c->n_recs = 0; c->lit_bytes = 0;
    MS_CUDA(c, c->recs.ensure(64));
    MS_CUDA(c, c->lit.ensure(64));
    if (K == 0 || c->n_ranges == 0) return MS_OK;

    int rc = draw_and_sort(c, seed, P_RANGE_KEY, c->min_dist, 0, c->contigs.as<Contig>());
    if (rc) return rc;

    const int64_t* d_gpos = c->svec.as<int64_t>();
    const int64_t* d_reach = c->cand_reach.as<int64_t>();
    const uint8_t* d_type = c->cand_type.as<uint8_t>();
    const uint32_t* d_len = c->cand_len.as<uint32_t>();
    const uint32_t* d_crange = c->lvec.as<uint32_t>();
    const Range* d_ranges = c->ranges.as<Range>();
    const Contig* d_contigs = c->contigs.as<Contig>();

    // ---- K3: rejection -------------------------------------------------------------
    stage_begin(c, ST_SAMPLE_RESOLVE);
    MS_CUDA(c, c->cand_pm.ensure((size_t)K + 16));
    MS_CUDA(c, c->cand_accept.ensure((size_t)K + 16));
    uint8_t* d_anchor = c->cand_pm.as<uint8_t>();
    uint8_t* d_accept = c->cand_accept.as<uint8_t>();
    MS_CUDA(c, cudaMemsetAsync(d_accept, 0, (size_t)K, st));
    const int64_t maxspan = c->maxspan;   // (per-range host loops live in upload_ranges: C5 has 200 k ranges)
    if (maxspan <= 4096) {
        k_resolve_local<<<(unsigned)ceil_div(ceil_div(K, RESOLVE_OWN) * 32, 256), 256, 0, st>>>(K, d_gpos, d_reach, d_type, maxspan, d_accept);
        MS_LAUNCH_CHECK(c);
    } else {
        auto in = [=] __device__(int64_t i) -> int64_t { return d_reach[i]; };
        auto out = [=] __device__(int64_t i, int64_t ex, int64_t) {
            d_anchor[i] = (d_type[i] != T_DEAD && d_gpos[i] >= ex) ? 1 : 0;
        };
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, K, (int64_t)0, MaxOp(), c->scan_tmp, (int64_t**)nullptr)));
        k_resolve<<<(unsigned)ceil_div(K, 256), 256, 0, st>>>(K, d_gpos, d_reach, d_type, d_anchor, d_accept);
        MS_LAUNCH_CHECK(c);
    }
    // compaction of accepted candidates + TL / TLI lists in one pass
    MS_CUDA(c, c->link.ensure((size_t)K * 4 + 16));
    MS_CUDA(c, c->acc_idx.ensure((size_t)K * 4 + 16));
    MS_CUDA(c, c->tl_list.ensure((size_t)K * 4 + 16));
    MS_CUDA(c, c->tli_list.ensure((size_t)K * 4 + 16));
    uint32_t* d_acc = c->acc_idx.as<uint32_t>();
    uint32_t* d_tl = c->tl_list.as<uint32_t>();
    uint32_t* d_tli = c->tli_list.as<uint32_t>();
    {
        const int64_t nt = ceil_div(K, SCAN_TILE);
        MS_CUDA(c, c->scan_tmp.ensure((size_t)(nt + 1) * sizeof(I64x3)));
        I64x3* ts = c->scan_tmp.as<I64x3>();
        k_compact_reduce<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(d_accept, d_type, K, ts);
        MS_LAUNCH_CHECK(c);
        MS_CUDA(c, (scan_mid_phase<I64x3>(c, ts, nt, I64x3{0, 0, 0}, SumOp())));
        k_compact_down<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(d_accept, d_type, K, ts, d_acc, d_tl, d_tli, c->link.as<int32_t>());
        MS_LAUNCH_CHECK(c);
        k_store_counts<<<1, 1, 0, st>>>(ts + nt, d_tot);      // accepted / TL / TLI counts stay on the device: no host round trip
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_SAMPLE_RESOLVE);

    // ---- K4: TL <-> TLI linking -------------------------------------------------------
    stage_begin(c, ST_SAMPLE_LINK);
    int32_t* d_link = c->link.as<int32_t>();       // TL / TLI entries were set to -1 (unlinked) by the compaction
    {
        MS_CUDA(c, c->contig_tl.ensure((size_t)(c->n_contigs + 1) * 16));
        int64_t* d_tlb = c->contig_tl.as<int64_t>();
        int64_t* d_tlib = d_tlb + (c->n_contigs + 1);
        k_contig_tl_bounds<<<(unsigned)ceil_div(2 * (int64_t)(c->n_contigs + 1) * 32, 128), 128, 0, st>>>(d_contigs, c->n_contigs, d_gpos, d_tl, d_tli,
                                                                                                     d_tot, d_tlb, d_tlib);
        MS_LAUNCH_CHECK(c);
        k_link<<<NUM_SMS_B200 * 8, 256, 0, st>>>(d_contigs, d_ranges, d_crange, d_tl, d_tli, d_tot, d_tlb, d_tlib, seed, d_link);
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_SAMPLE_LINK);

    // ---- K4b: records (buffers sized from the candidate count, an upper bound of the accepted count) ------------------
    stage_begin(c, ST_SAMPLE_FINAL);
    c->seed_last = seed;
    MS_CUDA(c, c->recs.ensure((size_t)(K + 1) * sizeof(Rec)));
    MS_CUDA(c, c->keep.ensure((size_t)(K + 1) * 4));
    MS_CUDA(c, c->cand_val.ensure((size_t)(K + 1) * 4));
    {
        const Tables* d_tab = c->tables.as<Tables>();
        VcfView vv{c->genome.as<uint8_t>(), c->lit.as<uint8_t>(), c->names.as<uint8_t>(), d_tab->conv, d_tab->comp, seed};
        k_build_records<<<(unsigned)ceil_div(K, 256), 256, 0, st>>>(d_tot, d_acc, d_gpos, d_type, d_len, d_crange, d_link, d_ranges,
                                                                    d_contigs, vv, d_tab, seed, c->p_ti, c->recs.as<Rec>(),
                                                                    c->keep.as<int32_t>(), c->cand_val.as<uint32_t>(), defer_bases);
        MS_LAUNCH_CHECK(c);
    }
    MS_CUDA(c, cudaMemcpyAsync(c->h_totals, d_tot, sizeof(Totals), cudaMemcpyDeviceToHost, st));
    stage_end(c, ST_SAMPLE_FINAL);
    MS_CUDA(c, cudaStreamSynchronize(st));
    if (c->h_totals->error) MS_FAIL(c, (int)c->h_totals->error, "ms_sample: kernel error %lld (arg %lld)", (long long)c->h_totals->error,
                                    (long long)c->h_totals->error_arg);
    const int64_t n_acc = c->h_totals->n_accepted;
    c->last_totals.n_accepted = n_acc;
    c->n_recs = n_acc;
    c->lit_bytes = 0;
    c->last_totals.n_recs = n_acc;
    c->last_totals.lit_bytes = 0;
    c->counts_valid = false;
    c->sizes_valid = true;
    c->rec_out_valid = true;      // nothing to fill in until the next plan (svec is the candidates' scratch here)
    return MS_OK;
}

int count_types(ms_ctx* c) {
    if (c->counts_valid) return MS_OK;
    Totals* d_tot = c->totals.as<Totals>();
    MS_CUDA(c, cudaMemsetAsync(d_tot->counts, 0, sizeof(d_tot->counts), c->stream));
    if (c->n_recs > 0) {
        k_count_types<<<NUM_SMS_B200 * 4, 256, 0, c->stream>>>(c->recs.as<Rec>(), c->n_recs, d_tot);
        MS_LAUNCH_CHECK(c);
    }
    MS_CUDA(c, cudaMemcpyAsync(c->h_totals, d_tot, sizeof(Totals), cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int t = 0; t < 8; ++t) c->last_totals.counts[t] = c->h_totals->counts[t];
    c->counts_valid = true;
    return MS_OK;
}

// Range table upload shared by ms_set_ranges and ms_it_breakpoints.
static int upload_ranges(ms_ctx* c, int32_t min_dist, const std::vector<Contig>& ctg) {
    const int32_t R = (int32_t)c->h_ranges.size();
    std::vector<int64_t> cand_lo(R + 1), bucket_lo(R + 1);
    int64_t K = 0, NB = 0;
    uint32_t max_top = 0;
    std::vector<uint32_t> big;                             // ranges with more than SPLIT_LEAF buckets
    for (int32_t r = 0; r < R; ++r) {
        Range& g = c->h_ranges[r];
        const int64_t n = (int64_t)g.stop - ((int64_t)g.k - 1) * min_dist - (int64_t)g.start;   // util.py:104
        if ((int64_t)g.k > n || n <= 0)
            MS_FAIL(c, MS_ERR_SAMPLE, "Sample larger than population or is negative (range %u-%u of contig %u: k=%u, population=%lld)",
                    g.start + 1, g.stop + 1, g.contig + 1, g.k, (long long)n);
        g.n = (uint32_t)n;
        g.cand_lo = K;
        g.nb = (uint32_t)std::max<int64_t>(1, ceil_div(g.k, BUCKET_TARGET));
        g.bscale = g.nb == 1u ? 0u : (uint32_t)((((uint64_t)g.nb) << 32) / (uint64_t)n);
        g.bucket_lo = (uint32_t)NB;
        g.top_levels = 0u;                                 // halvings until every node spans at most SPLIT_LEAF buckets
        while ((((uint64_t)g.nb + (1ull << g.top_levels) - 1) >> g.top_levels) > SPLIT_LEAF) ++g.top_levels;
        if (g.top_levels) { big.push_back((uint32_t)r); max_top = std::max(max_top, g.top_levels); }
        g.gstart = ctg[g.contig].goff + g.start;
        cand_lo[r] = K; bucket_lo[r] = NB;
        K += g.k; NB += g.nb;
    }
    cand_lo[R] = K; bucket_lo[R] = NB;
    // longest stretch a candidate can block past its own start (reach - pos), over all ranges and types; bucket classes
    c->maxspan = 2; c->any_small = 0; c->any_large = 0;
    for (const Range& g : c->h_ranges) {
        for (int t = 0; t < 7; ++t) {
            const int64_t len = (t == T_SN || t == T_IN || t == T_TLI) ? 1 : g.maxlen[t];
            c->maxspan = std::max<int64_t>(c->maxspan, len + c->block[t] + 1);
        }
        if (g.nb == 1u && g.k <= (uint32_t)SMALL_BUCKET) c->any_small = 1; else c->any_large = 1;
    }
    if (K >= (int64_t)0x7FFFFFF0) MS_FAIL(c, MS_ERR_LIMIT, "more than 2^31 candidates in one call");
    c->n_ranges = R; c->n_candidates = K; c->n_buckets = NB; c->min_dist = min_dist;
    c->split_levels = (int)max_top; c->n_big = (int32_t)big.size();
    MS_CUDA(c, c->big_ranges.ensure(big.size() * 4 + 16));
    if (!big.empty()) MS_CUDA(c, cudaMemcpyAsync(c->big_ranges.p, big.data(), big.size() * 4, cudaMemcpyHostToDevice, c->stream));
    const size_t bytes = sizeof(Range) * (size_t)R + 2 * sizeof(int64_t) * (size_t)(R + 1) + sizeof(Seed) * (size_t)R + 64;
    MS_CUDA(c, c->ranges.ensure(bytes));
    uint8_t* base = c->ranges.as<uint8_t>();
    cudaStream_t st = c->stream;
    if (R > 0) MS_CUDA(c, cudaMemcpyAsync(base, c->h_ranges.data(), sizeof(Range) * (size_t)R, cudaMemcpyHostToDevice, st));
    int64_t* d_cand_lo = reinterpret_cast<int64_t*>(base + sizeof(Range) * (size_t)R);
    MS_CUDA(c, cudaMemcpyAsync(d_cand_lo, cand_lo.data(), sizeof(int64_t) * (size_t)(R + 1), cudaMemcpyHostToDevice, st));
    MS_CUDA(c, cudaMemcpyAsync(d_cand_lo + (R + 1), bucket_lo.data(), sizeof(int64_t) * (size_t)(R + 1), cudaMemcpyHostToDevice, st));
    int32_t* d_block = reinterpret_cast<int32_t*>(reinterpret_cast<Seed*>(d_cand_lo + 2 * (R + 1)) + R);
    MS_CUDA(c, cudaMemcpyAsync(d_block, c->block, sizeof(int32_t) * 7, cudaMemcpyHostToDevice, st));
    std::vector<BucketInfo> br((size_t)NB + 1, BucketInfo{});   // per sort bucket: range and value span
    for (int32_t r = 0; r < R; ++r) {
        const Range& g = c->h_ranges[r];
        const uint64_t sc = g.bscale;
        for (uint64_t bl = 0; bl < g.nb; ++bl) {
            // values of bucket bl: mulhi32(v, bscale) == bl  <=>  ceil(bl * 2^32 / bscale) <= v < ceil((bl + 1) * 2^32 / bscale)
            const uint64_t vlo = (g.nb == 1u || bl == 0) ? 0ull : ((bl << 32) + sc - 1) / sc;
            const uint64_t vhi = (g.nb == 1u || bl + 1 == g.nb) ? (uint64_t)g.n : (((bl + 1) << 32) + sc - 1) / sc;
            BucketInfo& bi = br[(size_t)(bucket_lo[r] + (int64_t)bl)];
            bi.ridx = (uint32_t)r; bi.vlo = (uint32_t)vlo; bi.width = (uint32_t)(vhi - vlo); bi.nw = (uint32_t)((vhi - vlo + 31) >> 5);
        }
    }
    MS_CUDA(c, c->bucket_range.ensure(br.size() * sizeof(BucketInfo)));
    MS_CUDA(c, cudaMemcpyAsync(c->bucket_range.p, br.data(), br.size() * sizeof(BucketInfo), cudaMemcpyHostToDevice, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    return MS_OK;
}

}  // namespace ms

using namespace ms;

extern "C" {

int ms_set_ranges(ms_ctx* c, const ms_range* ranges, int32_t n_ranges, const int32_t* block, int32_t min_dist, double p_ti) {
    if (!c || n_ranges < 0 || (n_ranges > 0 && !ranges) || !block) return MS_ERR_ARG;
    if (c->n_contigs <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_set_ranges: upload a genome first");
    if (min_dist < 0) MS_FAIL(c, MS_ERR_ARG, "min_dist must be >= 0");
    MS_CUDA(c, cudaSetDevice(c->device));
    for (int t = 0; t < 7; ++t) c->block[t] = block[t];
    c->p_ti = p_ti;
    c->h_ranges.clear();
    c->n_ranges = -1;
    for (int32_t r = 0; r < n_ranges; ++r) {
        const ms_range& in = ranges[r];
        if (in.contig >= (uint32_t)c->n_contigs) MS_FAIL(c, MS_ERR_ARG, "range %d: contig out of range", r);
        const int64_t L = c->h_contigs[in.contig].len;
        if (in.stop < in.start || (int64_t)in.stop > L) MS_FAIL(c, MS_ERR_ARG, "range %d: %u-%u outside contig of length %lld", r, in.start, in.stop, (long long)L);
        if (r && (in.contig < ranges[r - 1].contig || (in.contig == ranges[r - 1].contig && in.start <= ranges[r - 1].stop)))
            MS_FAIL(c, MS_ERR_ARG, "range %d: ranges must be sorted by (contig, start) and must not overlap", r);
        if (in.k == 0) continue;  // random.sample(population, 0) == []
        Range g{};
        g.contig = in.contig; g.start = in.start; g.stop = in.stop; g.k = in.k;
        g.limit = (in.limit > 0 && in.limit <= L) ? in.limit : L;
        for (int t = 0; t < 7; ++t) {
            g.cdf[t] = in.cdf[t]; g.minlen[t] = in.minlen[t]; g.maxlen[t] = in.maxlen[t];
            if (g.maxlen[t] < g.minlen[t] || g.minlen[t] < 0) MS_FAIL(c, MS_ERR_ARG, "range %d: bad length bounds for type %d", r, t);
        }
        c->h_ranges.push_back(g);
    }
    return upload_ranges(c, min_dist, c->h_contigs);
}

int ms_sample(ms_ctx* c, uint64_t seed) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    chain_invalidate(c);
    genotype_clear(c);
    return sample_pipeline(c, seed);
}

int ms_sample_positions(ms_ctx* c, uint64_t seed, int32_t n, const uint32_t* gid, const uint32_t* start, const uint32_t* stop,
                        const uint32_t* k, int32_t min_dist, uint32_t* out) {
    if (!c || n < 0 || (n > 0 && (!gid || !start || !stop || !k || !out)) || min_dist < 0) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    // a private contig table: one pseudo contig per range, long enough to hold it
    std::vector<Contig> ctg((size_t)n);
    c->h_ranges.clear();
    c->n_ranges = -1;
    int64_t off = 0;
    for (int32_t i = 0; i < n; ++i) {
        Contig& q = ctg[i];
        q = Contig{};
        q.goff = off; q.len = (int64_t)stop[i] + 1; q.gid = gid[i]; q.bpl = 60;
        off += q.len;
        if (k[i] == 0) continue;
        Range g{};
        g.contig = (uint32_t)i; g.start = start[i]; g.stop = stop[i]; g.k = k[i]; g.limit = q.len;
        for (int t = 0; t < 7; ++t) { g.cdf[t] = 1.0; g.minlen[t] = 1; g.maxlen[t] = 1; }
        c->h_ranges.push_back(g);
    }
    int rc = upload_ranges(c, min_dist, ctg);
    if (rc) { c->n_ranges = -1; return rc; }
    const int64_t K = c->n_candidates;
    if (K == 0) { c->n_ranges = -1; return MS_OK; }
    MS_CUDA(c, c->tmp_contigs.ensure(sizeof(Contig) * (size_t)n));
    MS_CUDA(c, cudaMemcpyAsync(c->tmp_contigs.p, ctg.data(), sizeof(Contig) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaMemsetAsync(c->totals.p, 0, sizeof(Totals), c->stream));
    rc = draw_and_sort(c, make_seed(seed), P_IT_KEY, min_dist, 1, c->tmp_contigs.as<Contig>());
    c->n_ranges = -1;  // the range table now holds position-only ranges: ms_sample needs ms_set_ranges again
    if (rc) return rc;
    std::vector<int64_t> gpos((size_t)K);
    MS_CUDA(c, cudaMemcpyAsync(gpos.data(), c->svec.p, (size_t)K * 8, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaMemcpyAsync(c->h_totals, c->totals.p, sizeof(Totals), cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));   // also keeps ctg alive until the async copy is done
    if (c->h_totals->error) MS_FAIL(c, (int)c->h_totals->error, "ms_sample_positions: kernel error %lld", (long long)c->h_totals->error);
    int64_t s = 0;
    for (int32_t i = 0; i < n; ++i) {
        for (uint32_t j = 0; j < k[i]; ++j) out[s + j] = (uint32_t)(gpos[(size_t)(s + j)] - ctg[i].goff);
        s += k[i];
    }
    return MS_OK;
}

int ms_it_breakpoints(ms_ctx* c, uint64_t seed, int32_t n_pairs, const uint32_t* contig_a, const uint32_t* contig_b,
                      const uint32_t* n, uint32_t* bp_a, uint32_t* bp_b) {
    if (!c || n_pairs < 0 || !contig_a || !contig_b || !n || !bp_a || !bp_b) return MS_ERR_ARG;
    if (c->n_contigs <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_it_breakpoints: upload a genome first");
    // pair-major: all of a's breakpoints, then all of b's: sample_with_minimum_distance(1, len, n, 1) each (it_mutator.py:108-111)
    std::vector<uint32_t> gid, start, stop, k;
    int64_t total = 0;
    for (int32_t p = 0; p < n_pairs; ++p) {
        for (int side = 0; side < 2; ++side) {
            const uint32_t ci = side ? contig_b[p] : contig_a[p];
            if (ci >= (uint32_t)c->n_contigs) MS_FAIL(c, MS_ERR_ARG, "pair %d: contig out of range", p);
            gid.push_back(c->h_contigs[ci].gid); start.push_back(1u); stop.push_back((uint32_t)c->h_contigs[ci].len); k.push_back(n[p]);
        }
        total += n[p];
    }
    std::vector<uint32_t> out((size_t)(2 * total) + 1);
    int rc = ms_sample_positions(c, seed, (int32_t)gid.size(), gid.data(), start.data(), stop.data(), k.data(), 1, out.data());
    if (rc) return rc;
    int64_t s = 0, o = 0;
    for (int32_t p = 0; p < n_pairs; ++p) {
        for (uint32_t i = 0; i < n[p]; ++i) bp_a[o + i] = out[(size_t)(s + i)];
        s += n[p];
        for (uint32_t i = 0; i < n[p]; ++i) bp_b[o + i] = out[(size_t)(s + i)];
        s += n[p];
        o += n[p];
    }
    return MS_OK;
}

int ms_debug_candidates(ms_ctx* c, int64_t cap, int64_t* gpos, uint8_t* type, uint32_t* len, uint8_t* accept, int64_t* n) {
    if (!c || !n) return MS_ERR_ARG;
    *n = c->n_candidates;
    if (cap < c->n_candidates) return MS_OK;
    const size_t K = (size_t)c->n_candidates;
    MS_CUDA(c, cudaSetDevice(c->device));
    if (gpos) MS_CUDA(c, cudaMemcpyAsync(gpos, c->svec.p, K * 8, cudaMemcpyDeviceToHost, c->stream));
    if (type) MS_CUDA(c, cudaMemcpyAsync(type, c->cand_type.p, K, cudaMemcpyDeviceToHost, c->stream));
    if (len) MS_CUDA(c, cudaMemcpyAsync(len, c->cand_len.p, K * 4, cudaMemcpyDeviceToHost, c->stream));
    if (accept) MS_CUDA(c, cudaMemcpyAsync(accept, c->cand_accept.p, K, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    return MS_OK;
}

}  // extern "C"
