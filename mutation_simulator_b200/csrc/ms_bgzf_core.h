// ms_bgzf_core.h — BGZF member encoder shared by the device kernel (ms_bgzf.cu) and the host (VCF header, tests).
//
// A member holds at most one 16 KiB cell of input.  Its deflate stream is one final block: dynamic Huffman with
// literals only (RFC 1951 BTYPE=10, HLIT = 257, HDIST = 1 with one distance code of length 1), or a stored block
// (BTYPE=00) when that is smaller.  Every choice below (symbol order, tie breaks, the length limit repair, the
// run-length coding of the code lengths) is a pure function of the block's histogram, so the serial host encoder
// and the parallel device encoder emit the same bytes.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define MS_BGZF_HD __host__ __device__ __forceinline__
#else
#define MS_BGZF_HD inline
#endif

namespace ms {
namespace bgzf {

constexpr int CELL = 16384;                 // input bytes per member at most (= the splice kernel's output tile)
constexpr int HDR = 18, FTR = 8;            // gzip header with the BC extra subfield; CRC32 + ISIZE
constexpr int MAX_MEMBER = CELL + 5 + HDR + FTR;   // stored fallback: input + 31
constexpr int SLOT = 16448;                 // device scratch bytes per member (>= MAX_MEMBER, multiple of 16)
constexpr int NLIT = 257;                   // literal/length alphabet: bytes 0..255 and end-of-block
constexpr int NCL = 19;                     // code-length alphabet
constexpr int WORDS = (CELL + 5 + 8) / 4 + 4;      // 32-bit words of the deflate bit buffer
constexpr uint32_t CRC_POLY = 0xEDB88320u;  // reflected CRC-32 (gzip)

// order in which the code-length code's lengths are sent (RFC 1951 3.2.7)
MS_BGZF_HD int cl_order(int i) {
    switch (i) {
        case 0: return 16; case 1: return 17; case 2: return 18; case 3: return 0; case 4: return 8; case 5: return 7;
        case 6: return 9; case 7: return 6; case 8: return 10; case 9: return 5; case 10: return 11; case 11: return 4;
        case 12: return 12; case 13: return 3; case 14: return 13; case 15: return 2; case 16: return 14; case 17: return 1;
        default: return 15;
    }
}

// ---- CRC-32 ----------------------------------------------------------------------------------------------------
MS_BGZF_HD uint32_t crc_table_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
    return c;
}

// a * b modulo the CRC polynomial (bit-reflected: bit 31 is x^0), as in zlib's crc32_combine
MS_BGZF_HD uint32_t gf2_mul(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int k = 0; k < 32; ++k) {
        if (a & (0x80000000u >> k)) p ^= b;
        b = (b & 1) ? (b >> 1) ^ CRC_POLY : b >> 1;
    }
    return p;
}

// x^(8 n) modulo the polynomial: the operator that appends n zero bytes to a CRC register
MS_BGZF_HD uint32_t crc_shift_op(uint64_t n) {
    uint32_t p = 0x80000000u;        // x^0
    uint32_t sq = 0x00800000u;       // x^8 (one byte)
    while (n) {
        if (n & 1) p = gf2_mul(sq, p);
        sq = gf2_mul(sq, sq);
        n >>= 1;
    }
    return p;
}

// crc32(A || B) from crc32(A), crc32(B) and |B|
MS_BGZF_HD uint32_t crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b) {
    return gf2_mul(crc_shift_op(len_b), crc_a) ^ crc_b;
}

// the standard CRC-32 of a message whose CRC register, run from 0 without the final xor, ends at `raw`
MS_BGZF_HD uint32_t crc32_finish(uint32_t raw, uint64_t n) {
    return ~(gf2_mul(crc_shift_op(n), 0xFFFFFFFFu) ^ raw);
}

// ---- Huffman code construction -----------------------------------------------------------------------------------
// Code tables hold, per symbol, (length << 16) | code with the code's bits reversed (deflate sends codes MSB first
// into an LSB-first bit stream).
MS_BGZF_HD int code_len(uint32_t lc) { return (int)(lc >> 16); }

// Lengths of a length-limited Huffman code for freq[0..nsym) into out[] (as length << 16; unused symbols 0).
// Symbols are ordered by (frequency, symbol); Moffat & Katajainen's in-place algorithm gives the optimal lengths,
// lengths over `limit` are clamped and the Kraft sum repaired as zlib / miniz do, and the longest lengths go to the
// least frequent symbols.  Fewer than two used symbols are padded with the lowest unused ones (frequency 0), so the
// code is always complete.  sym / w: work arrays of nsym entries.
MS_BGZF_HD void huff_lengths(const uint32_t* freq, int nsym, int limit, uint32_t* out, uint16_t* sym, uint32_t* w) {
    int n = 0;
    for (int s = 0; s < nsym; ++s) {
        out[s] = 0;
        if (freq[s]) { sym[n] = (uint16_t)s; w[n] = freq[s]; ++n; }
    }
    for (int s = 0; n < 2 && s < nsym; ++s)
        if (!freq[s]) { sym[n] = (uint16_t)s; w[n] = 0; ++n; }
    for (int i = 1; i < n; ++i) {       // insertion sort by (w, sym): blocks use few distinct bytes
        const uint16_t s = sym[i];
        const uint32_t f = w[i];
        int j = i - 1;
        while (j >= 0 && (w[j] > f || (w[j] == f && sym[j] > s))) { sym[j + 1] = sym[j]; w[j + 1] = w[j]; --j; }
        sym[j + 1] = s; w[j + 1] = f;
    }
    // Moffat & Katajainen, "In-place calculation of minimum-redundancy codes" (1995): w[] becomes the code lengths
    uint32_t* A = w;
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < n - 1; ++next) {
        if (leaf >= n || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = (uint32_t)next; }
        else A[next] = A[leaf++];
        if (leaf >= n || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = (uint32_t)next; }
        else A[next] += A[leaf++];
    }
    A[n - 2] = 0;
    for (int next = n - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
    int avbl = 1, used = 0, dpth = 0;
    root = n - 2;
    int next = n - 1;
    while (avbl > 0) {
        while (root >= 0 && (int)A[root] == dpth) { ++used; --root; }
        while (avbl > used) { A[next--] = (uint32_t)dpth; --avbl; }
        avbl = 2 * used; ++dpth; used = 0;
    }
    // lengths per count, clamped to the limit, Kraft sum repaired
    uint32_t cnt[16];
    for (int L = 0; L < 16; ++L) cnt[L] = 0;
    for (int i = 0; i < n; ++i) cnt[A[i] > (uint32_t)limit ? limit : A[i]]++;
    uint32_t total = 0;
    for (int L = 1; L <= limit; ++L) total += cnt[L] << (limit - L);
    while (total != (1u << limit)) {
        cnt[limit]--;
        for (int L = limit - 1; L > 0; --L)
            if (cnt[L]) { cnt[L]--; cnt[L + 1] += 2; break; }
        total--;
    }
    int i = 0;
    for (int L = limit; L >= 1; --L)
        for (uint32_t k = 0; k < cnt[L]; ++k) out[sym[i++]] = (uint32_t)L << 16;
}

// canonical codes (RFC 1951 3.2.2) for the lengths in lc[], bit-reversed
MS_BGZF_HD void canonical_codes(uint32_t* lc, int nsym) {
    uint32_t cnt[16], next[16];
    for (int L = 0; L < 16; ++L) cnt[L] = 0;
    for (int s = 0; s < nsym; ++s) cnt[code_len(lc[s])]++;
    cnt[0] = 0;
    uint32_t code = 0;
    for (int L = 1; L < 16; ++L) { code = (code + cnt[L - 1]) << 1; next[L] = code; }
    for (int s = 0; s < nsym; ++s) {
        const int L = code_len(lc[s]);
        if (!L) continue;
        const uint32_t c = next[L]++;
        uint32_t r = 0;
        for (int k = 0; k < L; ++k) r |= ((c >> k) & 1u) << (L - 1 - k);
        lc[s] = ((uint32_t)L << 16) | r;
    }
}

// ---- one block's code and header -------------------------------------------------------------------------------
struct BlockCode {
    uint32_t freq[NLIT];      // byte histogram + end-of-block (filled by the caller for 0..255)
    uint32_t lit[NLIT];       // literal/length code
    uint32_t cl[NCL];         // code-length code
    uint32_t clf[NCL];
    uint16_t sym[NLIT + 1];   // work
    uint32_t w[NLIT + 1];     // work
    uint16_t rle[NLIT + 1];   // code-length symbols (sym | extra << 5)
    int n_rle, hclen;
    uint32_t hdr_bits, data_bits;   // data_bits includes the end-of-block code
    int stored;
};

MS_BGZF_HD int rle_len_at(const uint32_t* lit, int i) { return i < NLIT ? code_len(lit[i]) : 1; }

// Builds both codes for an input of m bytes whose histogram is in bc.freq[0..255]; decides dynamic vs stored.
MS_BGZF_HD void plan_block(BlockCode& bc, int m) {
    bc.freq[256] = 1;
    huff_lengths(bc.freq, NLIT, 15, bc.lit, bc.sym, bc.w);
    canonical_codes(bc.lit, NLIT);
    // the 257 literal/length lengths and the one distance length, run-length coded with 16 / 17 / 18
    int n = 0;
    const int N = NLIT + 1;
    for (int i = 0; i < N;) {
        const int v = rle_len_at(bc.lit, i);
        int run = 1;
        while (i + run < N && rle_len_at(bc.lit, i + run) == v) ++run;
        i += run;
        if (v == 0) {
            while (run >= 11) { const int r = run < 138 ? run : 138; bc.rle[n++] = (uint16_t)(18 | (r - 11) << 5); run -= r; }
            if (run >= 3) { bc.rle[n++] = (uint16_t)(17 | (run - 3) << 5); run = 0; }
            while (run-- > 0) bc.rle[n++] = 0;
        } else {
            bc.rle[n++] = (uint16_t)v;
            --run;
            while (run >= 3) { const int r = run < 6 ? run : 6; bc.rle[n++] = (uint16_t)(16 | (r - 3) << 5); run -= r; }
            while (run-- > 0) bc.rle[n++] = (uint16_t)v;
        }
    }
    bc.n_rle = n;
    for (int s = 0; s < NCL; ++s) bc.clf[s] = 0;
    for (int k = 0; k < n; ++k) bc.clf[bc.rle[k] & 31]++;
    huff_lengths(bc.clf, NCL, 7, bc.cl, bc.sym, bc.w);
    canonical_codes(bc.cl, NCL);
    int hclen = NCL;
    while (hclen > 4 && !code_len(bc.cl[cl_order(hclen - 1)])) --hclen;
    bc.hclen = hclen;
    uint32_t bits = 3 + 5 + 5 + 4 + 3 * (uint32_t)hclen;
    for (int k = 0; k < n; ++k) {
        const int s = bc.rle[k] & 31;
        bits += (uint32_t)code_len(bc.cl[s]) + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
    }
    bc.hdr_bits = bits;
    uint32_t data = 0;
    for (int s = 0; s < NLIT; ++s) data += bc.freq[s] * (uint32_t)code_len(bc.lit[s]);
    bc.data_bits = data;
    bc.stored = (int)((bits + data + 7) / 8) > m + 5;
}

// OR n <= 32 bits of v into the little-endian bit stream w[] at bit position pos (w must be zeroed)
MS_BGZF_HD void or_bits(uint32_t* w, uint32_t pos, uint32_t v, int n) {
    const uint32_t i = pos >> 5, s = pos & 31;
    w[i] |= v << s;
    if (s + (uint32_t)n > 32) w[i + 1] |= v >> (32 - s);
}

// block header (BFINAL=1, BTYPE=10, HLIT/HDIST/HCLEN, both code descriptions); returns its bit length
MS_BGZF_HD uint32_t write_dyn_header(const BlockCode& bc, uint32_t* w) {
    uint32_t p = 0;
    or_bits(w, p, 1u | (2u << 1), 3); p += 3;
    p += 10;                                          // HLIT - 257 = 0, HDIST - 1 = 0
    or_bits(w, p, (uint32_t)(bc.hclen - 4), 4); p += 4;
    for (int k = 0; k < bc.hclen; ++k) { or_bits(w, p, (uint32_t)code_len(bc.cl[cl_order(k)]), 3); p += 3; }
    for (int k = 0; k < bc.n_rle; ++k) {
        const int s = bc.rle[k] & 31;
        const uint32_t c = bc.cl[s];
        or_bits(w, p, c & 0xFFFFu, code_len(c)); p += (uint32_t)code_len(c);
        const int eb = s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0;
        if (eb) { or_bits(w, p, (uint32_t)(bc.rle[k] >> 5), eb); p += (uint32_t)eb; }
    }
    return p;
}

// gzip member header with the BGZF extra subfield (BSIZE = member bytes - 1)
MS_BGZF_HD uint8_t member_header_byte(int i, int member_bytes) {
    switch (i) {
        case 0: return 0x1f; case 1: return 0x8b; case 2: return 8; case 3: return 4;   // ID1 ID2 CM FLG.FEXTRA
        case 9: return 0xff;                                                            // OS unknown (MTIME, XFL = 0)
        case 10: return 6;                                                              // XLEN
        case 12: return 'B'; case 13: return 'C'; case 14: return 2;
        case 16: return (uint8_t)((member_bytes - 1) & 0xff);
        case 17: return (uint8_t)((member_bytes - 1) >> 8);
        default: return 0;
    }
}

// byte j of the stored deflate block of m input bytes (bytes 0..4; the input follows)
MS_BGZF_HD uint8_t stored_head_byte(int j, int m) {
    switch (j) {
        case 0: return 1;                                   // BFINAL=1, BTYPE=00
        case 1: return (uint8_t)(m & 0xff); case 2: return (uint8_t)(m >> 8);
        case 3: return (uint8_t)(~m & 0xff); default: return (uint8_t)((~m >> 8) & 0xff);
    }
}

// ---- serial encoder (host) ---------------------------------------------------------------------------------------
struct CrcTable {
    uint32_t t[256];
    CrcTable() { for (uint32_t i = 0; i < 256; ++i) t[i] = crc_table_entry(i); }
};

inline uint32_t crc32_bytes(const uint8_t* p, int64_t n, uint32_t crc = 0) {
    static const CrcTable tab;
    crc = ~crc;
    for (int64_t i = 0; i < n; ++i) crc = tab.t[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
    return ~crc;
}

// One member for in[0..m), m <= CELL, into dst (>= MAX_MEMBER bytes); returns the member's size.
inline int encode_member(const uint8_t* in, int m, uint8_t* dst) {
    BlockCode bc;
    static thread_local uint32_t w[WORDS];
    for (int s = 0; s < 256; ++s) bc.freq[s] = 0;
    for (int i = 0; i < m; ++i) bc.freq[in[i]]++;
    plan_block(bc, m);
    int dbytes;
    if (bc.stored) {
        for (int j = 0; j < 5; ++j) dst[HDR + j] = stored_head_byte(j, m);
        if (m) memcpy(dst + HDR + 5, in, (size_t)m);
        dbytes = m + 5;
    } else {
        memset(w, 0, sizeof(w));
        uint32_t p = write_dyn_header(bc, w);
        for (int i = 0; i < m; ++i) { const uint32_t c = bc.lit[in[i]]; or_bits(w, p, c & 0xFFFFu, code_len(c)); p += (uint32_t)code_len(c); }
        const uint32_t e = bc.lit[256];
        or_bits(w, p, e & 0xFFFFu, code_len(e)); p += (uint32_t)code_len(e);
        dbytes = (int)((p + 7) / 8);
        for (int j = 0; j < dbytes; ++j) dst[HDR + j] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
    }
    const int total = HDR + dbytes + FTR;
    for (int i = 0; i < HDR; ++i) dst[i] = member_header_byte(i, total);
    const uint32_t crc = crc32_bytes(in, m);
    uint8_t* f = dst + HDR + dbytes;
    for (int k = 0; k < 4; ++k) { f[k] = (uint8_t)(crc >> (8 * k)); f[4 + k] = (uint8_t)((uint32_t)m >> (8 * k)); }
    return total;
}

}  // namespace bgzf
}  // namespace ms
