// Host build of ms_bgzf_core.h for tests/test_bgzf_core.py (g++, no CUDA).
#include <stdint.h>
#include "../../mutation_simulator_b200/csrc/ms_bgzf_core.h"

using namespace ms::bgzf;

extern "C" {

int bgzf_max_member(void) { return MAX_MEMBER; }

// one BGZF member for in[0..n), n <= 16384; returns its size
int bgzf_encode_member(const uint8_t* in, int n, uint8_t* dst) { return encode_member(in, n, dst); }

// 1 when the block would take the stored fallback
int bgzf_is_stored(const uint8_t* in, int n) {
    static BlockCode bc;
    for (int s = 0; s < 256; ++s) bc.freq[s] = 0;
    for (int i = 0; i < n; ++i) bc.freq[in[i]]++;
    plan_block(bc, n);
    return bc.stored;
}

// code lengths of the length-limited Huffman code for freq[0..nsym), nsym <= 257
void bgzf_huff_lengths(const uint32_t* freq, int nsym, int limit, uint32_t* len) {
    uint16_t sym[NLIT + 1];
    uint32_t w[NLIT + 1], out[NLIT + 1];
    huff_lengths(freq, nsym, limit, out, sym, w);
    for (int s = 0; s < nsym; ++s) len[s] = (uint32_t)code_len(out[s]);
}

uint32_t bgzf_crc32(const uint8_t* p, int64_t n) { return crc32_bytes(p, n); }

uint32_t bgzf_crc32_combine(uint32_t a, uint32_t b, uint64_t len_b) { return crc32_combine(a, b, len_b); }

// the device kernel's CRC: raw (init 0, no final xor) register over the data, finished with crc32_finish
uint32_t bgzf_crc32_raw_finish(const uint8_t* p, int64_t n) {
    uint32_t raw = 0;
    for (int64_t i = 0; i < n; ++i) raw = crc_table_entry((raw ^ p[i]) & 0xff) ^ (raw >> 8);
    return crc32_finish(raw, (uint64_t)n);
}

}  // extern "C"
