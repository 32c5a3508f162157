// TEST HARNESS, not product code: runs the BGZF encoder's phases (tagdigger_b200/csrc/tdg_bgzf.cuh)
// on the CPU, one "thread" after the other between the kernel's barriers, so that the code the GPU
// executes per member can be held to zlib without a GPU.  Built by tests/bgzf_check.py.
#include <cstdint>
#include <cstring>
#include <memory>
#include <vector>

#include <zlib.h>

#include "../../tagdigger_b200/csrc/tdg_bgzf.cuh"

using namespace tdg::bz;

extern "C" {

// code lengths of bz::huff_lengths for freq[0..n) (freq is updated with the codes it adds)
int bzc_huff_lengths(uint32_t *freq, uint32_t n, uint32_t maxbits, uint8_t *len)
{
    std::vector<uint32_t> scratch(2 * n + 2);
    huff_lengths(freq, n, maxbits, len, scratch.data());
    return 0;
}

// One member of n <= 65,280 bytes, as bgzf_deflate writes it, into out (>= n + 64 bytes).  m: the
// per-position matches to use (len << 16 | (dist - 1), 0 = literal) instead of the encoder's own
// search, or null.  info[0] = 1 when the block is dynamic.  Returns the member's size.
long long bzc_member(const uint8_t *in, uint32_t n, const uint32_t *m, uint8_t *out, uint32_t *info)
{
    if (n > BLOCK) return -1;
    if (n == 0) {
        for (uint32_t i = 0; i < EOF_BYTES; i++) out[i] = eof_byte(i);
        info[0] = 0;
        return EOF_BYTES;
    }
    std::unique_ptr<Shared> sp(new Shared());
    Shared &s = *sp;
    std::vector<uint32_t> match(n + 1, 0);
    Job j;
    j.src0 = in;
    j.len0 = n / 3;                      // two sources, as for a member that starts in a pending tail
    j.src1 = in + n / 3;
    j.len1 = n - n / 3;
    j.n = n;
    j.m = match.data();
    j.out = out;
    for (uint32_t t = 0; t < THREADS; t++) phase_load(s, j, t);
    if (m) {
        memcpy(match.data(), m, (size_t)n * 4);
    } else {
        for (uint32_t ws = 0; ws < n; ws += THREADS) {
            for (uint32_t t = 0; t < THREADS; t++) phase_find(s, j, ws, t);
            for (uint32_t t = 0; t < THREADS; t++) phase_insert(s, j, ws, t);
        }
    }
    for (uint32_t t = 0; t < THREADS; t++) phase_walk(s, j, t);
    phase_join(s, j);
    for (uint32_t t = 0; t < THREADS; t++) phase_hist(s, j, t);
    phase_tree(s, 0);
    phase_tree(s, 1);
    phase_header(s);
    for (uint32_t t = 0; t < THREADS; t++) phase_seg_bits(s, j, t);
    phase_scan(s, j);
    for (uint32_t t = 0; t < THREADS; t++) phase_emit(s, j, t);
    const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), in, n);
    info[0] = s.dynamic;
    return write_frame(out, data_bytes(s, j), crc, n);
}

}  // extern "C"
