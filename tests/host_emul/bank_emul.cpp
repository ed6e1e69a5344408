// Shared-memory addresses of the stream kernel's table reads, from the same header functions the kernel
// uses (kmer_core.cuh: SmemLayout).  Built with g++ by tests/test_host_banks.py, which models the banks.
#include <stdint.h>

#include "../../hymet_b200/csrc/kmer_core.cuh"

template <class Lay>
static void addrs(int k, const uint64_t *ct, int word, uint32_t lut, uint32_t *out)
{
    for (uint32_t lane = 0; lane < 32; lane++)
        out[lane] = word < 0 ? Lay::tail_addr(ct[lane], k, Lay::tail_base(lut, lane)) + 2 * Lay::kBytes
                             : Lay::word_addr(ct[lane], word, k, Lay::lane_base(lut, lane), Lay::kStride);
}

extern "C" {
// copies = 16: the layout of the screen kernels (16 lane copies, 2 tail copies); copies = 8: 8 lane copies,
// one tail copy (the probe-everything kernel's premultiplied tables).  word < 0 asks for the tail entry.
// out[lane] = shared address of lane's read for the top-aligned k-mers ct[0..31], table window at lut.
int lane_addrs(int copies, int k, const uint64_t *ct, int word, uint32_t lut, uint32_t *out)
{
    if (copies == 16) addrs<hs::SmemLayout<16, 2>>(k, ct, word, lut, out);
    else if (copies == 8) addrs<hs::SmemLayout<8, 1>>(k, ct, word, lut, out);
    else return -1;
    return 0;
}
uint32_t table_bytes(int copies) { return copies == 16 ? hs::SmemLayout<16, 2>::kBytes : hs::SmemLayout<8, 1>::kBytes; }
uint32_t word_index(uint64_t ct, int i, int k) { return hs::top_word_index(ct, i, k, 0); }
}
