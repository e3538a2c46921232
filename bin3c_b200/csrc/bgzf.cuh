// Inflating a table of BGZF blocks on the device (bgzf.cu), shared by the BAM decoder (bamdec.cu) and the stage
// hand-off reader (b3c_bgzf_inflate).
#pragma once

#include "common.cuh"

namespace b3c {

struct BgzfBlocks {
    const uint8_t *comp;              // the compressed blocks
    const int64_t *blocks;            // [3 nb]: offset in comp, BSIZE | ISIZE << 32, offset of the inflated bytes in u
    int32_t nb;
    uint8_t *u;                       // the inflated bytes go to u[0, u_cap)
    int64_t u_cap;
    unsigned long long *err;          // atomicMin of (err_base + the block's u offset) << 8 | code
    int64_t err_base;
    int e_inflate, e_crc;             // codes of a block that does not inflate to ISIZE bytes / fails its CRC-32
};

// k_inflate (one thread per block: raw inflate of inflate.cuh, output size == ISIZE), then k_crc (one warp per block:
// CRC-32 of 32 lane pieces joined with crc32_combine, against the trailer).  Blocks of ISIZE 0 are skipped.
int bgzf_inflate_blocks(const BgzfBlocks &B, cudaStream_t s);

}  // namespace b3c
