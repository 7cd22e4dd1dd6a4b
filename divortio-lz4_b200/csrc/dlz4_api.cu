// dlz4_api.cu -- C ABI (include/dlz4_b200.h) over the sm_100a kernels in dlz4_kernels.cuh.
// Host code here only moves bytes, launches kernels and writes the frame header/footer; every block is
// compressed, decoded and hashed on the GPU.  There is no CPU path.
#include "../../include/dlz4_b200.h"
#include "dlz4_kernels.cuh"
#include "dlz4_frames.cuh"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <functional>
#include <mutex>
#include <thread>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace dlz4;

#include "api_ctx.inc"
#include "api_launch.inc"
#include "api_segments.inc"
#include "api_jump.inc"
int launch_chain(dlz4_ctx *ctx, const uint8_t *work, int32_t start, int32_t total, int32_t block, uint32_t nblocks,
                 int32_t *table_io, uint8_t *dst, uint64_t stride, uint32_t *comp_len, cudaStream_t st) {
    k_compress_chain<<<1, 32, kHashEntries * 4 + kRingBytes, st>>>(work, start, total, block, nblocks, table_io, dst, stride, comp_len);
    ctx->launches++;
    CK(cudaGetLastError());
    return DLZ4_OK;
}

}  // namespace

// =====================================================================================================
extern "C" {

#include "api_lifecycle.inc"
#include "api_batch.inc"
#include "api_xxh32.inc"
#include "api_frame_compress.inc"
#include "api_frame_decompress.inc"
#include "api_frame_batch.inc"
#include "api_frame_dev.inc"
#include "api_frames_dev.inc"
#include "api_stream.inc"
}  // extern "C"
