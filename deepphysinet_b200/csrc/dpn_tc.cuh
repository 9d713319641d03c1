// DPN_MODE_BF16 / DPN_MODE_BF16X3: tcgen05 / TMEM / bulk-copy path (see dpn_tc.cu); planes = 1 / 2 bf16 terms per operand.
#pragma once
#include "dpn_fp32.cuh"

namespace dpn {
namespace tc {

constexpr int DEFAULT_POINTS_IN_FLIGHT = 1048576;  // B * chunk * planes: bounds the workspace (~24 KB per point in the split modes, ~13 KB in bf16 mode):
                                                   // the B = 8 x 65 536 configuration runs as ONE pass over a 12.1 GiB workspace

int default_chunk(int B, int planes);              // points per sample per pass (multiple of 128)
size_t workspace_bytes(int chunk, int Kn, int B, int planes);
size_t lattice_workspace_bytes(int chunk, int Kn, int B, int planes);   // the values-only prefix of the carve + lattice staging
int run(const Job& job, cudaStream_t st);

}  // namespace tc
}  // namespace dpn
