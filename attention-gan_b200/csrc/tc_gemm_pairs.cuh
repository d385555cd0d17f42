// Pair-list instantiation of the tensor-core GEMM (tc_gemm.cu), used by the pair-list backward (damsm_tc.cu).
#pragma once
#include "tc_common.cuh"

namespace agb {
namespace tc {

// Pair-list extensions (agb_damsm_pairs_bwd), a kernel instantiation of their own:
//   koff != null: batch z reduces only the 128-row tiles [koff[z], koff[z+1]) clipped to [kt0, kt0 + kct), i.e. the
//                 K rows (koff[z] - kt0) * 128 ... of the tile window; a batch with an empty range writes zeros
//                 (accumulate == 0) or nothing (accumulate != 0)
//   bsel != null: batch z is word tile dyn_t0 + z; its B operand is batch bsel[dyn_t0 + z] of map B, and z at or
//                 beyond *dyn_tiles does nothing
struct TcGemmPairArgs : TcGemmArgs {
  const int32_t* koff;
  const int32_t* bsel;
  int kt0, kct;
};
int tc_gemm_pairs(const TcGemmPairArgs& g, const CUtensorMap& mapA, const CUtensorMap& mapB, const CUtensorMap& mapA2,
                  const CUtensorMap& mapB2, int batch, cudaStream_t st);

}  // namespace tc
}  // namespace agb
