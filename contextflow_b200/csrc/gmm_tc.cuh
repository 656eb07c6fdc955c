// Interface of the tensor-core Gaussian-mixture kernel (gmm_tc.cu) to gmm_tile.cu, which buckets, routes and finishes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cfpp {
namespace gtc {

constexpr int TS = 128;                 // samples per tile (MMA M)

struct Args {
  const float* x; int64_t x_bstride;
  const float2* PT; const float* LB;                             // gmm_tile.cu's table: [Vs][EP][MKP] (mu, a), [Vs][MKP] LB
  const int* perm; const int* tile_vs; const int* n_tiles;       // bucketing at TS (NULL: identity order, no context)
  int key_div, scale_in_low;
  const float* mtab; int mwidth, moff;
  float* part; int* flags;                                       // [nsplit][slots][MKP] partial sums, [nsplit][tiles] guard flags
  int has_logp;
  int B, K, MK, MKP, N, D, HW, E, EP, esplit, nsplit, slots, tiles;
};

int n_of(int MK);                                                // N: components padded to 16 (<= 128)
int splits_for(int B, int n_keys, int E, int MK);                // slices of e per tile
int launch(const Args& a, cudaStream_t st);

}  // namespace gtc
}  // namespace cfpp
