// pixel selection for new keyframes (ps_select.cu), shared with the C ABI in ct_kernels.cu
#pragma once
#include "../../include/dmvio_b200.h"
#include <cuda_runtime.h>
#include <cstdint>
namespace dmv {
// device buffers of the selector of one coarse-tracker handle, allocated on first use for its level-0 size
struct PSState {
  int w = 0, h = 0;
  float* ag[3] = {nullptr, nullptr, nullptr};  // absSquaredGrad of levels 0..2
  float *ths = nullptr, *thsSmoothed = nullptr;
  uint8_t* rp = nullptr;                        // PixelSelector::randomPattern, w*h bytes
  uint16_t* mask = nullptr;                     // per pot-cell, in select()'s walk order: bit d = the cell gets a level-0 pick with directions[d]
  int* n2start = nullptr;                       // per pot-cell, in walk order: n2 when select() enters the cell
  float* map = nullptr;                         // map_out, w*h
  int* rowcnt = nullptr;                        // per row of level 0
  int* d_cnt = nullptr;                         // [n2, n3, n4, removed by the sub-sample, compacted, n2 of the chain, -, -]
  int* h_cnt = nullptr;                         // pinned copy of d_cnt
};
int ps_alloc(PSState& S, int w, int h);
void ps_free(PSState& S);
// PixelSelector::makeMaps (PixelSelector2.cpp:L94-454) on the resident frame img[0..2] ({I, dx, dy, 0} planes); the map stays in S.map.
// *launches counts kernel launches; one read-back of the pick counts per select() pass.
int ps_make_maps(PSState& S, const float4* const img[3], const dmv_ps_args& a, cudaStream_t st, long long* launches, dmv_ps_result* r);
// FullSystem::makeNewTraces' pixel loop (FullSystem.cpp:L1652-1664): the non-zero pixels of S.map with x, y in [pad+1, dim-pad-2), compacted in
// raster order into u, v (int) and type (float); *n = their count (one read-back)
int ps_compact(PSState& S, int pad, int* u, int* v, float* type, cudaStream_t st, long long* launches, int* n);
}  // namespace dmv
