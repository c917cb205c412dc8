// Pixel selection for new keyframes on the device: PixelSelector::makeHists / select / makeMaps (FullSystem/PixelSelector2.cpp:L94-454)
// on the frame resident in a coarse-tracker handle, and the pixel loop of FullSystem::makeNewTraces (FullSystem.cpp:L1640-1665).
//
// Bit-identical to the reference's CPU code: compiled with -fmad=false (no FMA contraction), IEEE sqrtf (makeHists truncates it to an int),
// the reference's operation order everywhere.  select() is one sequential raster walk whose only global dependency is n2, the number of
// pot-cells picked before the current one, which chooses each block's direction (directions[randomPattern[n2] & 0xF]).  It is kept exact
// in three steps per pass (DESIGN.md §5e):
//   ps_mask_kernel     per pot-cell, the 16-bit set of directions for which the cell gets a level-0 pick (written in walk order);
//   ps_chain_kernel    one block: prefix sums over the cells whose outcome is direction-independent (mask 0 or 0xFFFF), one thread walking
//                      only the direction-dependent cells in order to fix n2 -> n2 at the entry of every cell;
//   ps_resolve_kernel  per 4pot block, the reference's loop verbatim with the directions of the n2 values above (including the
//                      bestIdx3 == -2 / bestIdx4 == -2 early-outs, which are local to the block).
#include "../../include/dmvio_b200.h"
#include "common_host.h"
#include "ps_select.h"
#include <cuda_runtime.h>
#include <math.h>
#include <vector>

namespace dmv {

__constant__ float c_dirs[16][2] = {  // PixelSelector2.cpp:L328-344
    {0, 1.0000f},       {0.3827f, 0.9239f}, {0.1951f, 0.9808f}, {0.9239f, 0.3827f},  {0.7071f, 0.7071f}, {0.3827f, -0.9239f},
    {0.8315f, 0.5556f}, {0.8315f, -0.5556f}, {0.5556f, -0.8315f}, {0.9808f, 0.1951f}, {0.9239f, -0.3827f}, {0.7071f, -0.7071f},
    {0.5556f, 0.8315f}, {0.9808f, -0.1951f}, {1.0000f, 0.0000f}, {0.1951f, -0.9808f}};

struct PSGradArgs {
  const float4* img[3];
  float* ag[3];
  int w, h;
  int useB;
  float B[256];
};

// absSquaredGrad of levels 0..2 (HessianBlocks.cpp:L168-188, CalibHessian::getBGradOnly HessianBlocks.h:L394-400); blockIdx.y = level.
// The first and last rows are 0 (the reference leaves them uninitialised).
__global__ void ps_grad_kernel(const __grid_constant__ PSGradArgs A) {
  const int l = blockIdx.y, wl = A.w >> l, hl = A.h >> l;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= wl * hl) return;
  float a = 0.f;
  if (idx >= wl && idx < wl * (hl - 1)) {
    const float4 p = A.img[l][idx];
    a = p.y * p.y + p.z * p.z;
    if (A.useB) {
      int c = (int)(p.x + 0.5f);
      if (c < 5) c = 5;
      if (c > 250) c = 250;
      const float gw = A.B[c + 1] - A.B[c];
      a *= gw * gw;
    }
  }
  A.ag[l][idx] = a;
}

// makeHists' first loop (L106-125): one block of 256 threads per 16x16 block; the 50-bin counts are exact integers
__global__ void __launch_bounds__(256) ps_hist_kernel(const float* __restrict__ ag0, int w, int h, float minGradHistCut, float minGradHistAdd,
                                                      float* __restrict__ ths) {
  __shared__ int hist[91];   // computeHistQuantil reads bins up to 90; the reference clears 50, bins past 49 are taken as 0
  const int tid = threadIdx.x, bx = blockIdx.x, by = blockIdx.y;
  if (tid < 91) hist[tid] = 0;
  __syncthreads();
  const int it = (tid & 15) + 16 * bx, jt = (tid >> 4) + 16 * by;
  if (!(it > w - 2 || jt > h - 2 || it < 1 || jt < 1)) {
    int g = (int)sqrtf(ag0[it + jt * w]);
    if (g > 48) g = 48;
    atomicAdd(&hist[g + 1], 1);
    atomicAdd(&hist[0], 1);
  }
  __syncthreads();
  if (tid == 0) {  // computeHistQuantil (L82-91)
    int th = (int)(hist[0] * minGradHistCut + 0.5f);
    int q = 90;
    for (int i = 0; i < 90; i++) {
      th -= hist[i + 1];
      if (th < 0) { q = i; break; }
    }
    ths[bx + by * gridDim.x] = q + minGradHistAdd;
  }
}

// makeHists' second loop (L127-151): the 3x3 mean of ths, squared, in the reference's summation order
__global__ void ps_smooth_kernel(const float* __restrict__ ths, float* __restrict__ thsSmoothed, int w32, int h32) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w32 * h32) return;
  const int x = i % w32, y = i / w32;
  float sum = 0, num = 0;
  if (x > 0) {
    if (y > 0) { num++; sum += ths[x - 1 + (y - 1) * w32]; }
    if (y < h32 - 1) { num++; sum += ths[x - 1 + (y + 1) * w32]; }
    num++; sum += ths[x - 1 + y * w32];
  }
  if (x < w32 - 1) {
    if (y > 0) { num++; sum += ths[x + 1 + (y - 1) * w32]; }
    if (y < h32 - 1) { num++; sum += ths[x + 1 + (y + 1) * w32]; }
    num++; sum += ths[x + 1 + y * w32];
  }
  if (y > 0) { num++; sum += ths[x + (y - 1) * w32]; }
  if (y < h32 - 1) { num++; sum += ths[x + (y + 1) * w32]; }
  num++; sum += ths[x + y * w32];
  thsSmoothed[i] = (sum / num) * (sum / num);
}

struct PSPass {
  const float4* img0;
  const float *ag0, *ag1, *ag2, *thsSmoothed;
  const uint8_t* rp;
  uint16_t* mask;
  int* n2start;
  float* map;
  int* cnt;
  int w, h, pot, ncx, ncy, nbW;
  float thFactor, dw1, dw2;
  int useDir;
};

// index of pot-cell (cx, cy) in select()'s walk order: 4pot blocks in raster order, their 2pot blocks in raster order, their cells in
// raster order, every block clipped at the image border
__device__ __forceinline__ int ps_walk(int cx, int cy, int ncx, int ncy) {
  const int ch4 = min(4, ncy - (cy & ~3)), cw4 = min(4, ncx - (cx & ~3));
  const int lx = cx & 3, ly = cy & 3, sx = lx >> 1, sy = ly >> 1;
  const int sh = min(2, ch4 - 2 * sy), sw = min(2, cw4 - 2 * sx);
  return ncx * (cy & ~3) + (cx & ~3) * ch4 + cw4 * 2 * sy + 2 * sx * sh + (ly & 1) * sw + (lx & 1);
}

__device__ __forceinline__ bool ps_inside(int xf, int yf, int w, int h) { return !(xf < 4 || xf >= w - 5 || yf < 4 || yf > h - 4); }

// per pot-cell: for which of the 16 directions does select() pick a level-0 pixel in it (some pixel above pixelTH0*thFactor with
// |g . dir| > 0, L393-402)?
__global__ void ps_mask_kernel(const __grid_constant__ PSPass P) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= P.ncx * P.ncy) return;
  const int cx = c % P.ncx, cy = c / P.ncx;
  const int x0 = cx * P.pot, y0 = cy * P.pot, x1 = min(x0 + P.pot, P.w), y1 = min(y0 + P.pot, P.h);
  unsigned m = 0;
  for (int yf = y0; yf < y1 && m != 0xFFFFu; yf++)
    for (int xf = x0; xf < x1; xf++) {
      if (!ps_inside(xf, yf, P.w, P.h)) continue;
      const int idx = xf + P.w * yf;
      const float pixelTH0 = P.thsSmoothed[xf / 16 + (yf / 16) * P.nbW];
      const float ag0 = P.ag0[idx];
      if (!(ag0 > pixelTH0 * P.thFactor)) continue;
      if (!P.useDir) {
        if (ag0 > 0.f) m = 0xFFFFu;
        continue;
      }
      const float4 g = P.img0[idx];
#pragma unroll
      for (int d = 0; d < 16; d++)
        if (fabsf(g.y * c_dirs[d][0] + g.z * c_dirs[d][1]) > 0.f) m |= 1u << d;
    }
  P.mask[ps_walk(cx, cy, P.ncx, P.ncy)] = (uint16_t)m;
}

// exclusive prefix count of f over the block (1024 threads); *total = the block's count
__device__ __forceinline__ int ps_block_scan(bool f, int* total, int* s_warp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned b = __ballot_sync(0xFFFFFFFFu, f);
  if (lane == 0) s_warp[warp] = __popc(b);
  __syncthreads();
  int off = 0, tot = 0;
  for (int i = 0; i < 32; i++) {
    const int v = s_warp[i];
    off += i < warp ? v : 0;
    tot += v;
  }
  __syncthreads();
  *total = tot;
  return off + __popc(b & ((1u << lane) - 1u));
}

// n2 at the entry of every pot-cell (walk order).  Cells with mask 0 / 0xFFFF add 0 / 1 whatever n2 is; the direction-dependent cells are
// walked in order by one thread, chunk by chunk of 1024 cells.
__global__ void __launch_bounds__(1024) ps_chain_kernel(const __grid_constant__ PSPass P) {
  __shared__ int s_warp[32], s_fix[1024];
  __shared__ unsigned s_part[32], s_sel[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, ncell = P.ncx * P.ncy;
  if (tid < 8) P.cnt[tid] = 0;
  int base = 0;
  for (int c0 = 0; c0 < ncell; c0 += 1024) {
    const int k = c0 + tid;
    const unsigned m = k < ncell ? P.mask[k] : 0u;
    const bool fixed1 = m == 0xFFFFu, part = m != 0u && m != 0xFFFFu;
    int tot;
    s_fix[tid] = ps_block_scan(fixed1, &tot, s_warp);
    const unsigned pb = __ballot_sync(0xFFFFFFFFu, part);
    if (lane == 0) s_part[warp] = pb;
    __syncthreads();
    if (tid == 0) {
      int nsel = 0;
      for (int wi = 0; wi < 32; wi++) {
        unsigned b = s_part[wi], sel = 0;
        while (b) {
          const int l = __ffs(b) - 1;
          b &= b - 1;
          const int t = wi * 32 + l;
          const int n2 = base + s_fix[t] + nsel;
          if ((P.mask[c0 + t] >> (P.rp[n2] & 0xF)) & 1u) { sel |= 1u << l; nsel++; }
        }
        s_sel[wi] = sel;
      }
    }
    __syncthreads();
    const bool picked = fixed1 || ((s_sel[warp] >> lane) & 1u);
    const int pre = ps_block_scan(picked, &tot, s_warp);
    if (k < ncell) P.n2start[k] = base + pre;
    base += tot;
  }
  if (tid == 0) P.cnt[5] = base;
}

// select()'s loop (L355-450) for one 4pot block per thread, with the directions the n2 chain gives
__global__ void ps_resolve_kernel(const __grid_constant__ PSPass P) {
  const int pot = P.pot, w = P.w, h = P.h, w1 = w / 2, w2 = w / 4;
  const int nb4x = (P.ncx + 3) / 4, nb4y = (P.ncy + 3) / 4;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb4x * nb4y) return;
  const int x4 = (b % nb4x) * 4 * pot, y4 = (b / nb4x) * 4 * pot;
  auto dir_of = [&](int x, int y) { return P.rp[P.n2start[ps_walk(x / pot, y / pot, P.ncx, P.ncy)]] & 0xF; };
  const int my3 = min(4 * pot, h - y4), mx3 = min(4 * pot, w - x4);
  int bestIdx4 = -1;
  float bestVal4 = 0;
  const int d4 = dir_of(x4, y4);
  for (int y3 = 0; y3 < my3; y3 += 2 * pot)
    for (int x3 = 0; x3 < mx3; x3 += 2 * pot) {
      const int x34 = x3 + x4, y34 = y3 + y4;
      const int my2 = min(2 * pot, h - y34), mx2 = min(2 * pot, w - x34);
      int bestIdx3 = -1;
      float bestVal3 = 0;
      const int d3 = dir_of(x34, y34);
      for (int y2 = 0; y2 < my2; y2 += pot)
        for (int x2 = 0; x2 < mx2; x2 += pot) {
          const int x234 = x2 + x34, y234 = y2 + y34;
          const int my1 = min(pot, h - y234), mx1 = min(pot, w - x234);
          int bestIdx2 = -1;
          float bestVal2 = 0;
          const int d2 = dir_of(x234, y234);
          for (int y1 = 0; y1 < my1; y1++)
            for (int x1 = 0; x1 < mx1; x1++) {
              const int xf = x1 + x234, yf = y1 + y234, idx = xf + w * yf;
              if (!ps_inside(xf, yf, w, h)) continue;
              const float pixelTH0 = P.thsSmoothed[xf / 16 + (yf / 16) * P.nbW];
              const float pixelTH1 = pixelTH0 * P.dw1;
              const float pixelTH2 = pixelTH1 * P.dw2;
              const float ag0 = P.ag0[idx];
              if (ag0 > pixelTH0 * P.thFactor) {
                const float4 g = P.img0[idx];
                const float dn = P.useDir ? fabsf(g.y * c_dirs[d2][0] + g.z * c_dirs[d2][1]) : ag0;
                if (dn > bestVal2) { bestVal2 = dn; bestIdx2 = idx; bestIdx3 = -2; bestIdx4 = -2; }
              }
              if (bestIdx3 == -2) continue;
              const float ag1 = P.ag1[(int)(xf * 0.5f + 0.25f) + (int)(yf * 0.5f + 0.25f) * w1];
              if (ag1 > pixelTH1 * P.thFactor) {
                const float4 g = P.img0[idx];
                const float dn = P.useDir ? fabsf(g.y * c_dirs[d3][0] + g.z * c_dirs[d3][1]) : ag1;
                if (dn > bestVal3) { bestVal3 = dn; bestIdx3 = idx; bestIdx4 = -2; }
              }
              if (bestIdx4 == -2) continue;
              const float ag2 = P.ag2[(int)(xf * 0.25f + 0.125) + (int)(yf * 0.25f + 0.125) * w2];
              if (ag2 > pixelTH2 * P.thFactor) {
                const float4 g = P.img0[idx];
                const float dn = P.useDir ? fabsf(g.y * c_dirs[d4][0] + g.z * c_dirs[d4][1]) : ag2;
                if (dn > bestVal4) { bestVal4 = dn; bestIdx4 = idx; }
              }
            }
          if (bestIdx2 > 0) { P.map[bestIdx2] = 1; bestVal3 = 1e10f; atomicAdd(&P.cnt[0], 1); }
        }
      if (bestIdx3 > 0) { P.map[bestIdx3] = 2; bestVal4 = 1e10f; atomicAdd(&P.cnt[1], 1); }
    }
  if (bestIdx4 > 0) { P.map[bestIdx4] = 4; atomicAdd(&P.cnt[2], 1); }
}

// per row: number of non-zero map pixels, over the whole row (lo = 0, hi = w; sub-sample) or over x in [lo, hi) for rows in [ylo, yhi)
// (makeNewTraces); one block of 128 threads per row.  cnt[4] += the total.
__global__ void __launch_bounds__(128) ps_rowcount_kernel(const float* __restrict__ map, int w, int lo, int hi, int ylo, int yhi, int* rowcnt, int* cnt) {
  __shared__ int s;
  const int y = blockIdx.x;
  if (threadIdx.x == 0) s = 0;
  __syncthreads();
  int n = 0;
  if (y >= ylo && y < yhi)
    for (int x = lo + threadIdx.x; x < hi; x += 128) n += map[x + y * w] != 0.f;
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xFFFFFFFFu, n, o);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(&s, n);
  __syncthreads();
  if (threadIdx.x == 0) { rowcnt[y] = s; if (s) atomicAdd(&cnt[4], s); }
}

// the rank of every counted pixel in image raster order (rows before it, then a scan along its row); mode 0 = the sub-sample of makeMaps
// (L248-265: drop the pixel when randomPattern[rank] > charTH, cnt[3] += dropped), mode 1 = makeNewTraces' compaction into u / v / type
__global__ void __launch_bounds__(128) ps_rowapply_kernel(float* __restrict__ map, int w, int lo, int hi, int ylo, int yhi, const int* __restrict__ rowcnt,
                                                          int mode, const uint8_t* __restrict__ rp, unsigned charTH, int* cnt, int* u, int* v, float* type) {
  __shared__ int s_red[4], s_warp[4];
  const int y = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (y < ylo || y >= yhi || rowcnt[y] == 0) return;
  int off = 0;
  for (int r = tid; r < y; r += 128) off += rowcnt[r];
  for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(0xFFFFFFFFu, off, o);
  if (lane == 0) s_red[warp] = off;
  __syncthreads();
  int rank = s_red[0] + s_red[1] + s_red[2] + s_red[3];
  int dropped = 0;
  for (int x0 = lo; x0 < hi; x0 += 128) {
    const int x = x0 + tid;
    const float m = x < hi ? map[x + y * w] : 0.f;
    const unsigned b = __ballot_sync(0xFFFFFFFFu, m != 0.f);
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    int pre = 0, tot = 0;
    for (int i = 0; i < 4; i++) { pre += i < warp ? s_warp[i] : 0; tot += s_warp[i]; }
    __syncthreads();
    if (m != 0.f) {
      const int rn = rank + pre + __popc(b & ((1u << lane) - 1u));
      if (mode == 0) {
        if (rp[rn] > charTH) { map[x + y * w] = 0.f; dropped++; }
      } else {
        u[rn] = x; v[rn] = y; type[rn] = m;
      }
    }
    rank += tot;
  }
  if (dropped) atomicAdd(&cnt[3], dropped);
}

#define PS_CK(call)                                                                                                   \
  do {                                                                                                                \
    cudaError_t _e = (call);                                                                                          \
    if (_e != cudaSuccess) return set_error(DMV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e));            \
  } while (0)

void ps_free(PSState& S) {
  for (int l = 0; l < 3; l++) cudaFree(S.ag[l]);
  cudaFree(S.ths); cudaFree(S.thsSmoothed); cudaFree(S.rp); cudaFree(S.mask); cudaFree(S.n2start); cudaFree(S.map); cudaFree(S.rowcnt);
  cudaFree(S.d_cnt); cudaFreeHost(S.h_cnt);
  S = PSState();
}

// PixelSelector::PixelSelector (L45-47): std::srand(3141592); rand() & 0xFF.  glibc's rand() restated (TYPE_3 additive generator,
// random_r.c), so that the caller's rand() state is left alone: 31 words seeded by the Park-Miller step, 310 outputs discarded, then
// r[i] = r[i-31] + r[i-3] (mod 2^32), rand() = r[i] >> 1.
static void ps_random_pattern(std::vector<uint8_t>& out) {
  std::vector<uint32_t> r(out.size() + 344);
  int32_t word = 3141592;
  r[0] = (uint32_t)word;
  for (int i = 1; i < 31; i++) {
    const int32_t hi = word / 127773, lo = word % 127773;
    word = 16807 * lo - 2836 * hi;
    if (word < 0) word += 2147483647;
    r[i] = (uint32_t)word;
  }
  for (int i = 31; i < 34; i++) r[i] = r[i - 31];
  for (size_t i = 34; i < r.size(); i++) r[i] = r[i - 31] + r[i - 3];
  for (size_t i = 0; i < out.size(); i++) out[i] = (uint8_t)((r[i + 344] >> 1) & 0xFF);
}

int ps_alloc(PSState& S, int w, int h) {
  if (S.map) return DMV_OK;
  const size_t npx = (size_t)w * h;
  for (int l = 0; l < 3; l++) PS_CK(cudaMalloc(&S.ag[l], sizeof(float) * (npx >> (2 * l))));
  PS_CK(cudaMalloc(&S.ths, sizeof(float) * (w / 16) * (h / 16)));
  PS_CK(cudaMalloc(&S.thsSmoothed, sizeof(float) * (w / 16) * (h / 16)));
  PS_CK(cudaMalloc(&S.rp, npx));
  PS_CK(cudaMalloc(&S.mask, sizeof(uint16_t) * npx));   // at most one pot-cell per pixel (pot = 1)
  PS_CK(cudaMalloc(&S.n2start, sizeof(int) * npx));
  PS_CK(cudaMalloc(&S.rowcnt, sizeof(int) * h));
  PS_CK(cudaMalloc(&S.d_cnt, sizeof(int) * 8));
  PS_CK(cudaMallocHost(&S.h_cnt, sizeof(int) * 8));
  std::vector<uint8_t> rp(npx);
  ps_random_pattern(rp);
  PS_CK(cudaMemcpy(S.rp, rp.data(), npx, cudaMemcpyHostToDevice));
  PS_CK(cudaMalloc(&S.map, sizeof(float) * npx));
  S.w = w; S.h = h;
  return DMV_OK;
}

// one select() pass at potential pot: the map in S.map, (n2, n3, n4) in S.h_cnt[0..2]
static int ps_select_pass(PSState& S, PSPass& P, int pot, cudaStream_t st, long long* launches) {
  P.pot = pot;
  P.ncx = (S.w + pot - 1) / pot; P.ncy = (S.h + pot - 1) / pot;
  const int ncell = P.ncx * P.ncy, nb4 = ((P.ncx + 3) / 4) * ((P.ncy + 3) / 4);
  PS_CK(cudaMemsetAsync(S.map, 0, sizeof(float) * S.w * S.h, st));
  ps_mask_kernel<<<(ncell + 127) / 128, 128, 0, st>>>(P);
  ps_chain_kernel<<<1, 1024, 0, st>>>(P);
  ps_resolve_kernel<<<(nb4 + 63) / 64, 64, 0, st>>>(P);
  *launches += 3;
  PS_CK(cudaGetLastError());
  PS_CK(cudaMemcpyAsync(S.h_cnt, S.d_cnt, sizeof(int) * 8, cudaMemcpyDeviceToHost, st));
  PS_CK(cudaStreamSynchronize(st));
  if (S.h_cnt[0] != S.h_cnt[5]) return set_error(DMV_ERR_CUDA, "pixel selection: %d level-0 picks, but the n2 chain counted %d", S.h_cnt[0], S.h_cnt[5]);
  return DMV_OK;
}

int ps_make_maps(PSState& S, const float4* const img[3], const dmv_ps_args& a, cudaStream_t st, long long* launches, dmv_ps_result* r) {
  const int w = S.w, h = S.h;
  dmv_ps_settings s;
  if (a.settings) s = *a.settings; else dmv_ps_default_settings(&s);
  // makeHists (L94-157) on this frame's absSquaredGrad
  PSGradArgs G;
  for (int l = 0; l < 3; l++) { G.img[l] = img[l]; G.ag[l] = S.ag[l]; }
  G.w = w; G.h = h; G.useB = a.B256 != nullptr;
  for (int i = 0; i < 256; i++) G.B[i] = a.B256 ? a.B256[i] : 0.f;
  ps_grad_kernel<<<dim3((w * h + 255) / 256, 3), 256, 0, st>>>(G);
  ps_hist_kernel<<<dim3(w / 16, h / 16), 256, 0, st>>>(S.ag[0], w, h, s.minGradHistCut, s.minGradHistAdd, S.ths);
  ps_smooth_kernel<<<((w / 16) * (h / 16) + 255) / 256, 256, 0, st>>>(S.ths, S.thsSmoothed, w / 16, h / 16);
  *launches += 3;
  PS_CK(cudaGetLastError());
  PSPass P;
  P.img0 = img[0]; P.ag0 = S.ag[0]; P.ag1 = S.ag[1]; P.ag2 = S.ag[2]; P.thsSmoothed = S.thsSmoothed; P.rp = S.rp;
  P.mask = S.mask; P.n2start = S.n2start; P.map = S.map; P.cnt = S.d_cnt;
  P.w = w; P.h = h; P.nbW = w / 16; P.thFactor = a.thFactor;
  P.dw1 = s.gradDownweightPerLevel; P.dw2 = P.dw1 * P.dw1; P.useDir = s.selectDirectionDistribution != 0;
  // makeMaps' control (L158-265): the recursion needs only n2 + n3 + n4 of each pass
  int currentPotential = a.currentPotential, recursionsLeft = a.recursionsLeft;
  float numHave, quotia;
  int idealPotential;
  for (;;) {
    const int rc = ps_select_pass(S, P, currentPotential, st, launches);
    if (rc != DMV_OK) return rc;
    numHave = S.h_cnt[0] + S.h_cnt[1] + S.h_cnt[2];
    quotia = a.density / numHave;
    const float K = numHave * (currentPotential + 1) * (currentPotential + 1);
    idealPotential = sqrtf(K / a.density) - 1;
    if (idealPotential < 1) idealPotential = 1;
    if (recursionsLeft > 0 && quotia > 1.25 && currentPotential > 1) {
      if (idealPotential >= currentPotential) idealPotential = currentPotential - 1;
    } else if (recursionsLeft > 0 && quotia < 0.25) {
      if (idealPotential <= currentPotential) idealPotential = currentPotential + 1;
    } else {
      break;
    }
    currentPotential = idealPotential;
    recursionsLeft--;
  }
  int numHaveSub = numHave;
  if (quotia < 0.95) {  // sub-sample by randomPattern[rank in raster order]
    const unsigned char charTH = 255 * quotia;
    ps_rowcount_kernel<<<h, 128, 0, st>>>(S.map, w, 0, w, 0, h, S.rowcnt, S.d_cnt);
    ps_rowapply_kernel<<<h, 128, 0, st>>>(S.map, w, 0, w, 0, h, S.rowcnt, 0, S.rp, charTH, S.d_cnt, nullptr, nullptr, nullptr);
    *launches += 2;
    PS_CK(cudaGetLastError());
    PS_CK(cudaMemcpyAsync(S.h_cnt, S.d_cnt, sizeof(int) * 8, cudaMemcpyDeviceToHost, st));
    PS_CK(cudaStreamSynchronize(st));
    numHaveSub -= S.h_cnt[3];
  }
  r->numHaveSub = numHaveSub;
  r->currentPotential = idealPotential;
  return DMV_OK;
}

int ps_compact(PSState& S, int pad, int* u, int* v, float* type, cudaStream_t st, long long* launches, int* n) {
  const int w = S.w, h = S.h, lo = pad + 1, hi = w - pad - 2, ylo = pad + 1, yhi = h - pad - 2;
  PS_CK(cudaMemsetAsync(S.d_cnt + 4, 0, sizeof(int), st));
  ps_rowcount_kernel<<<h, 128, 0, st>>>(S.map, w, lo, hi, ylo, yhi, S.rowcnt, S.d_cnt);
  ps_rowapply_kernel<<<h, 128, 0, st>>>(S.map, w, lo, hi, ylo, yhi, S.rowcnt, 1, S.rp, 0, S.d_cnt, u, v, type);
  *launches += 2;
  PS_CK(cudaGetLastError());
  PS_CK(cudaMemcpyAsync(S.h_cnt + 4, S.d_cnt + 4, sizeof(int), cudaMemcpyDeviceToHost, st));
  PS_CK(cudaStreamSynchronize(st));
  *n = S.h_cnt[4];
  return DMV_OK;
}

}  // namespace dmv

extern "C" void dmv_ps_default_settings(dmv_ps_settings* s) {  // util/settings.cpp:L167-170
  s->minGradHistCut = 0.5f;
  s->minGradHistAdd = 7.f;
  s->gradDownweightPerLevel = 0.75f;
  s->selectDirectionDistribution = 1;
}
