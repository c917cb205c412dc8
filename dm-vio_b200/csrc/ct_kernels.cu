// sm_100a kernels + C-ABI of the coarse direct-image-alignment path (DESIGN.md §5).
//
//   ct_res_gs_kernel   CoarseTracker::calcRes (CoarseTracker.cpp:L361-517) fused with calcGSSSE (L299-356): one thread per
//                      reference point: project, 4-tap float4 gather from the new frame's level plane, Huber residual,
//                      energy / saturation counters / flow indicators and the 45 unique entries of the weighted 9x9
//                      outer product.  Warp-shuffle + shared-memory block reduction, per-block fp64 partials, and the last
//                      block to finish (threadfence + ticket) folds the partials in a fixed order -> deterministic, one launch.
//                      The buf_warped_* lists of the reference are never materialised.
//   pyr_down_kernel / grad_kernel   FrameHessian::makeImages (HessianBlocks.cpp:L128-191) on the device.
#include "../../include/dmvio_b200.h"
#include "common_host.h"
#include "inv3.h"
#include "ip_trace.h"
#include "ct_depth.h"
#include "ps_select.h"
#include <cmath>
#include <cuda.h>
#include <unordered_map>
#include <algorithm>
#include <cstring>
#include <vector>

namespace dmv {

constexpr int CT_NRED = 45 + 8;  // 45 outer-product entries + E, nE, nSat, nWarped, shiftT, shiftRT, shiftNum, pad
constexpr int CT_THREADS = 256;

struct CTParams {
  float RKi[9], t[3], Ki[9];
  float fx, fy, cx, cy;
  float affa, affb, a_gs, b0;
  float cutoff, huber, maxEnergy;
  int w, h, n, lvl, want_gs;
};

// one reference point: CoarseTracker::calcRes (L399-483) + its row of calcGSSSE (L316-336), added into v[].  The 4 taps are gathered from
// the level plane in global memory (SMEM = false) or from its copy staged in shared memory (SMEM = true).
template <bool SMEM>
__device__ __forceinline__ void ct_eval_point(const CTParams& P, int i, const float x, const float y, const float id, const float refColor,
                                              const float4* __restrict__ img, float v[CT_NRED]) {
  const float p0 = P.RKi[0] * x + P.RKi[1] * y + P.RKi[2] + P.t[0] * id;
  const float p1 = P.RKi[3] * x + P.RKi[4] * y + P.RKi[5] + P.t[1] * id;
  const float p2 = P.RKi[6] * x + P.RKi[7] * y + P.RKi[8] + P.t[2] * id;
  const float u = p0 / p2, vv = p1 / p2;
  const float Ku = P.fx * u + P.cx, Kv = P.fy * vv + P.cy;
  const float new_idepth = id / p2;
  if (P.lvl == 0 && (i & 31) == 0) {  // flow indicators (L416-447)
    const float k0 = P.Ki[0] * x + P.Ki[1] * y + P.Ki[2], k1 = P.Ki[3] * x + P.Ki[4] * y + P.Ki[5], k2 = P.Ki[6] * x + P.Ki[7] * y + P.Ki[8];
    const float T0 = k0 + P.t[0] * id, T1 = k1 + P.t[1] * id, T2 = k2 + P.t[2] * id;
    const float M0 = k0 - P.t[0] * id, M1 = k1 - P.t[1] * id, M2 = k2 - P.t[2] * id;
    const float q0 = P.RKi[0] * x + P.RKi[1] * y + P.RKi[2] - P.t[0] * id;
    const float q1 = P.RKi[3] * x + P.RKi[4] * y + P.RKi[5] - P.t[1] * id;
    const float q2 = P.RKi[6] * x + P.RKi[7] * y + P.RKi[8] - P.t[2] * id;
    const float KuT = P.fx * (T0 / T2) + P.cx, KvT = P.fy * (T1 / T2) + P.cy;
    const float KuT2 = P.fx * (M0 / M2) + P.cx, KvT2 = P.fy * (M1 / M2) + P.cy;
    const float Ku3 = P.fx * (q0 / q2) + P.cx, Kv3 = P.fy * (q1 / q2) + P.cy;
    v[49] += (KuT - x) * (KuT - x) + (KvT - y) * (KvT - y) + (KuT2 - x) * (KuT2 - x) + (KvT2 - y) * (KvT2 - y);
    v[50] += (Ku - x) * (Ku - x) + (Kv - y) * (Kv - y) + (Ku3 - x) * (Ku3 - x) + (Kv3 - y) * (Kv3 - y);
    v[51] += 2.f;
  }
  if (Ku > 2.f && Kv > 2.f && Ku < (float)(P.w - 3) && Kv < (float)(P.h - 3) && new_idepth > 0.f) {
    const int ix = (int)Ku, iy = (int)Kv;
    const float dx = Ku - ix, dy = Kv - iy, dxdy = dx * dy;
    float4 tl, tr, bl, br;
    if constexpr (SMEM) {
      const float4* bp = img + iy * P.w + ix;
      tl = bp[0]; tr = bp[1]; bl = bp[P.w]; br = bp[P.w + 1];
    } else {
      const float4* bp = img + (size_t)iy * P.w + ix;
      tl = __ldg(bp); tr = __ldg(bp + 1); bl = __ldg(bp + P.w); br = __ldg(bp + P.w + 1);
    }
    const float w11 = dxdy, w10 = dy - dxdy, w01 = dx - dxdy, w00 = 1 - dx - dy + dxdy;
    const float h0 = w11 * br.x + w10 * bl.x + w01 * tr.x + w00 * tl.x;
    const float h1 = w11 * br.y + w10 * bl.y + w01 * tr.y + w00 * tl.y;
    const float h2 = w11 * br.z + w10 * bl.z + w01 * tr.z + w00 * tl.z;
    if (isfinite(h0)) {
      const float residual = h0 - (P.affa * refColor + P.affb);
      const float ar = fabsf(residual);
      const float hw = ar < P.huber ? 1.f : P.huber / ar;
      if (ar > P.cutoff) {
        v[45] += P.maxEnergy; v[46] += 1.f; v[47] += 1.f;
      } else {
        v[45] += hw * residual * residual * (2.f - hw); v[46] += 1.f; v[48] += 1.f;
        if (P.want_gs) {  // calcGSSSE row (L316-336) and Accumulator9::updateSSE_eighted (MatrixAccumulators.h:L1091-1166)
          const float gx = h1 * P.fx, gy = h2 * P.fy;
          float J[9];
          J[0] = new_idepth * gx;
          J[1] = new_idepth * gy;
          J[2] = 0.f - new_idepth * (u * gx + vv * gy);
          J[3] = 0.f - ((u * vv) * gx + gy * (1.f + vv * vv));
          J[4] = (u * vv) * gy + gx * (1.f + u * u);
          J[5] = u * gy - vv * gx;
          J[6] = P.a_gs * (P.b0 - refColor);
          J[7] = -1.f;
          J[8] = residual;
          int e = 0;
#pragma unroll
          for (int r = 0; r < 9; r++) {
            const float Jw = J[r] * hw;
#pragma unroll
            for (int c = r; c < 9; c++) v[e++] += Jw * J[c];
          }
        }
      }
    }
  }
}

// block reduction: warp shuffles, then the 8 warp partials through shared memory; thread k < CT_NRED returns the block's sum of v[k] in fp64
__device__ __forceinline__ double ct_block_reduce(const float v[CT_NRED], float (*s_red)[CT_NRED]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < CT_NRED; k++) {
    float a = v[k];
    a += __shfl_xor_sync(0xffffffffu, a, 16);
    a += __shfl_xor_sync(0xffffffffu, a, 8);
    a += __shfl_xor_sync(0xffffffffu, a, 4);
    a += __shfl_xor_sync(0xffffffffu, a, 2);
    a += __shfl_xor_sync(0xffffffffu, a, 1);
    if (lane == 0) s_red[warp][k] = a;
  }
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x < CT_NRED) {
#pragma unroll
    for (int wv = 0; wv < CT_THREADS / 32; wv++) s += (double)s_red[wv][threadIdx.x];
  }
  return s;
}

// fold of the per-CTA fp64 partials in a FIXED order with the loads in flight together: thread (q, k) adds quarter q of the CTAs for
// entry k (independent loads, batches of 8), then thread k adds the four quarter sums.  A plain `for (bk) s += partial[bk]` loop issues
// one L2 round trip per CTA (~0.35 us each, 13 us for 39 CTAs) because every add waits for its own load.
__device__ __forceinline__ void ct_fold(const double* __restrict__ partial, int G, double (*s_q)[CT_NRED], double* s_sum) {
  const int tid = threadIdx.x;
  if (tid < 4 * CT_NRED) {
    const int q = tid / CT_NRED, k = tid - q * CT_NRED;
    const int per = (G + 3) >> 2, b0 = q * per, b1 = min(G, b0 + per);
    double sm = 0.0;
    for (int bk = b0; bk < b1; bk += 8) {
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; u++) v[u] = (bk + u < b1) ? __ldcg(&partial[(size_t)(bk + u) * CT_NRED + k]) : 0.0;
#pragma unroll
      for (int u = 0; u < 8; u++) sm += v[u];
    }
    s_q[q][k] = sm;
  }
  __syncthreads();
  if (tid < CT_NRED) s_sum[tid] = ((s_q[0][tid] + s_q[1][tid]) + s_q[2][tid]) + s_q[3][tid];
}

__global__ void __launch_bounds__(CT_THREADS) ct_res_gs_kernel(CTParams P, const float* __restrict__ pc_u, const float* __restrict__ pc_v,
                                                               const float* __restrict__ pc_id, const float* __restrict__ pc_col,
                                                               const float4* __restrict__ img, double* __restrict__ partial,
                                                               unsigned int* __restrict__ ticket, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float v[CT_NRED];
#pragma unroll
  for (int k = 0; k < CT_NRED; k++) v[k] = 0.f;
  if (i < P.n) ct_eval_point<false>(P, i, pc_u[i], pc_v[i], pc_id[i], pc_col[i], img, v);
  __shared__ float s_red[CT_THREADS / 32][CT_NRED];
  const double bs = ct_block_reduce(v, s_red);
  if (threadIdx.x < CT_NRED) partial[(size_t)blockIdx.x * CT_NRED + threadIdx.x] = bs;
  // ---- last block folds the per-block partials in block order
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int tk = atomicAdd(ticket, 1u);
    s_last = (tk == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {  // block-uniform
    __threadfence();
    __shared__ double s_q[4][CT_NRED];
    __shared__ double s_sum[CT_NRED];
    ct_fold(partial, (int)gridDim.x, s_q, s_sum);
    __syncthreads();
    if (threadIdx.x < CT_NRED) out[threadIdx.x] = s_sum[threadIdx.x];
    if (threadIdx.x == 0) *ticket = 0u;
  }
}

// Vec6 of calcRes (L508-516) and H, b of calcGSSSE (L341-355) from the 53 folded sums o[]: output k < 64 is H[k], 64 <= k < 72 is
// b[k - 64], k == 72 is all of res6.  H and b are divided by the 4-padded warped count (buf_warped_n), then scaled by SCALE_A / SCALE_B.
__host__ __device__ __forceinline__ void ct_finish(const double* o, int k, double* res6, double* H, double* b) {
  const int npad = ((int)o[48] + 3) & ~3;
  const double inv = (double)(1.0f / (float)npad);
  if (k < 72) {
    const int r = (k < 64) ? (k >> 3) : (k - 64), c = (k < 64) ? (k & 7) : 8;   // c = 8: the b column of the 9x9 accumulator
    const int lo = r < c ? r : c, hi = r < c ? c : r;
    const int e = lo * 9 - (lo * (lo - 1)) / 2 + (hi - lo);     // upper-triangular index of the 9x9 accumulator
    const double scr = (r == 6) ? 10.0 : (r == 7 ? 1000.0 : 1.0);
    if (k < 64) {
      const double scc = (c == 6) ? 10.0 : (c == 7 ? 1000.0 : 1.0);
      H[k] = o[e] * inv * scr * scc;
    } else {
      b[r] = o[e] * inv * scr;
    }
  } else if (k == 72) {
    res6[0] = o[45]; res6[1] = o[46];
    res6[2] = (double)((float)o[49] / ((float)o[51] + 0.1f));
    res6[3] = 0;
    res6[4] = (double)((float)o[50] / ((float)o[51] + 0.1f));
    res6[5] = (double)((float)o[47] / (float)o[46]);
  }
}

constexpr int CT_L = DMV_MAX_PYR_LEVELS;
struct CTTrack {
  int coarsest;
  int n[CT_L], w[CT_L], h[CT_L];
  float fx[CT_L], fy[CT_L], cx[CT_L], cy[CT_L];
  float Ki[CT_L][9];
  const float *u[CT_L], *v[CT_L], *id[CT_L], *col[CT_L];
  const float4* img[CT_L];
  double R0[9], t0[3], a0, b0;   // lastToNew_out / aff_g2l_out on entry
  double ref_a, ref_b;           // lastRef_aff_g2l
  float ref_exposure, new_exposure;
  float huber, cutoffTH, affModeA, affModeB;
  double minRes[5];
  double* out;                   // pinned host: R[9] t[3] a b lastResiduals[5] flow[3] good iterations evaluations status point-evaluations
};

struct CTLM {  // the scalar state of trackNewestCoarse, one copy per CTA (shared memory), advanced by thread 0
  double R[9], t[3], a, b;          // refToNew_current, aff_g2l_current
  double Rn[9], tn[3], an, bn;      // candidate
  double H[2][64], bb[2][8], res[2][6];   // [cur]: linearisation at the current pose (resOld); [cur^1]: the evaluation that just finished
  int cur;
  double inc[8];
  double lastResiduals[5], flow[3];
  float RKi[9], tf[3], affLL[2], cutoff;  // operands of the pending evaluation
  float lambda, rep;
  int lvl, iteration, phase, haveRepeated, iterations, evaluations, done, good, status;
  double A[64], rhs[8], Lf[64], Df[8], incs[8], EV[18];   // the damped 8x8 system of the pending LM step, its LDL^T factors, its solution
  double pevals;                  // sum over the evaluations of the level's reference-point count (measurement: algorithmic bytes = 64 B each)
  int need_solve, need_request;   // need_request: 1 = evaluate at (R, t, a, b), 2 = at the candidate (Rn, tn, an, bn) = exp(incs) * (R, t)
};
enum { CT_PH_INIT = 0, CT_PH_LM = 1 };

__device__ void ct_begin_level(CTLM& S) {
  S.rep = 1.f;
  S.phase = CT_PH_INIT;
  S.need_request = 1;
}
// one LM trial step from the current linearisation (L605-683), in three parts: the warp sets up the damped system and factorises it
// (row i of L in lane i: the 8^3/3 multiply-adds and the 28 divisions of the scalar version collapse to 8 dependent column steps), lane 0
// substitutes and updates the pose.  Every element sees the same operations in the same order as the scalar LDL^T: bit-identical result.
// Hl.ldlt().solve(-b) for the 8x8 system (L639-665): plain LDL^T.  A parameter that is not optimised (setting_affineOptModeA/B < 0: the
// reference solves the 6x6 / 7x7 sub-system) is padded with an identity row/column and a zero right-hand side: the extra terms are exact
// zeros, the other components come out bit-identical.
__device__ __forceinline__ void ct_build_system_warp(const CTTrack& T, CTLM& S) {
  const int lane = threadIdx.x & 31;
  const double* Hc = S.H[S.cur];
  const double* bc = S.bb[S.cur];
  const bool fixA = T.affModeA < 0, fixB = T.affModeB < 0;
#pragma unroll
  for (int e = lane; e < 64; e += 32) {
    const int i = e >> 3, j = e & 7;
    const bool fi = (i == 6 && fixA) || (i == 7 && fixB), fj = (j == 6 && fixA) || (j == 7 && fixB);
    double vv = Hc[e];
    if (i == j) vv *= (1 + S.lambda);
    S.A[e] = (fi || fj) ? ((i == j) ? 1.0 : 0.0) : vv;
  }
  if (lane < 8) {
    const bool fi = (lane == 6 && fixA) || (lane == 7 && fixB);
    S.rhs[lane] = fi ? 0.0 : -bc[lane];
  }
}
// LDL^T of S.A by one warp (all 32 lanes execute; lane i & 7 mirrors row i, lanes 0..7 write)
__device__ __forceinline__ void ct_factor_warp(CTLM& S) {
  const int lane = threadIdx.x & 31, i = lane & 7;
  double Ai[8], Li[8], D[8];
#pragma unroll
  for (int k = 0; k < 8; k++) { Ai[k] = S.A[i * 8 + k]; Li[k] = 0.0; }
#pragma unroll
  for (int j = 0; j < 8; j++) {
    double sm = Ai[j];
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (k < j) {
        const double Ljk = __shfl_sync(0xffffffffu, Li[k], j);   // row j's entry (lane j's own row when i == j)
        sm -= Li[k] * Ljk * D[k];
      }
    const double dj = __shfl_sync(0xffffffffu, sm, j);
    D[j] = dj;
    if (i > j) Li[j] = dj != 0.0 ? sm / dj : 0.0;
  }
  if (lane < 8) {
#pragma unroll
    for (int k = 0; k < 8; k++) S.Lf[i * 8 + k] = Li[k];
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < 8; k++) S.Df[k] = D[k];
    }
  }
}
__device__ void ct_propose_post(const CTTrack& T, CTLM& S) {
  double y[8], inc[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    double sm = S.rhs[i];
#pragma unroll
    for (int k = 0; k < 8; k++) if (k < i) sm -= S.Lf[i * 8 + k] * y[k];
    y[i] = sm;
  }
#pragma unroll
  for (int i = 0; i < 8; i++) y[i] = S.Df[i] != 0.0 ? y[i] / S.Df[i] : 0.0;
#pragma unroll
  for (int i = 7; i >= 0; i--) {
    double sm = y[i];
#pragma unroll
    for (int k = 0; k < 8; k++) if (k > i) sm -= S.Lf[k * 8 + i] * inc[k];
    inc[i] = sm;
  }
  float extrapFac = 1;
  const float lambdaExtrapolationLimit = 0.001f;
  if (S.lambda < lambdaExtrapolationLimit) extrapFac = sqrtf(sqrtf(lambdaExtrapolationLimit / S.lambda));
#pragma unroll
  for (int i = 0; i < 8; i++) inc[i] *= extrapFac;
  double incScaled[8];
#pragma unroll
  for (int i = 0; i < 8; i++) incScaled[i] = inc[i];
  incScaled[6] *= 10.0;    // SCALE_A
  incScaled[7] *= 1000.0;  // SCALE_B
  double ssum = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) ssum += incScaled[i];
  if (!isfinite(ssum)) {
#pragma unroll
    for (int i = 0; i < 8; i++) incScaled[i] = 0;
  }
#pragma unroll
  for (int i = 0; i < 8; i++) { S.incs[i] = incScaled[i]; S.inc[i] = inc[i]; }
  S.an = S.a + incScaled[6];
  S.bn = S.b + incScaled[7];
  S.phase = CT_PH_LM;
  S.need_solve = 0;
  S.need_request = 2;   // evaluate at the candidate exp(incs) * (R, t)
}
// SE3::exp(incs) * (R, t) -> (Rn, tn) and the operands of the next calcRes, spread over the lanes of warp 0: every output element is formed
// by exactly the expression of the scalar code, only by a different lane.
__device__ __forceinline__ void ct_pose_request_warp(const CTTrack& T, CTLM& S, const bool from_candidate) {
  const int lane = threadIdx.x & 31;
  if (from_candidate) {
    const double* xi = S.incs;
    const double wx = xi[3], wy = xi[4], wz = xi[5];
    const double th2 = wx * wx + wy * wy + wz * wz, th = sqrt(th2);
    double ca, cb, cc;
    if (th < 1e-8) { ca = 1.0 - th2 / 6.0; cb = 0.5 - th2 / 24.0; cc = 1.0 / 6.0 - th2 / 120.0; }
    else { double sn, cs; sincos(th, &sn, &cs); ca = sn / th; cb = (1.0 - cs) / th2; cc = (th - sn) / (th2 * th); }
    const double W[9] = {0, -wz, wy, wz, 0, -wx, -wy, wx, 0};
    if (lane < 18) {  // lanes 0..8: E = I + ca W + cb W^2, lanes 9..17: V = I + cb W + cc W^2
      const int e = lane % 9, i = e / 3, j = e - 3 * i;
      const double w2 = W[i * 3] * W[j] + W[i * 3 + 1] * W[3 + j] + W[i * 3 + 2] * W[6 + j];
      const double I = (e % 4 == 0) ? 1.0 : 0.0;
      S.EV[lane] = (lane < 9) ? I + ca * W[e] + cb * w2 : I + cb * W[e] + cc * w2;
    }
    __syncwarp();
    const double* E = S.EV;
    const double* V = S.EV + 9;
    if (lane < 9) {
      const int i = lane / 3, j = lane - 3 * i;
      S.Rn[lane] = E[i * 3] * S.R[j] + E[i * 3 + 1] * S.R[3 + j] + E[i * 3 + 2] * S.R[6 + j];
    } else if (lane < 12) {
      const int i = lane - 9;
      const double et = V[i * 3] * xi[0] + V[i * 3 + 1] * xi[1] + V[i * 3 + 2] * xi[2];
      S.tn[i] = E[i * 3] * S.t[0] + E[i * 3 + 1] * S.t[1] + E[i * 3 + 2] * S.t[2] + et;
    }
    __syncwarp();
  }
  // operands of calcRes (CoarseTracker.cpp:L377-379): RKi = R.cast<float>() * Ki[lvl], t.cast<float>(), affLL.cast<float>()
  const double* R = from_candidate ? S.Rn : S.R;
  const double* t = from_candidate ? S.tn : S.t;
  const double a = from_candidate ? S.an : S.a, b = from_candidate ? S.bn : S.b;
  if (lane < 9) {
    const int i = lane / 3, j = lane - 3 * i;
    const float* Ki = T.Ki[S.lvl];
    S.RKi[lane] = (float)R[i * 3] * Ki[j] + (float)R[i * 3 + 1] * Ki[3 + j] + (float)R[i * 3 + 2] * Ki[6 + j];
  } else if (lane < 12) {
    S.tf[lane - 9] = (float)t[lane - 9];
  } else if (lane == 12) {
    float eF = T.ref_exposure, eT = T.new_exposure;  // AffLight::fromToVecExposure (util/NumType.h:L174-186)
    if (eF == 0 || eT == 0) eT = eF = 1;
    const double aa = exp(a - T.ref_a) * eT / eF;
    S.affLL[0] = (float)aa;
    S.affLL[1] = (float)(b - aa * T.ref_b);
    S.cutoff = T.cutoffTH * S.rep;
    S.evaluations++;
    S.pevals += (double)T.n[S.lvl];
  }
}
__device__ void ct_end_level(const CTTrack& T, CTLM& S) {  // L722-745
  const int lvl = S.lvl;
  const double* resOld = S.res[S.cur];
  S.lastResiduals[lvl] = sqrtf((float)(resOld[0] / resOld[1]));
  S.flow[0] = resOld[2]; S.flow[1] = resOld[3]; S.flow[2] = resOld[4];
  if (isnan(S.lastResiduals[lvl]) || S.lastResiduals[lvl] > 1.5 * T.minRes[lvl]) { S.done = 1; S.good = 0; S.status = 2; return; }
  if (S.rep > 1 && !S.haveRepeated) { S.haveRepeated = 1; ct_begin_level(S); return; }  // lvl++ ; continue  => the same level again
  S.lvl = lvl - 1;
  if (S.lvl < 0) {  // L747-769
    S.done = 1;
    bool good = true;
    if ((T.affModeA != 0 && (fabsf((float)S.a) > 1.2f)) || (T.affModeB != 0 && (fabsf((float)S.b) > 200.f))) good = false;
    float eF = T.ref_exposure, eT = T.new_exposure;
    if (eF == 0 || eT == 0) eT = eF = 1;
    const double ra = exp(S.a - T.ref_a) * eT / eF, rb = S.b - ra * T.ref_b;
    if ((T.affModeA == 0 && (fabsf(logf((float)ra)) > 1.5f)) || (T.affModeB == 0 && (fabsf((float)rb) > 200.f))) good = false;
    if (T.affModeA < 0) S.a = 0;
    if (T.affModeB < 0) S.b = 0;
    S.good = good ? 1 : 0;
    return;
  }
  ct_begin_level(S);
}
// thread 0: the evaluation that just finished sits in S.res/H/bb[cur^1] (ct_finish); decide what to evaluate next: the same pose again
// (need_request = 1), an LM step from the current linearisation (need_solve), or the next level
__device__ void ct_advance(const CTTrack& T, CTLM& S) {
  const int maxIterations[5] = {10, 20, 50, 50, 50};
  const int nw = S.cur ^ 1;
  const double* res = S.res[nw];
  if (S.phase == CT_PH_INIT) {  // L566-578: first evaluation of a level, cutoff doubling while too many residuals saturate
    S.cur = nw;                 // this evaluation becomes the current linearisation (resOld, H, b)
    if (res[5] > 0.6 && (S.rep < 50 || res[5] > 0.99)) { S.rep *= 2; S.need_request = 1; return; }
    S.lambda = 0.01f;
    S.iteration = 0;
    if (S.iteration >= maxIterations[S.lvl]) { ct_end_level(T, S); return; }
    S.iterations++;
    S.need_solve = 1;
    return;
  }
  // CT_PH_LM: accept / reject (L686-716)
  const double* resOld = S.res[S.cur];
  const bool accept = (res[0] / res[1]) < (resOld[0] / resOld[1]);
  if (accept) {
    S.cur = nw;  // calcGSSSE at the accepted pose == the H,b of the evaluation that just finished
    S.a = S.an; S.b = S.bn;
    for (int i = 0; i < 9; i++) S.R[i] = S.Rn[i];
    for (int i = 0; i < 3; i++) S.t[i] = S.tn[i];
    S.lambda *= 0.5f;
  } else {
    S.lambda *= 4;
    if (S.lambda < 0.001f) S.lambda = 0.001f;
  }
  double incNorm = 0;
  for (int i = 0; i < 8; i++) incNorm += S.inc[i] * S.inc[i];
  incNorm = sqrt(incNorm);
  S.iteration++;
  if (!(incNorm > 1e-3) || S.iteration >= maxIterations[S.lvl]) { ct_end_level(T, S); return; }
  S.iterations++;
  S.need_solve = 1;
}
// the scalar state machine step, executed by warp 0 of every CTA
__device__ __forceinline__ void ct_advance_warp(const CTTrack& T, CTLM& S) {
  const int lane = threadIdx.x & 31;
  if (lane == 0) { S.need_request = 0; ct_advance(T, S); }
  __syncwarp();
  if (S.need_solve) {  // warp-uniform (shared memory)
    ct_build_system_warp(T, S);
    __syncwarp();
    ct_factor_warp(S);
    __syncwarp();
    if (lane == 0) ct_propose_post(T, S);
    __syncwarp();
  }
  if (S.need_request) ct_pose_request_warp(T, S, S.need_request == 2);
}

// ---------------------------------------------------------------------------------------------------------------------
// ct_track_cluster_kernel — CoarseTracker::trackNewestCoarse (CoarseTracker.cpp:L539-770, visual-only branch L639-683) as ONE persistent
// launch on ONE THREAD-BLOCK CLUSTER (sm_90+ hardware feature): the Levenberg-Marquardt loop over all pyramid levels runs on the device and
// replaces ~21 launch + sync round trips per frame.  One evaluation = every CTA evaluates its points (calcRes + calcGSSSE row, the same
// ct_eval_point as ct_res_gs_kernel), then EVERY CTA folds the cluster's partials in rank order and its warp 0 advances the same scalar
// state machine in double (8x8 LDLT, SE3 exp, accept/reject, level schedule): identical inputs, identical decisions, so no second
// barrier and no broadcast.
//   * the CTAs of the cluster exchange their fp64 partials through DISTRIBUTED SHARED MEMORY (st.shared::cluster into every peer's
//     slot) and meet at the hardware cluster barrier (barrier.cluster.arrive/wait): no global-memory partials, no atomics, no spinning
//     on an L2 counter, a few hundred ns per evaluation;
//   * pyramid levels whose float4 plane fits in shared memory (80x60 at 640x480: 76.8 KB; 64x64 at 512^2; 40x30) are staged ONCE per
//     level by TMA (cp.async.bulk.tensor.2d, multicast to every CTA of the cluster, completion on an mbarrier) and every Levenberg-
//     Marquardt evaluation of that level gathers its 4 taps per point from shared memory instead of L2;
//   * the block reduction of the 53 sums per point is a transposing butterfly (62 shuffles per warp instead of 265);
//   * each thread keeps CTC_SLOTS reference points of the level in registers and streams the rest, so any point count is tracked.
// A sequential LM chain is latency-bound: fewer, closer SMs with a hardware barrier beat a chip-wide software barrier (DESIGN.md §5).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int CTC_THREADS = 512;
constexpr int CTC_SLOTS = 2;                // reference points per thread kept in registers (2 x 16 x 512 = 16384 points per level)
constexpr int CTC_MAXC = 16;                 // CTAs per cluster (8 portable, 16 with the non-portable opt-in)
constexpr int CTC_PLANE_BYTES = 80 * 1024;   // largest level plane staged in shared memory
struct alignas(64) CTMaps { CUtensorMap lvl[CT_L]; };   // level planes as 2-D tensors of 16-byte texels (encoded as pairs of fp64)

struct alignas(128) CTCSmem {
  unsigned char plane[CTC_PLANE_BYTES];      // TMA destination: the staged level, row-major float4
  double xch[2][CTC_MAXC][CT_NRED + 3];      // [parity][source CTA][sum]: written by every CTA of the cluster through DSMEM
  float red[CTC_THREADS / 32][64];           // per-warp sums (transposed butterfly output)
  double s_sum[CT_NRED + 3];
  CTLM S;
  unsigned long long mbar;                   // TMA completion barrier
};

__device__ __forceinline__ unsigned ctc_rank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned ctc_size() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void ctc_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned ctc_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__global__ void __launch_bounds__(CTC_THREADS, 1) ct_track_cluster_kernel(const __grid_constant__ CTTrack T, const __grid_constant__ CTMaps maps) {
  extern __shared__ __align__(128) unsigned char ctc_raw[];
  CTCSmem& M = *reinterpret_cast<CTCSmem*>(ctc_raw);
  CTLM& S = M.S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned rank = ctc_rank(), NC = ctc_size();
  int par = 0, staged_lvl = -1, cached_lvl = -1;
  unsigned mphase = 0;
  float4 pts[CTC_SLOTS];
  if (tid == 0) {
    for (int i = 0; i < 9; i++) S.R[i] = T.R0[i];
    for (int i = 0; i < 3; i++) S.t[i] = T.t0[i];
    S.a = T.a0; S.b = T.b0;
    for (int i = 0; i < 5; i++) S.lastResiduals[i] = __longlong_as_double(0x7ff8000000000000ll);  // NAN
    for (int i = 0; i < 3; i++) S.flow[i] = 1000;
    S.haveRepeated = 0; S.iterations = 0; S.evaluations = 0; S.done = 0; S.good = 0; S.status = 0; S.cur = 0; S.need_solve = 0; S.pevals = 0;
    S.lvl = T.coarsest;
    ct_begin_level(S);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ctc_smem_u32(&M.mbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid < 32) ct_pose_request_warp(T, S, false);
  __syncthreads();
  ctc_cluster_sync();  // every CTA's mbarrier exists before the first multicast copy can signal it
  while (!S.done) {
    const int l = S.lvl;
    // ---- level change: stage the plane with TMA if it fits (one multicast copy issued by CTA 0 lands in every CTA's shared memory)
    const bool fits = (size_t)T.w[l] * T.h[l] * sizeof(float4) <= (size_t)CTC_PLANE_BYTES;
    if (fits && staged_lvl != l) {
      const unsigned bytes = (unsigned)(T.w[l] * T.h[l] * sizeof(float4));
      if (tid == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ctc_smem_u32(&M.mbar)), "r"(bytes) : "memory");
      ctc_cluster_sync();  // all barriers armed (and nobody still reads the previous level's plane)
      if (rank == 0 && tid == 0) {
        const unsigned short mask = (unsigned short)((1u << NC) - 1u);
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
                ctc_smem_u32(M.plane)),
            "l"(&maps.lvl[l]), "r"(ctc_smem_u32(&M.mbar)), "r"(0), "r"(0), "h"(mask)
            : "memory");
      }
      {  // wait for the bytes (try_wait suspends the thread between probes)
        const unsigned mb = ctc_smem_u32(&M.mbar);
        unsigned done = 0;
        while (!done)
          asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(mb), "r"(mphase) : "memory");
      }
      mphase ^= 1u;
      staged_lvl = l;
    }
    // ---- one evaluation: calcRes + calcGSSSE at the requested pose
    CTParams P;
#pragma unroll
    for (int i = 0; i < 9; i++) { P.RKi[i] = S.RKi[i]; P.Ki[i] = T.Ki[l][i]; }
#pragma unroll
    for (int i = 0; i < 3; i++) P.t[i] = S.tf[i];
    P.fx = T.fx[l]; P.fy = T.fy[l]; P.cx = T.cx[l]; P.cy = T.cy[l];
    P.affa = S.affLL[0]; P.affb = S.affLL[1]; P.a_gs = S.affLL[0]; P.b0 = (float)T.ref_b;
    P.cutoff = S.cutoff; P.huber = T.huber; P.maxEnergy = 2 * T.huber * S.cutoff - T.huber * T.huber;
    P.w = T.w[l]; P.h = T.h[l]; P.n = T.n[l]; P.lvl = l; P.want_gs = 1;
    float v[64];
#pragma unroll
    for (int k = 0; k < 64; k++) v[k] = 0.f;
    const int stride = (int)NC * CTC_THREADS, first = (int)rank * CTC_THREADS + tid;
    if (cached_lvl != l) {  // the level's reference points of this thread stay in registers for all evaluations of the level
#pragma unroll
      for (int k = 0; k < CTC_SLOTS; k++) {
        const int i = first + k * stride;
        if (i < P.n) { pts[k] = make_float4(__ldg(T.u[l] + i), __ldg(T.v[l] + i), __ldg(T.id[l] + i), __ldg(T.col[l] + i)); }
      }
      cached_lvl = l;
    }
#pragma unroll
    for (int k = 0; k < CTC_SLOTS; k++) {
      const int i = first + k * stride;
      if (i < P.n) {
        if (fits) ct_eval_point<true>(P, i, pts[k].x, pts[k].y, pts[k].z, pts[k].w, reinterpret_cast<const float4*>(M.plane), v);
        else ct_eval_point<false>(P, i, pts[k].x, pts[k].y, pts[k].z, pts[k].w, T.img[l], v);
      }
    }
    for (int i = first + CTC_SLOTS * stride; i < P.n; i += stride) {  // more points than register slots: stream the rest
      if (fits) ct_eval_point<true>(P, i, __ldg(T.u[l] + i), __ldg(T.v[l] + i), __ldg(T.id[l] + i), __ldg(T.col[l] + i), reinterpret_cast<const float4*>(M.plane), v);
      else ct_eval_point<false>(P, i, __ldg(T.u[l] + i), __ldg(T.v[l] + i), __ldg(T.id[l] + i), __ldg(T.col[l] + i), T.img[l], v);
    }
    // ---- warp: transposing butterfly, lane L ends with the warp sums of entries 2L, 2L+1
    {
      static_assert(CT_NRED <= 64, "");
#pragma unroll
      for (int st2 = 0; st2 < 5; st2++) {
        const int hstep = 32 >> st2, m = 16 >> st2;
        const bool up = (lane & m) != 0;
#pragma unroll
        for (int k = 0; k < 32; k++)
          if (k < hstep) v[k] = (up ? v[k + hstep] : v[k]) + __shfl_xor_sync(0xffffffffu, up ? v[k] : v[k + hstep], m);
      }
      // entry index of v[k] in lane L: 32 b4 + 16 b3 + 8 b2 + 4 b1 + 2 b0 + k = 2 * bitrev-free L' ... = 2 L + k with L's bits in natural order
      M.red[warp][2 * lane] = v[0];
      M.red[warp][2 * lane + 1] = v[1];
    }
    __syncthreads();
    // ---- CTA: fp64 sum over the warps, pushed into EVERY CTA's exchange slot through distributed shared memory
    if (tid < CT_NRED) {
      double sm = 0.0;
#pragma unroll
      for (int wv = 0; wv < CTC_THREADS / 32; wv++) sm += (double)M.red[wv][tid];
      const unsigned local = ctc_smem_u32(&M.xch[par][rank][tid]);
      for (unsigned c = 0; c < NC; c++) {
        unsigned remote;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(c));
        asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(remote), "d"(sm) : "memory");
      }
    }
    ctc_cluster_sync();  // release / acquire at cluster scope: every CTA's partials are visible in every CTA's shared memory
    if (tid < CT_NRED) {
      double sm = 0.0;
      for (unsigned c = 0; c < NC; c++) sm += M.xch[par][c][tid];  // rank order: bit-identical in every CTA
      M.s_sum[tid] = sm;
    }
    par ^= 1;
    __syncthreads();
    ct_finish(M.s_sum, tid, S.res[S.cur ^ 1], S.H[S.cur ^ 1], S.bb[S.cur ^ 1]);
    __syncthreads();
    if (tid < 32) ct_advance_warp(T, S);
    __syncthreads();
  }
  ctc_cluster_sync();  // nobody leaves while a peer may still write into its shared memory
  if (rank == 0 && tid == 0) {  // an aborted track (status 2) returns the input pose and affine parameters, like the reference's early return
    double* o = T.out;
    const bool ok = (S.status == 0);
    for (int i = 0; i < 9; i++) o[i] = ok ? S.R[i] : T.R0[i];
    for (int i = 0; i < 3; i++) o[9 + i] = ok ? S.t[i] : T.t0[i];
    o[12] = ok ? S.a : T.a0; o[13] = ok ? S.b : T.b0;
    for (int i = 0; i < 5; i++) o[14 + i] = S.lastResiduals[i];
    for (int i = 0; i < 3; i++) o[19 + i] = S.flow[i];
    o[22] = S.good; o[23] = S.iterations; o[24] = S.evaluations; o[25] = S.status; o[26] = S.pevals;
  }
}

__global__ void ct_repack_kernel(const float* __restrict__ src, float4* __restrict__ dst, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = make_float4(src[3 * i], src[3 * i + 1], src[3 * i + 2], 0.f);
}
// level l+1 intensity = 2x2 box mean of level l (HessianBlocks.cpp:L159-166)
__global__ void pyr_down_kernel(const float4* __restrict__ src, float* __restrict__ dst, int wl, int hl, int wlm1) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= wl || y >= hl) return;
  const float4* p = src + (size_t)2 * y * wlm1 + 2 * x;
  dst[(size_t)y * wl + x] = 0.25f * (p[0].x + p[1].x + p[wlm1].x + p[wlm1 + 1].x);
}
__global__ void grad_kernel(const float* __restrict__ img, float4* __restrict__ dst, int w, int h) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= w * h) return;
  float dx = 0.f, dy = 0.f;
  if (idx >= w && idx < w * (h - 1)) {
    dx = 0.5f * (img[idx + 1] - img[idx - 1]);
    dy = 0.5f * (img[idx + w] - img[idx - w]);
    if (!isfinite(dx)) dx = 0.f;
    if (!isfinite(dy)) dy = 0.f;
  }
  dst[idx] = make_float4(img[idx], dx, dy, 0.f);
}

}  // namespace dmv

using namespace dmv;

struct dmv_ct {
  dmv_ct_config cfg;
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  bool staging_busy = false;  // an asynchronous upload from h_scratch may be in flight
  bool timing = false;  // CUDA-event timing of every evaluation (dmv_ct_set_timing); off by default: two event records per launch
  int w[DMV_MAX_PYR_LEVELS], h[DMV_MAX_PYR_LEVELS];
  float fx[DMV_MAX_PYR_LEVELS], fy[DMV_MAX_PYR_LEVELS], cx[DMV_MAX_PYR_LEVELS], cy[DMV_MAX_PYR_LEVELS];
  bool haveK[DMV_MAX_PYR_LEVELS];
  float4* d_img[DMV_MAX_PYR_LEVELS] = {nullptr};
  float* d_gray[DMV_MAX_PYR_LEVELS] = {nullptr};
  float* d_stage = nullptr;
  float *d_u[DMV_MAX_PYR_LEVELS] = {nullptr}, *d_v[DMV_MAX_PYR_LEVELS] = {nullptr}, *d_id[DMV_MAX_PYR_LEVELS] = {nullptr},
        *d_col[DMV_MAX_PYR_LEVELS] = {nullptr};
  int n[DMV_MAX_PYR_LEVELS];
  double* d_partial = nullptr;
  unsigned int* d_ticket = nullptr;
  double* d_out = nullptr;
  double* h_out = nullptr;
  float* h_scratch = nullptr;
  // device-side makeCoarseDepthL0 (ct_depth.cu)
  float *cd_idepth[DMV_MAX_PYR_LEVELS] = {nullptr}, *cd_ws[DMV_MAX_PYR_LEVELS] = {nullptr}, *cd_ws2[DMV_MAX_PYR_LEVELS] = {nullptr};
  int *cd_rowcnt = nullptr, *cd_rowoff = nullptr, *cd_totals = nullptr;  // cd_totals: pinned host, device-visible
  float* d_ip = nullptr;   // immature-point arrays (dmv_ct_trace_points)
  float* h_ip = nullptr;
  int ip_cap = 0;
  float huber = 9.f;
  int cluster_size = 0;        // CTAs of ct_track_cluster_kernel's cluster (0 = not probed yet, -1 = no TMA descriptors, -2 = no cluster fits)
  CTMaps* maps = nullptr;      // TMA descriptors of the level planes (host copy; passed as a kernel parameter)
  long long launches = 0;
  float last_ms[4] = {0, 0, 0, 0};
  unsigned resident = 0;       // bit l: a frame's level l is resident (dmv_ct_upload_new_image sets every level, dmv_ct_upload_new its own)
  PSState* ps = nullptr;       // pixel selection buffers (ps_select.cu), allocated on first use
};

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return dmv::set_error(DMV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)); \
  } while (0)

extern "C" {

static int ct_allocate(dmv_ct* c, const dmv_ct_config* cfg);

int dmv_ct_create(const dmv_ct_config* cfg, dmv_ct** out) {
  if (!cfg || !out) return set_error(DMV_ERR_INVALID, "null argument");
  if (cfg->levels < 1 || cfg->levels > DMV_MAX_PYR_LEVELS || cfg->w < 16 || cfg->h < 16 || cfg->max_points < 1)
    return set_error(DMV_ERR_INVALID, "bad config");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return set_error(DMV_ERR_NO_DEVICE, "no CUDA device: dmvio_b200 has no CPU path");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return set_error(DMV_ERR_INVALID, "device out of range");
  CK(cudaSetDevice(cfg->device));
  dmv_ct* c = new dmv_ct();
  const int rc = ct_allocate(c, cfg);
  if (rc != DMV_OK) {  // allocation failed half-way: release what exists, keep the failing call's error message
    dmv_ct_destroy(c);
    return rc;
  }
  *out = c;
  return DMV_OK;
}

static int ct_allocate(dmv_ct* c, const dmv_ct_config* cfg) {
  c->cfg = *cfg;
  c->device = cfg->device;
  CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&c->ev[0]));
  CK(cudaEventCreate(&c->ev[1]));
  for (int l = 0; l < cfg->levels; l++) {
    c->w[l] = cfg->w >> l; c->h[l] = cfg->h >> l; c->haveK[l] = false; c->n[l] = 0;
    const size_t npx = (size_t)c->w[l] * c->h[l];
    CK(cudaMalloc(&c->d_img[l], npx * sizeof(float4)));
    CK(cudaMalloc(&c->d_gray[l], npx * sizeof(float)));
    CK(cudaMalloc(&c->d_u[l], sizeof(float) * cfg->max_points));
    CK(cudaMalloc(&c->d_v[l], sizeof(float) * cfg->max_points));
    CK(cudaMalloc(&c->d_id[l], sizeof(float) * cfg->max_points));
    CK(cudaMalloc(&c->d_col[l], sizeof(float) * cfg->max_points));
  }
  const size_t npx0 = (size_t)cfg->w * cfg->h;
  CK(cudaMalloc(&c->d_stage, npx0 * 3 * sizeof(float)));
  const int maxBlocks = (cfg->max_points + CT_THREADS - 1) / CT_THREADS;
  CK(cudaMalloc(&c->d_partial, sizeof(double) * CT_NRED * maxBlocks));
  CK(cudaMalloc(&c->d_ticket, sizeof(unsigned int)));
  CK(cudaMemset(c->d_ticket, 0, sizeof(unsigned int)));
  CK(cudaMalloc(&c->d_out, sizeof(double) * 64));
  CK(cudaMallocHost(&c->h_out, sizeof(double) * 64));
  CK(cudaMallocHost(&c->h_scratch, sizeof(float) * std::max(npx0 * 3, (size_t)cfg->max_points * 4)));
  return DMV_OK;
}

int dmv_ct_destroy(dmv_ct* c) {
  if (!c) return DMV_OK;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (int l = 0; l < DMV_MAX_PYR_LEVELS; l++) {
    cudaFree(c->d_img[l]); cudaFree(c->d_gray[l]); cudaFree(c->d_u[l]); cudaFree(c->d_v[l]); cudaFree(c->d_id[l]); cudaFree(c->d_col[l]);
  }
  cudaFree(c->d_stage); cudaFree(c->d_partial); cudaFree(c->d_ticket); cudaFree(c->d_out);
  cudaFreeHost(c->h_out); cudaFreeHost(c->h_scratch); cudaFree(c->d_ip); cudaFreeHost(c->h_ip);
  for (int l = 0; l < DMV_MAX_PYR_LEVELS; l++) { cudaFree(c->cd_idepth[l]); cudaFree(c->cd_ws[l]); cudaFree(c->cd_ws2[l]); }
  cudaFree(c->cd_rowcnt); cudaFree(c->cd_rowoff); cudaFreeHost(c->cd_totals);
  if (c->ev[0]) cudaEventDestroy(c->ev[0]);
  if (c->ev[1]) cudaEventDestroy(c->ev[1]);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c->maps;
  if (c->ps) { ps_free(*c->ps); delete c->ps; }
  delete c;
  return DMV_OK;
}

int dmv_ct_set_K(dmv_ct* c, int l, float fx, float fy, float cx, float cy) {
  if (!c || l < 0 || l >= c->cfg.levels) return set_error(DMV_ERR_INVALID, "bad level");
  c->fx[l] = fx; c->fy[l] = fy; c->cx[l] = cx; c->cy[l] = cy; c->haveK[l] = true;
  return DMV_OK;
}
int dmv_ct_set_huber(dmv_ct* c, float huberTH) {
  if (!c) return set_error(DMV_ERR_INVALID, "null handle");
  c->huber = huberTH;
  return DMV_OK;
}

int dmv_ct_set_ref(dmv_ct* c, int l, int n, const float* u, const float* v, const float* id, const float* col) {
  if (!c || l < 0 || l >= c->cfg.levels || n < 0 || n > c->cfg.max_points) return set_error(DMV_ERR_INVALID, "bad level / count");
  if (n > 0 && (!u || !v || !id || !col)) return set_error(DMV_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  c->n[l] = n;
  if (n > 0) {
    if (c->staging_busy) { CK(cudaStreamSynchronize(c->stream)); c->staging_busy = false; }
    float* s = c->h_scratch;
    std::memcpy(s, u, 4 * (size_t)n); std::memcpy(s + n, v, 4 * (size_t)n); std::memcpy(s + 2 * (size_t)n, id, 4 * (size_t)n);
    std::memcpy(s + 3 * (size_t)n, col, 4 * (size_t)n);
    CK(cudaMemcpyAsync(c->d_u[l], s, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->d_v[l], s + n, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->d_id[l], s + 2 * (size_t)n, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->d_col[l], s + 3 * (size_t)n, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  return DMV_OK;
}

int dmv_ct_upload_new(dmv_ct* c, int l, const float* dIp) {
  if (!c || !dIp || l < 0 || l >= c->cfg.levels) return set_error(DMV_ERR_INVALID, "bad level / pointer");
  CK(cudaSetDevice(c->device));
  const size_t npx = (size_t)c->w[l] * c->h[l];
  if (c->staging_busy) { CK(cudaStreamSynchronize(c->stream)); c->staging_busy = false; }
  std::memcpy(c->h_scratch, dIp, npx * 3 * sizeof(float));
  CK(cudaMemcpyAsync(c->d_stage, c->h_scratch, npx * 3 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  ct_repack_kernel<<<(unsigned)((npx + 255) / 256), 256, 0, c->stream>>>(c->d_stage, c->d_img[l], (int)npx);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(c->stream));
  c->resident |= 1u << l;
  return DMV_OK;
}

int dmv_ct_upload_new_image(dmv_ct* c, const float* image) {
  if (!c || !image) return set_error(DMV_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  const size_t npx = (size_t)c->w[0] * c->h[0];
  if (c->staging_busy) { CK(cudaStreamSynchronize(c->stream)); c->staging_busy = false; }  // a previous upload may still read the staging buffer
  std::memcpy(c->h_scratch, image, npx * sizeof(float));
  CK(cudaMemcpyAsync(c->d_gray[0], c->h_scratch, npx * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  for (int l = 0; l < c->cfg.levels; l++) {
    const int wl = c->w[l], hl = c->h[l];
    if (l > 0) {
      dim3 grid((wl + 127) / 128, hl);
      pyr_down_kernel<<<grid, 128, 0, c->stream>>>(c->d_img[l - 1], c->d_gray[l], wl, hl, c->w[l - 1]);
      c->launches++;
    }
    grad_kernel<<<(wl * hl + 255) / 256, 256, 0, c->stream>>>(c->d_gray[l], c->d_img[l], wl, hl);
    c->launches++;
  }
  CK(cudaGetLastError());
  // no synchronisation: every consumer (dmv_ct_calc_res_gs / dmv_ct_track) runs on the same stream and synchronises itself; the image
  // was copied into the handle's pinned staging buffer above, so the caller's buffer is already free
  c->staging_busy = true;
  c->resident = (1u << c->cfg.levels) - 1;
  return DMV_OK;
}

int dmv_ct_calc_res_gs(dmv_ct* c, int l, const float RKi[9], const float t[3], const float affLL[2], float b0, float cutoffTH, int want_gs,
                       double res6[6], double H[64], double b[8], int* n_warped) {
  if (!c || !RKi || !t || !affLL || !res6 || l < 0 || l >= c->cfg.levels) return set_error(DMV_ERR_INVALID, "bad argument");
  if (!c->haveK[l]) return set_error(DMV_ERR_STATE, "dmv_ct_set_K(level) first");
  if (want_gs && (!H || !b)) return set_error(DMV_ERR_INVALID, "H/b required with want_gs");
  CK(cudaSetDevice(c->device));
  CTParams P;
  std::memcpy(P.RKi, RKi, sizeof(P.RKi));
  std::memcpy(P.t, t, sizeof(P.t));
  // Ki[lvl] = K^-1 (CoarseTracker.cpp:L126-133)
  {
    const float Kl[9] = {c->fx[l], 0.f, c->cx[l], 0.f, c->fy[l], c->cy[l], 0.f, 0.f, 1.f};
    inv3_cofactor(Kl, P.Ki);
  }
  P.fx = c->fx[l]; P.fy = c->fy[l]; P.cx = c->cx[l]; P.cy = c->cy[l];
  P.affa = affLL[0]; P.affb = affLL[1]; P.a_gs = affLL[0]; P.b0 = b0;
  P.cutoff = cutoffTH; P.huber = c->huber;
  P.maxEnergy = 2 * c->huber * cutoffTH - c->huber * c->huber;
  P.w = c->w[l]; P.h = c->h[l]; P.n = c->n[l]; P.lvl = l; P.want_gs = want_gs;
  const int nb = std::max(1, (c->n[l] + CT_THREADS - 1) / CT_THREADS);
  if (c->timing) CK(cudaEventRecord(c->ev[0], c->stream));
  // the last block writes the 53 reduced doubles straight into the pinned host buffer (zero-copy): no D2H copy node per evaluation
  ct_res_gs_kernel<<<nb, CT_THREADS, 0, c->stream>>>(P, c->d_u[l], c->d_v[l], c->d_id[l], c->d_col[l], c->d_img[l], c->d_partial, c->d_ticket,
                                                      c->h_out);
  c->launches++;
  if (c->timing) CK(cudaEventRecord(c->ev[1], c->stream));
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(c->stream));
  c->staging_busy = false;
  if (c->timing) cudaEventElapsedTime(&c->last_ms[0], c->ev[0], c->ev[1]);
  const double* o = c->h_out;
  for (int k = want_gs ? 0 : 72; k <= 72; k++) ct_finish(o, k, res6, H, b);
  if (n_warped) *n_warped = ((int)o[48] + 3) & ~3;
  return DMV_OK;
}

// TMA descriptors of the level planes: a w x h plane of float4 texels = a 2-D tensor of (2w) x h fp64 elements (the widest element type a
// tensor map knows; 16-byte texels = pairs), one box = the whole plane.  Only levels that fit CTC_PLANE_BYTES are ever copied.
static int ct_make_tensor_maps(dmv_ct* c) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                               CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn || qres != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    return set_error(DMV_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
  }
  if (!c->maps) c->maps = new CTMaps();
  std::memset(c->maps, 0, sizeof(CTMaps));
  for (int l = 0; l < c->cfg.levels; l++) {
    const size_t bytes = (size_t)c->w[l] * c->h[l] * sizeof(float4);
    if (bytes > (size_t)CTC_PLANE_BYTES || 2 * c->w[l] > 256 || c->h[l] > 256) continue;   // never staged (box limits: 256 elements per dimension)
    const cuuint64_t gdim[2] = {(cuuint64_t)(2 * c->w[l]), (cuuint64_t)c->h[l]};
    const cuuint64_t gstride[1] = {(cuuint64_t)c->w[l] * sizeof(float4)};
    const cuuint32_t box[2] = {(cuuint32_t)(2 * c->w[l]), (cuuint32_t)c->h[l]};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<EncodeFn>(fn)(&c->maps->lvl[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, c->d_img[l], gdim, gstride, box, estr,
                                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(DMV_ERR_CUDA, "cuTensorMapEncodeTiled failed for level %d (CUresult %d)", l, (int)r);
  }
  return DMV_OK;
}

// CoarseTracker::trackNewestCoarse (CoarseTracker.cpp:L539-770, visual-only branch) in one persistent cluster launch
int dmv_ct_track(dmv_ct* c, const dmv_ct_track_args* in, dmv_ct_track_result* out) {
  if (!c || !in || !out) return set_error(DMV_ERR_INVALID, "null argument");
  if (in->coarsestLvl < 0 || in->coarsestLvl >= c->cfg.levels || in->coarsestLvl >= 5) return set_error(DMV_ERR_INVALID, "coarsestLvl out of range");
  CK(cudaSetDevice(c->device));
  CTTrack T;
  std::memset(&T, 0, sizeof(T));
  T.coarsest = in->coarsestLvl;
  for (int l = 0; l < c->cfg.levels; l++) {
    if (!c->haveK[l]) return set_error(DMV_ERR_STATE, "dmv_ct_set_K(level) first");
    T.n[l] = c->n[l]; T.w[l] = c->w[l]; T.h[l] = c->h[l];
    T.fx[l] = c->fx[l]; T.fy[l] = c->fy[l]; T.cx[l] = c->cx[l]; T.cy[l] = c->cy[l];
    const float Kl[9] = {c->fx[l], 0.f, c->cx[l], 0.f, c->fy[l], c->cy[l], 0.f, 0.f, 1.f};
    inv3_cofactor(Kl, T.Ki[l]);
    T.u[l] = c->d_u[l]; T.v[l] = c->d_v[l]; T.id[l] = c->d_id[l]; T.col[l] = c->d_col[l]; T.img[l] = c->d_img[l];
  }
  for (int i = 0; i < 9; i++) T.R0[i] = in->R[i];
  for (int i = 0; i < 3; i++) T.t0[i] = in->t[i];
  T.a0 = in->a; T.b0 = in->b; T.ref_a = in->ref_a; T.ref_b = in->ref_b;
  T.ref_exposure = in->ref_exposure; T.new_exposure = in->new_exposure;
  T.huber = c->huber; T.cutoffTH = in->coarseCutoffTH; T.affModeA = in->affineOptModeA; T.affModeB = in->affineOptModeB;
  for (int i = 0; i < 5; i++) T.minRes[i] = in->minResForAbort[i];
  T.out = c->h_out;
  if (c->cluster_size == 0) {  // probe once: the largest cluster the device schedules for this kernel (16 needs the non-portable opt-in)
    c->cluster_size = -1;
    const int rc = ct_make_tensor_maps(c);
    if (rc != DMV_OK) return rc;
    c->cluster_size = -2;
    CK(cudaFuncSetAttribute(ct_track_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CTCSmem)));
    cudaFuncSetAttribute(ct_track_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaGetLastError();
    for (int nc : {16, 8, 4}) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(nc); cfg.blockDim = dim3(CTC_THREADS); cfg.dynamicSmemBytes = sizeof(CTCSmem); cfg.stream = c->stream;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = nc; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      int ncl = 0;
      if (cudaOccupancyMaxActiveClusters(&ncl, ct_track_cluster_kernel, &cfg) == cudaSuccess && ncl >= 1) { c->cluster_size = nc; break; }
      cudaGetLastError();
    }
  }
  if (c->cluster_size == -1) return set_error(DMV_ERR_CUDA, "dmv_ct_track: the TMA descriptors of the level planes could not be encoded");
  if (c->cluster_size < 0)
    return set_error(DMV_ERR_CUDA, "dmv_ct_track: no cluster of 16, 8 or 4 CTAs (%d threads, %zu B shared memory each) fits on device %d", CTC_THREADS,
                     sizeof(CTCSmem), c->device);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(c->cluster_size); cfg.blockDim = dim3(CTC_THREADS); cfg.dynamicSmemBytes = sizeof(CTCSmem); cfg.stream = c->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = c->cluster_size; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  CK(cudaLaunchKernelEx(&cfg, ct_track_cluster_kernel, T, *c->maps));
  c->launches++;
  CK(cudaStreamSynchronize(c->stream));
  c->staging_busy = false;
  const double* o = c->h_out;
  for (int i = 0; i < 9; i++) out->R[i] = o[i];
  for (int i = 0; i < 3; i++) out->t[i] = o[9 + i];
  out->a = o[12]; out->b = o[13];
  for (int i = 0; i < 5; i++) out->lastResiduals[i] = o[14 + i];
  for (int i = 0; i < 3; i++) out->flowIndicators[i] = o[19 + i];
  out->trackingGood = (int)o[22]; out->iterations = (int)o[23]; out->evaluations = (int)o[24]; out->status = (int)o[25];
  return DMV_OK;
}

void dmv_ip_default_settings(dmv_ip_settings* s) {
  s->maxPixSearch = 0.027f; s->trace_stepsize = 1.0f; s->trace_GNThreshold = 0.1f; s->trace_extraSlackOnTH = 1.2f; s->trace_slackInterval = 1.5f;
  s->trace_minImprovementFactor = 2.f; s->huberTH = 9.f; s->trace_GNIterations = 3; s->minTraceTestRadius = 2;
}

// the immature-point staging buffers d_ip / h_ip, shared by dmv_ct_make_coarse_depth, dmv_ct_init_points and dmv_ct_trace_points_multi:
// grown to hold n points of CT_IP_WORDS words each (23 read-only floats, 7 in/out words and the set index of dmv_ct_trace_points_multi)
// plus the per-frame tables (14 floats for each of up to 64 host frames)
constexpr int CT_IP_WORDS = 31;
static int ct_reserve_ip(dmv_ct* c, int n) {
  if (n <= c->ip_cap) return DMV_OK;
  cudaFree(c->d_ip);
  cudaFreeHost(c->h_ip);
  c->d_ip = nullptr; c->h_ip = nullptr; c->ip_cap = 0;
  const int cap = std::max(n, 2048);
  const size_t bytes = sizeof(float) * ((size_t)CT_IP_WORDS * cap + 14 * 64);
  CK(cudaMalloc(&c->d_ip, bytes));
  CK(cudaMallocHost(&c->h_ip, bytes));
  c->ip_cap = cap;
  return DMV_OK;
}

// CoarseTracker::setCoarseTrackingRef -> makeCoarseDepthL0 (CoarseTracker.cpp:L138-295) on the device (ct_depth.cu); the reference frame is
// the one resident in the handle (last dmv_ct_upload_new_image / dmv_ct_upload_new of every level)
int dmv_ct_make_coarse_depth(dmv_ct* c, int n, const float* Ku, const float* Kv, const float* new_idepth, const float* HdiF, int32_t* pc_n_out) {
  if (!c || n < 0 || (n > 0 && (!Ku || !Kv || !new_idepth || !HdiF))) return set_error(DMV_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  const int L = c->cfg.levels, w0 = c->w[0], h0 = c->h[0];
  if (!c->cd_totals) {
    for (int l = 0; l < L; l++) {
      const size_t npx = (size_t)c->w[l] * c->h[l];
      CK(cudaMalloc(&c->cd_idepth[l], npx * sizeof(float)));
      CK(cudaMalloc(&c->cd_ws[l], npx * sizeof(float)));
      CK(cudaMalloc(&c->cd_ws2[l], npx * sizeof(float)));
    }
    CK(cudaMalloc(&c->cd_rowcnt, sizeof(int) * h0));
    CK(cudaMalloc(&c->cd_rowoff, sizeof(int) * h0));
    CK(cudaMallocHost(&c->cd_totals, sizeof(int) * DMV_MAX_PYR_LEVELS));
  }
  // ---- the splat's only order-dependent part on the host: points hitting the same pixel are folded in input order (L144-160)
  {
    const int rc = ct_reserve_ip(c, n);
    if (rc != DMV_OK) return rc;
  }
  if (c->staging_busy) { CK(cudaStreamSynchronize(c->stream)); c->staging_busy = false; }
  const size_t cap = c->ip_cap;
  int* h_pix = reinterpret_cast<int*>(c->h_ip);
  float* h_idw = c->h_ip + cap;
  float* h_ws = c->h_ip + 2 * cap;
  int nu = 0;
  {
    std::unordered_map<int, int> slot;
    slot.reserve((size_t)n * 2);
    for (int i = 0; i < n; i++) {
      const int u = Ku[i] + 0.5f, v = Kv[i] + 0.5f;
      if (u < 0 || v < 0 || u >= w0 || v >= h0) return set_error(DMV_ERR_INVALID, "residual %d projects to (%d,%d) outside the image", i, u, v);
      const float weight = sqrtf(1e-3 / (HdiF[i] + 1e-12));
      const int pix = u + w0 * v;
      auto it = slot.find(pix);
      if (it == slot.end()) { slot.emplace(pix, nu); h_pix[nu] = pix; h_idw[nu] = 0.f + new_idepth[i] * weight; h_ws[nu] = 0.f + weight; nu++; }
      else { h_idw[it->second] += new_idepth[i] * weight; h_ws[it->second] += weight; }
    }
  }
  CK(cudaMemcpyAsync(c->d_ip, c->h_ip, sizeof(float) * 3 * cap, cudaMemcpyHostToDevice, c->stream));
  CDLevels Lv;
  Lv.levels = L; Lv.cap = c->cfg.max_points;
  for (int l = 0; l < L; l++) {
    Lv.w[l] = c->w[l]; Lv.h[l] = c->h[l];
    Lv.idepth[l] = c->cd_idepth[l]; Lv.ws[l] = c->cd_ws[l]; Lv.ws2[l] = c->cd_ws2[l]; Lv.img[l] = c->d_img[l];
    Lv.pc_u[l] = c->d_u[l]; Lv.pc_v[l] = c->d_v[l]; Lv.pc_id[l] = c->d_id[l]; Lv.pc_col[l] = c->d_col[l];
  }
  Lv.rowcnt = c->cd_rowcnt; Lv.rowoff = c->cd_rowoff; Lv.totals = c->cd_totals;
  cd_launch(Lv, nu, reinterpret_cast<const int*>(c->d_ip), c->d_ip + cap, c->d_ip + 2 * cap, c->stream);
  c->launches += 2 + 4 * L;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(c->stream));
  for (int l = 0; l < L; l++) {
    if (c->cd_totals[l] > c->cfg.max_points) return set_error(DMV_ERR_INVALID, "level %d: %d reference points exceed max_points %d", l, c->cd_totals[l], c->cfg.max_points);
    c->n[l] = c->cd_totals[l];
    if (pc_n_out) pc_n_out[l] = c->n[l];
  }
  return DMV_OK;
}

// pc_u / pc_v / pc_idepth / pc_color of a level as they sit on the device (tests; any pointer may be NULL); returns pc_n[level] in *n
int dmv_ct_get_ref(dmv_ct* c, int l, int* n, float* pc_u, float* pc_v, float* pc_idepth, float* pc_color) {
  if (!c || !n || l < 0 || l >= c->cfg.levels) return set_error(DMV_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  *n = c->n[l];
  const size_t bytes = sizeof(float) * c->n[l];
  if (pc_u) CK(cudaMemcpy(pc_u, c->d_u[l], bytes, cudaMemcpyDeviceToHost));
  if (pc_v) CK(cudaMemcpy(pc_v, c->d_v[l], bytes, cudaMemcpyDeviceToHost));
  if (pc_idepth) CK(cudaMemcpy(pc_idepth, c->d_id[l], bytes, cudaMemcpyDeviceToHost));
  if (pc_color) CK(cudaMemcpy(pc_color, c->d_col[l], bytes, cudaMemcpyDeviceToHost));
  return DMV_OK;
}

// ImmaturePoint constructor on the resident frame (ip_trace.cu)
int dmv_ct_init_points(dmv_ct* c, int n, const int32_t* u, const int32_t* v, float* color8, float* weights8, float* gradH4, float* energyTH, int32_t* ok) {
  if (!c || n < 0 || (n > 0 && (!u || !v || !color8 || !weights8 || !gradH4 || !energyTH || !ok))) return set_error(DMV_ERR_INVALID, "null argument");
  if (n == 0) return DMV_OK;
  for (int i = 0; i < n; i++)
    if (u[i] < 2 || v[i] < 2 || u[i] >= c->w[0] - 3 || v[i] >= c->h[0] - 3) return set_error(DMV_ERR_INVALID, "point %d (%d,%d): the pattern leaves the image", i, u[i], v[i]);
  CK(cudaSetDevice(c->device));
  {
    const int rc = ct_reserve_ip(c, n);
    if (rc != DMV_OK) return rc;
  }
  if (c->staging_busy) { CK(cudaStreamSynchronize(c->stream)); c->staging_busy = false; }
  const size_t cap = c->ip_cap;
  float* hb = c->h_ip;
  float* d = c->d_ip;
  // layout (words): u | v | color*8 | weights*8 | gradH*4 | energyTH | ok
  std::memcpy(hb, u, 4 * (size_t)n); std::memcpy(hb + cap, v, 4 * (size_t)n);
  CK(cudaMemcpyAsync(d, hb, sizeof(float) * 2 * cap, cudaMemcpyHostToDevice, c->stream));
  IPInitArgs A;
  A.n = n; A.w = c->w[0];
  A.outlierTHSumComponent = 50.f * 50.f; A.outlierTH = 12.f * 12.f; A.overallEnergyTHWeight = 1.f;  // util/settings.cpp:L111-114, L159
  A.u = reinterpret_cast<const int*>(d); A.v = reinterpret_cast<const int*>(d + cap);
  A.color = d + 2 * cap; A.weights = d + 10 * cap; A.gradH = d + 18 * cap; A.energyTH = d + 22 * cap; A.ok = reinterpret_cast<int*>(d + 23 * cap);
  A.img = c->d_img[0];
  launch_ip_init(A, c->stream);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(hb + 2 * cap, d + 2 * cap, sizeof(float) * 22 * cap, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  std::memcpy(color8, hb + 2 * cap, 32 * (size_t)n); std::memcpy(weights8, hb + 10 * cap, 32 * (size_t)n); std::memcpy(gradH4, hb + 18 * cap, 16 * (size_t)n);
  std::memcpy(energyTH, hb + 22 * cap, 4 * (size_t)n); std::memcpy(ok, hb + 23 * cap, 4 * (size_t)n);
  return DMV_OK;
}

// immature points of SEVERAL host frames traced against the resident newest frame in ONE launch (ip_trace.cu): FullSystem::traceNewCoarse's
// loop over the window's keyframes (FullSystem.cpp:L554-575) collapsed into one upload, one kernel, one download
int dmv_ct_trace_points_multi(dmv_ct* c, int nsets, const dmv_ip_points* sets, const float* tables14, const dmv_ip_settings* settings) {
  if (!c || nsets < 0 || (nsets > 0 && (!sets || !tables14))) return set_error(DMV_ERR_INVALID, "null argument");
  int n = 0;
  for (int k = 0; k < nsets; k++) {
    const dmv_ip_points* p = &sets[k];
    if (p->n < 0 || (p->n > 0 && (!p->u || !p->v || !p->color8 || !p->weights8 || !p->gradH4 || !p->energyTH || !p->idepth_min || !p->idepth_max || !p->quality ||
                                  !p->lastTraceStatus || !p->lastTraceUV2 || !p->lastTracePixelInterval)))
      return set_error(DMV_ERR_INVALID, "incomplete dmv_ip_points (set %d)", k);
    n += p->n;
  }
  if (n == 0) return DMV_OK;
  CK(cudaSetDevice(c->device));
  {
    const int rc = ct_reserve_ip(c, n);
    if (rc != DMV_OK) return rc;
  }
  if (nsets > 64) return set_error(DMV_ERR_INVALID, "at most 64 host frames per call");
  if (c->staging_busy) { CK(cudaStreamSynchronize(c->stream)); c->staging_busy = false; }
  const size_t cap = c->ip_cap;
  float* hb = c->h_ip;
  // layout (floats): u | v | color*8 | weights*8 | gradH*4 | energyTH | idmin | idmax | quality | status(int) | uv*2 | interval | set(int) | tables
  const size_t o_u = 0, o_v = cap, o_col = 2 * cap, o_wgt = 10 * cap, o_g = 18 * cap, o_eth = 22 * cap, o_min = 23 * cap, o_max = 24 * cap, o_q = 25 * cap,
               o_st = 26 * cap, o_uv = 27 * cap, o_iv = 29 * cap, o_set = 30 * cap, o_tab = 31 * cap;
  size_t at = 0;
  for (int k = 0; k < nsets; k++) {
    const dmv_ip_points* p = &sets[k];
    const size_t m = (size_t)p->n;
    if (m == 0) continue;
    std::memcpy(hb + o_u + at, p->u, 4 * m); std::memcpy(hb + o_v + at, p->v, 4 * m);
    std::memcpy(hb + o_col + 8 * at, p->color8, 32 * m); std::memcpy(hb + o_wgt + 8 * at, p->weights8, 32 * m);
    std::memcpy(hb + o_g + 4 * at, p->gradH4, 16 * m); std::memcpy(hb + o_eth + at, p->energyTH, 4 * m);
    std::memcpy(hb + o_min + at, p->idepth_min, 4 * m); std::memcpy(hb + o_max + at, p->idepth_max, 4 * m); std::memcpy(hb + o_q + at, p->quality, 4 * m);
    std::memcpy(hb + o_st + at, p->lastTraceStatus, 4 * m); std::memcpy(hb + o_uv + 2 * at, p->lastTraceUV2, 8 * m); std::memcpy(hb + o_iv + at, p->lastTracePixelInterval, 4 * m);
    int* setp = reinterpret_cast<int*>(hb + o_set + at);
    for (size_t q = 0; q < m; q++) setp[q] = k;
    at += m;
  }
  std::memcpy(hb + o_tab, tables14, sizeof(float) * 14 * (size_t)nsets);
  CK(cudaMemcpyAsync(c->d_ip, hb, sizeof(float) * ((size_t)CT_IP_WORDS * cap + 14 * (size_t)nsets), cudaMemcpyHostToDevice, c->stream));
  IPTraceArgs A;
  std::memset(&A, 0, sizeof(A));
  A.n = n; A.w = c->w[0]; A.h = c->h[0];
  if (settings) A.s = *settings; else dmv_ip_default_settings(&A.s);
  float* d = c->d_ip;
  A.tab = d + o_tab; A.set_of = reinterpret_cast<const int*>(d + o_set);
  A.u = d + o_u; A.v = d + o_v; A.color = d + o_col; A.weights = d + o_wgt; A.gradH = d + o_g; A.energyTH = d + o_eth;
  A.idepth_min = d + o_min; A.idepth_max = d + o_max; A.quality = d + o_q; A.status = reinterpret_cast<int*>(d + o_st); A.uv = d + o_uv; A.interval = d + o_iv;
  A.img = c->d_img[0];
  launch_ip_trace(A, c->stream);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(hb + o_min, d + o_min, sizeof(float) * 7 * cap, cudaMemcpyDeviceToHost, c->stream));  // the 7 in/out words per point
  CK(cudaStreamSynchronize(c->stream));
  at = 0;
  for (int k = 0; k < nsets; k++) {
    const dmv_ip_points* p = &sets[k];
    const size_t m = (size_t)p->n;
    if (m == 0) continue;
    std::memcpy(p->idepth_min, hb + o_min + at, 4 * m); std::memcpy(p->idepth_max, hb + o_max + at, 4 * m); std::memcpy(p->quality, hb + o_q + at, 4 * m);
    std::memcpy(p->lastTraceStatus, hb + o_st + at, 4 * m); std::memcpy(p->lastTraceUV2, hb + o_uv + 2 * at, 8 * m); std::memcpy(p->lastTracePixelInterval, hb + o_iv + at, 4 * m);
    at += m;
  }
  return DMV_OK;
}

// one host frame's immature points traced against the resident newest frame
int dmv_ct_trace_points(dmv_ct* c, const dmv_ip_points* p, const float KRKi[9], const float Kt[3], const float aff[2], const dmv_ip_settings* settings) {
  if (!c || !p || !KRKi || !Kt || !aff) return set_error(DMV_ERR_INVALID, "null argument");
  float tab[14];
  std::memcpy(tab, KRKi, 36); std::memcpy(tab + 9, Kt, 12); std::memcpy(tab + 12, aff, 8);
  return dmv_ct_trace_points_multi(c, 1, p, tab, settings);
}

// PixelSelector::makeMaps on the resident frame (ps_select.cu): argument checks shared by dmv_ct_select_pixels / dmv_ct_make_new_traces
static int ct_select(dmv_ct* c, const dmv_ps_args* a, dmv_ps_result* r) {
  if (!c || !a || !r) return set_error(DMV_ERR_INVALID, "null argument");
  if (c->w[0] % 16 || c->h[0] % 16) return set_error(DMV_ERR_INVALID, "pixel selection needs w and h divisible by 16 (have %dx%d)", c->w[0], c->h[0]);
  if (c->cfg.levels < 3) return set_error(DMV_ERR_INVALID, "pixel selection reads pyramid levels 0..2 (handle has %d)", c->cfg.levels);
  if (!(a->density > 0.f) || !std::isfinite(a->density) || a->currentPotential < 1 || !std::isfinite(a->thFactor))
    return set_error(DMV_ERR_INVALID, "bad dmv_ps_args (density %g, currentPotential %d, thFactor %g)", a->density, a->currentPotential, a->thFactor);
  if ((c->resident & 7u) != 7u) return set_error(DMV_ERR_STATE, "no frame resident: upload one first (dmv_ct_upload_new_image, or dmv_ct_upload_new of levels 0..2)");
  CK(cudaSetDevice(c->device));
  if (!c->ps) c->ps = new PSState();
  int rc = ps_alloc(*c->ps, c->w[0], c->h[0]);
  if (rc != DMV_OK) return rc;
  const float4* img[3] = {c->d_img[0], c->d_img[1], c->d_img[2]};
  return ps_make_maps(*c->ps, img, *a, c->stream, &c->launches, r);
}

int dmv_ct_select_pixels(dmv_ct* c, const dmv_ps_args* a, float* map_out, dmv_ps_result* r) {
  dmv_ps_result res;
  const int rc = ct_select(c, a, &res);
  if (rc != DMV_OK) return rc;
  if (map_out) {
    CK(cudaMemcpyAsync(map_out, c->ps->map, sizeof(float) * c->w[0] * c->h[0], cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  *r = res;
  return DMV_OK;
}

// FullSystem::makeNewTraces (FullSystem.cpp:L1640-1665): selection, compaction in raster order and the ImmaturePoint constructor
// (ip_trace.cu) on the device; one download of the points, of which the host keeps those with a finite energyTH
int dmv_ct_make_new_traces(dmv_ct* c, const dmv_ps_args* a, int cap, int* n, int32_t* u, int32_t* v, float* type, float* color8, float* weights8,
                           float* gradH4, float* energyTH, dmv_ps_result* r) {
  if (!n || cap < 0 || (cap > 0 && (!u || !v || !type || !color8 || !weights8 || !gradH4 || !energyTH))) return set_error(DMV_ERR_INVALID, "null argument");
  dmv_ps_result res;
  int rc = ct_select(c, a, &res);
  if (rc != DMV_OK) return rc;
  rc = ct_reserve_ip(c, std::max(res.numHaveSub, 1));
  if (rc != DMV_OK) return rc;
  // the compaction writes u | v | type at words 28, 29, 30 x cap (cap >= numHaveSub >= the count m); the constructor then works in the
  // stride-m layout u | v | color*8 | weights*8 | gradH*4 | energyTH | ok | type, which ends before word 25 x cap
  const size_t cap_ip = c->ip_cap;
  float* d = c->d_ip;
  float* scratch = d + 28 * cap_ip;
  int m = 0;
  rc = ps_compact(*c->ps, 2 /* patternPadding */, reinterpret_cast<int*>(scratch), reinterpret_cast<int*>(scratch + cap_ip), scratch + 2 * cap_ip, c->stream,
                  &c->launches, &m);
  if (rc != DMV_OK) return rc;
  int kept = 0;
  if (m > 0) {
    const size_t M = (size_t)m;
    float* hb = c->h_ip;
    CK(cudaMemcpyAsync(d, scratch, sizeof(float) * M, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(d + M, scratch + cap_ip, sizeof(float) * M, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(d + 24 * M, scratch + 2 * cap_ip, sizeof(float) * M, cudaMemcpyDeviceToDevice, c->stream));
    IPInitArgs A;
    A.n = m; A.w = c->w[0];
    A.outlierTHSumComponent = 50.f * 50.f; A.outlierTH = 12.f * 12.f; A.overallEnergyTHWeight = 1.f;  // util/settings.cpp:L111-114, L159
    A.u = reinterpret_cast<const int*>(d); A.v = reinterpret_cast<const int*>(d + M);
    A.color = d + 2 * M; A.weights = d + 10 * M; A.gradH = d + 18 * M; A.energyTH = d + 22 * M; A.ok = reinterpret_cast<int*>(d + 23 * M);
    A.img = c->d_img[0];
    launch_ip_init(A, c->stream);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hb, d, sizeof(float) * 25 * M, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    const int* ok = reinterpret_cast<const int*>(hb + 23 * M);
    for (int i = 0; i < m; i++) kept += ok[i] != 0;
    if (kept <= cap) {
      const int* hu = reinterpret_cast<const int*>(hb);
      const int* hv = reinterpret_cast<const int*>(hb + M);
      for (int i = 0, k = 0; i < m; i++) {
        if (!ok[i]) continue;
        u[k] = hu[i]; v[k] = hv[i]; type[k] = hb[24 * M + i];
        std::memcpy(color8 + 8 * k, hb + 2 * M + 8 * i, 32); std::memcpy(weights8 + 8 * k, hb + 10 * M + 8 * i, 32);
        std::memcpy(gradH4 + 4 * k, hb + 18 * M + 4 * i, 16); energyTH[k] = hb[22 * M + i];
        k++;
      }
    }
  }
  *n = kept;
  if (kept > cap) return set_error(DMV_ERR_INVALID, "%d new immature points, cap %d", kept, cap);
  *r = res;
  return DMV_OK;
}

// library-internal: the resident level-0 float4 plane of the coarse-tracker handle (dmv_ba_adopt_frame copies it device-to-device)
__attribute__((visibility("hidden"))) int dmv_ct_level0_plane(dmv_ct* c, const void** plane, int* w, int* h, int* device, cudaStream_t* stream) {
  if (!c) return set_error(DMV_ERR_INVALID, "null handle");
  *plane = c->d_img[0]; *w = c->w[0]; *h = c->h[0]; *device = c->device; *stream = c->stream;
  return DMV_OK;
}

int dmv_ct_set_timing(dmv_ct* c, int enable) {
  if (!c) return set_error(DMV_ERR_INVALID, "null handle");
  c->timing = enable != 0;
  return DMV_OK;
}
int dmv_ct_last_timing(dmv_ct* c, float ms[4]) {
  if (!c || !ms) return set_error(DMV_ERR_INVALID, "null argument");
  for (int i = 0; i < 4; i++) ms[i] = c->last_ms[i];
  return DMV_OK;
}
// instrumentation: reference points evaluated by the last dmv_ct_track, summed over its calcRes / calcGSSSE evaluations
int dmv_ct_last_point_evaluations(dmv_ct* c, double* n) {
  if (!c || !n) return set_error(DMV_ERR_INVALID, "null argument");
  *n = c->h_out[26];
  return DMV_OK;
}
int dmv_ct_kernel_launch_count(dmv_ct* c, long long* n) {
  if (!c || !n) return set_error(DMV_ERR_INVALID, "null argument");
  *n = c->launches;
  return DMV_OK;
}

}  // extern "C"
