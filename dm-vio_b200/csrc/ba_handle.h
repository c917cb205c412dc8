// Internal layout of the BA handle (shared by ba_api.cu and the measurement-only entry points in ba_bench.cu).
#pragma once
#include "../../include/dmvio_b200.h"
#include "ba_device.cuh"
#include "common_host.h"
#include <cstdint>
#include <vector>

namespace dmv {
cudaError_t launch_fused_kernel(BAWinDev& W, const BAIter& it, bool marg, cudaStream_t s, unsigned* bar_count);
cudaError_t launch_fused_batch_kernel(int P, const BAWinDev* gW, const BAIter* gIt, BABatchHdr& hdr, int max_nf, cudaStream_t s, unsigned* bar_count);
void launch_resub_kernel(const BAWinDev& W, const BAIter& it, int apply, double* sums, cudaStream_t s);
void launch_repack(const float* src, float4* dst, int n, cudaStream_t s);
void launch_make_dI(const float* img, float4* dst, int w, int h, cudaStream_t s);
void launch_l2_flush(float4* buf, size_t n, cudaStream_t s);
}  // namespace dmv

struct HostUpload {  // descriptor + per-iteration tables: passed BY VALUE as __grid_constant__ kernel parameters (no H2D copy)
  dmv::BAWinDev win;
  dmv::BAIter it;
};

using dmv::MAXF; using dmv::XCHG_MAXR; using dmv::BAAdj; using dmv::BAMarg;

struct dmv_ba {
  dmv_ba_config cfg;
  dmv_ba_params prm;
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  int P = 16;            // points per chunk of the CURRENT window (16 or 32)
  bool P_auto = true;    // dmv_ba_config::chunk_points == 0: chosen per window in dmv_ba_set_points
  int sms = 148;
  int mp = 0;  // point capacity (slot pitch)
  int nf = 0, npts = 0, nres = 0, nchunks = 0, max_chunks = 0;
  int N = 0, NW = 0, T = 0, ntiles = 0;
  int slots[MAXF];
  // device buffers
  float4* d_img[MAXF] = {nullptr};
  float* d_stage_img = nullptr;
  BAAdj* d_adj = nullptr;
  float2* d_uv = nullptr;
  float* d_idepth[2] = {nullptr, nullptr};  // ping-pong: [cur] current depths, [bak] FullSystem::backupState copy
  int id_cur = 0, id_bak = 0;
  bool zero_alias = false;                  // idepth_zero == idepth (true after any step / restore)
  float *d_idepth_zero = nullptr, *d_color = nullptr, *d_weights = nullptr, *d_priorF = nullptr;
  uint8_t* d_st_in = nullptr;
  float* d_en_in = nullptr;
  uint8_t* d_st_new[2] = {nullptr, nullptr};
  float *d_en_new[2] = {nullptr, nullptr}, *d_en_wo[2] = {nullptr, nullptr}, *d_cpt[2] = {nullptr, nullptr}, *d_jpjd[2] = {nullptr, nullptr},
        *d_pout[2] = {nullptr, nullptr};
  double* d_result[2] = {nullptr, nullptr};
  float* d_step = nullptr;
  double* d_part = nullptr;        // [max_chunks][PART_STRIDE] per-chunk partial blobs (scratch of one launch)
  float4* d_wg = nullptr;          // [WG_GROUPS][mp] Schur vectors, transposed (scratch)
  float* d_hdig = nullptr;         // [mp] HdiF (scratch)
  float* d_hdi_solve = nullptr;    // [mp] HdiF of the linearisation the last dmv_ba_accumulate returned (PointHessian::idepth_hessian)
  int hdi_solve_n = 0;
  unsigned int* d_bar = nullptr;   // grid-barrier arrival counter
  unsigned int bar_count = 0;      // arrivals issued so far (monotonic, wraps)
  double* d_resub_sums = nullptr;
  float4* d_flush = nullptr;
  size_t flush_n = 0;
  // pinned host
  HostUpload* h_up = nullptr;
  BAAdj* h_adj = nullptr;
  double* h_result[2] = {nullptr, nullptr};
  float* h_scratch = nullptr;  // max(mp*8, w*h*3) floats
  float* h_en_newest = nullptr; // [mp] en_wo of the residuals targeting the newest frame, written by the kernel itself (zero-copy)
  bool en_newest_valid = false; // h_en_newest belongs to the most recent linearisation
  size_t scratch_floats = 0;
  // host bookkeeping
  int host_start[MAXF + 1];
  int chunk_beg[MAXF + 1];
  std::vector<int> host_of_point;
  std::vector<int> res_slot;   // residual index -> slot (t*mp+p)
  std::vector<uint8_t> h_st_in;
  std::vector<float> h_en_in;
  bool st_in_clean = false;    // every existing residual's INPUT state on the device is IN with zero energy (dmv_ba_reset_oob becomes a flag flip)
  bool timing = false;         // record CUDA events around the kernels of every call (dmv_ba_set_timing)
  int tent = 0;                // index of the tentative buffer set; committed = 1 - tent
  bool have_tentative = false, have_committed = false, have_adj = false, have_state = false;
  long long launches = 0;
  float last_ms[4] = {0, 0, 0, 0};
  // NCCL
  void* nccl_comm = nullptr;
  int nranks = 1, rank = 0;
  // marginalisation launch (dmv_ba_marginalize_points): allocated on first use
  BAMarg* d_marg = nullptr;
  uint8_t* d_marg_mask = nullptr;
  float* d_marg_rtz = nullptr;
  double* d_marg_result = nullptr;
  double* h_marg_result = nullptr;
  float* d_act = nullptr;      // point-activation staging (dmv_ba_activate_points)
  float* h_act = nullptr;
  int act_cap = 0;
  // peer-memory exchange (inside ba_fused_kernel)
  void* xchg_own = nullptr;                 // this rank's inbox (cudaMalloc, exported through CUDA IPC)
  void* xchg_map[XCHG_MAXR] = {nullptr};    // every rank's inbox as mapped here ([rank] == xchg_own)
  int xchg_pitch = 0;
  bool xchg_on = false;
  unsigned int xchg_seq = 0;
};


#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return dmv::set_error(DMV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)); \
  } while (0)

// shared by the product path and the benches (library-internal: hidden from the dynamic symbol table)
#define DMV_INTERNAL extern "C" __attribute__((visibility("hidden")))
DMV_INTERNAL int dmv_ba_fill_descriptor(dmv_ba* b);
DMV_INTERNAL void dmv_ba_next_exchange(dmv_ba* b);
DMV_INTERNAL int dmv_ba_enqueue_exchange(dmv_ba* b);
DMV_INTERNAL void dmv_ba_stage_x(dmv_ba* b, const double* x);
DMV_INTERNAL int dmv_ba_check_ready(dmv_ba* b);
DMV_INTERNAL int dmv_ba_stage_state(dmv_ba* b, const dmv_ba_state* st);
DMV_INTERNAL int dmv_ba_finish_linearize(dmv_ba* b, dmv_ba_lin_result* out, double sums[3]);
