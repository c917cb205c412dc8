// C-ABI of the bundle-adjustment handle (include/dmvio_b200.h).  Host-side plumbing only: buffer ownership, the
// [target][point] residual-slot layout, tentative/committed double buffering, one stream + pinned staging per handle.
#include "ba_handle.h"
#include "ip_trace.h"
#include <algorithm>
#include <cstdlib>
#include <cstring>

using namespace dmv;

// all-reduce of the result blob across ranks: done inside ba_fused_kernel when the peer-memory exchange is on
// (fill_descriptor/next_exchange hand it the inbox table), otherwise one ncclAllReduce behind it
int dmv_ba_enqueue_exchange(dmv_ba* b) {
  if (b->xchg_on) return DMV_OK;
  if (b->nccl_comm) return dmv::nccl_allreduce_double(b->nccl_comm, b->d_result[b->tent], result_doubles(b->N, b->ntiles), b->stream);
  return DMV_OK;
}

int dmv_ba_fill_descriptor(dmv_ba* b) {
  BAWinDev& W = b->h_up->win;
  std::memset(&W, 0, sizeof(W));
  W.nf = b->nf; W.npts = b->npts; W.nchunks = b->nchunks; W.w = b->cfg.w; W.h = b->cfg.h;
  W.N = b->N; W.NW = b->NW; W.T = b->T; W.ntiles = b->ntiles; W.mp = b->mp; W.P = b->P;
  W.huberTH = b->prm.huberTH; W.outlierTHSum = b->prm.outlierTHSumComponent;
  W.zeroA = b->prm.affineOptModeA < 0; W.zeroB = b->prm.affineOptModeB < 0;
  for (int h = 0; h <= MAXF; h++) { W.host_start[h] = b->host_start[h]; W.chunk_beg[h] = b->chunk_beg[h]; }
  for (int f = 0; f < b->nf; f++) W.img[f] = b->d_img[b->slots[f]];
  W.adj = b->d_adj;
  W.uv = b->d_uv;
  W.idepth = b->d_idepth[b->id_cur];
  W.idepth_zero = b->zero_alias ? b->d_idepth[b->id_cur] : b->d_idepth_zero;
  W.idepth_backup = b->d_idepth[b->id_bak];
  W.idepth_out = b->d_idepth[1 - b->id_bak];
  W.color = b->d_color; W.weights = b->d_weights; W.priorF = b->d_priorF;
  const int t = b->tent, c2 = 1 - b->tent;
  // PointFrameResidual::applyRes made state_NewState / state_NewEnergy the residual's state (Residuals.cpp:L325-326): once a
  // linearisation has been committed, the committed outputs ARE the input states (OOB stays OOB, its energy is returned)
  W.st_in = b->have_committed ? b->d_st_new[c2] : b->d_st_in;
  W.en_in = b->have_committed ? b->d_en_new[c2] : b->d_en_in;
  W.en_wo_newest_host = b->h_en_newest;
  W.st_new = b->d_st_new[t]; W.en_new = b->d_en_new[t]; W.en_wo = b->d_en_wo[t]; W.cpt = b->d_cpt[t]; W.jpjd = b->d_jpjd[t]; W.pout = b->d_pout[t];
  W.c_st = b->d_st_new[c2]; W.c_jpjd = b->d_jpjd[c2]; W.c_pout = b->d_pout[c2];
  W.step = b->d_step;
  W.part = b->d_part; W.wg = b->d_wg; W.hdig = b->d_hdig;
  W.bar = b->d_bar;
  W.result = b->d_result[t];
  W.result_host = nullptr;
  W.xc.nranks = b->xchg_on ? b->nranks : 1;
  W.xc.rank = b->rank;
  W.xc.pitch = b->xchg_pitch;
  W.xc.seq = 0;
  for (int r = 0; r < XCHG_MAXR; r++) W.xc.inbox[r] = reinterpret_cast<uint4*>(b->xchg_map[r]);
  return DMV_OK;
}

// every launch of a sharded handle is one exchange: number it (all ranks make the same sequence of launches)
void dmv_ba_next_exchange(dmv_ba* b) {
  if (!b->xchg_on) return;
  b->xchg_seq++;
  if (b->xchg_seq == 0) b->xchg_seq = 2;  // 0 is the "empty" flag; keep the parity sequence alternating after a wrap
  b->h_up->win.xc.seq = b->xchg_seq;
}

extern "C" {

static int ba_allocate(dmv_ba* b, const dmv_ba_config* cfg);

void dmv_ba_default_params(dmv_ba_params* p) {
  p->huberTH = 9.f;
  p->outlierTHSumComponent = 50.f * 50.f;
  p->affineOptModeA = 1e12f;
  p->affineOptModeB = 1e8f;
}

int dmv_ba_create(const dmv_ba_config* cfg, dmv_ba** out) {
  if (!cfg || !out) return set_error(DMV_ERR_INVALID, "null argument");
  if (cfg->max_frames < 2 || cfg->max_frames > DMV_MAX_FRAMES) return set_error(DMV_ERR_INVALID, "max_frames must be in [2,%d]", DMV_MAX_FRAMES);
  if (cfg->w < 16 || cfg->h < 16 || cfg->max_points < 1) return set_error(DMV_ERR_INVALID, "bad size");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return set_error(DMV_ERR_NO_DEVICE, "no CUDA device: dmvio_b200 has no CPU path");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return set_error(DMV_ERR_INVALID, "device %d out of range (%d devices)", cfg->device, ndev);
  CK(cudaSetDevice(cfg->device));
  // L2 -> DRAM fetch granularity: 32 B instead of the driver default 64 B.  The hot path gathers 16-byte texels at data-dependent addresses;
  // with 64-byte fetches every missed 32-byte sector drags its neighbour along: measured 7.58 -> 5.69 MB DRAM reads per launch at C3 (1.38x ->
  // 1.04x the algorithmic bytes, profiles/r02_a_l2fetch_*), no change in kernel time.  A device-wide hint.
  cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32);
  cudaGetLastError();
  dmv_ba* b = new dmv_ba();
  const int rc = ba_allocate(b, cfg);
  if (rc != DMV_OK) {  // e.g. out of device memory half-way: release what was allocated (the error message of the failing call is kept)
    dmv_ba_destroy(b);
    return rc;
  }
  *out = b;
  return DMV_OK;
}

static int ba_allocate(dmv_ba* b, const dmv_ba_config* cfg) {
  b->cfg = *cfg;
  b->device = cfg->device;
  dmv_ba_default_params(&b->prm);
  // chunk_points 16 / 32 force the shape; 0 = per window (dmv_ba_set_points): 16 while the window is one wave of 16-point chunks, else 32
  b->P_auto = !(cfg->chunk_points == 16 || cfg->chunk_points == 32);
  b->P = b->P_auto ? 16 : cfg->chunk_points;
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device) != cudaSuccess || sms < 1) sms = 148;
    b->sms = sms;
  }
  b->mp = (cfg->max_points + 31) & ~31;
  const int MF = MAXF, mp = b->mp;
  b->max_chunks = (mp + (b->P_auto ? 16 : b->P) - 1) / (b->P_auto ? 16 : b->P) + MF;
  const size_t npx = (size_t)cfg->w * cfg->h;
  CK(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
  for (int i = 0; i < 4; i++) CK(cudaEventCreate(&b->ev[i]));
  for (int f = 0; f < cfg->max_frames; f++) CK(cudaMalloc(&b->d_img[f], npx * sizeof(float4)));
  CK(cudaMalloc(&b->d_stage_img, npx * 3 * sizeof(float)));
  CK(cudaMalloc(&b->d_adj, sizeof(BAAdj)));
  CK(cudaMalloc(&b->d_uv, sizeof(float2) * mp));
  CK(cudaMalloc(&b->d_idepth[0], sizeof(float) * mp));
  CK(cudaMalloc(&b->d_idepth[1], sizeof(float) * mp));
  CK(cudaMalloc(&b->d_idepth_zero, sizeof(float) * mp));
  CK(cudaMalloc(&b->d_color, sizeof(float) * mp * 8));
  CK(cudaMalloc(&b->d_weights, sizeof(float) * mp * 8));
  CK(cudaMalloc(&b->d_priorF, sizeof(float) * mp));
  CK(cudaMalloc(&b->d_st_in, (size_t)MF * mp));
  CK(cudaMalloc(&b->d_en_in, sizeof(float) * MF * mp));
  const int maxT0 = (8 * MF + 4 + 1 + 3) / 4, maxTiles0 = maxT0 * (maxT0 + 1) / 2;
  for (int k = 0; k < 2; k++) {
    CK(cudaMalloc(&b->d_st_new[k], (size_t)MF * mp));
    CK(cudaMemset(b->d_st_new[k], 0xff, (size_t)MF * mp));
    CK(cudaMalloc(&b->d_en_new[k], sizeof(float) * MF * mp));
    CK(cudaMalloc(&b->d_en_wo[k], sizeof(float) * MF * mp));
    CK(cudaMalloc(&b->d_cpt[k], sizeof(float) * 3 * MF * mp));
    CK(cudaMalloc(&b->d_jpjd[k], sizeof(float) * 8 * MF * mp));
    CK(cudaMalloc(&b->d_pout[k], sizeof(float) * 8 * mp));
    CK(cudaMemset(b->d_pout[k], 0, sizeof(float) * 8 * mp));
    CK(cudaMalloc(&b->d_result[k], sizeof(double) * result_doubles(8 * MF + 4, maxTiles0)));
    CK(cudaMallocHost(&b->h_result[k], sizeof(double) * result_doubles(8 * MF + 4, maxTiles0)));
  }
  CK(cudaMalloc(&b->d_step, sizeof(float) * mp));
  CK(cudaMemset(b->d_step, 0, sizeof(float) * mp));
  CK(cudaMalloc(&b->d_part, sizeof(double) * PART_STRIDE * (size_t)b->max_chunks));
  CK(cudaMalloc(&b->d_wg, sizeof(float4) * (size_t)maxT0 * mp));
  CK(cudaMalloc(&b->d_hdig, sizeof(float) * mp));
  CK(cudaMalloc(&b->d_hdi_solve, sizeof(float) * mp));
  CK(cudaMalloc(&b->d_bar, sizeof(unsigned int)));
  CK(cudaMemset(b->d_bar, 0, sizeof(unsigned int)));
  CK(cudaMalloc(&b->d_resub_sums, sizeof(double) * 4));
  CK(cudaMallocHost(&b->h_up, sizeof(HostUpload)));
  CK(cudaMallocHost(&b->h_adj, sizeof(BAAdj)));
  std::memset(b->h_up, 0, sizeof(HostUpload));
  b->scratch_floats = std::max((size_t)mp * std::max(8 * MF, 21), npx * 3);   // 21 floats per point: the staged upload of dmv_ba_set_points
  CK(cudaMallocHost(&b->h_scratch, sizeof(float) * b->scratch_floats));
  CK(cudaMallocHost(&b->h_en_newest, sizeof(float) * mp));
  for (int f = 0; f < MF; f++) b->slots[f] = f;
  return DMV_OK;
}

int dmv_ba_destroy(dmv_ba* b) {
  if (!b) return DMV_OK;
  cudaSetDevice(b->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  for (int f = 0; f < MAXF; f++) cudaFree(b->d_img[f]);
  cudaFree(b->d_stage_img); cudaFree(b->d_adj); cudaFree(b->d_uv); cudaFree(b->d_idepth[0]); cudaFree(b->d_idepth[1]);
  cudaFree(b->d_idepth_zero); cudaFree(b->d_color); cudaFree(b->d_weights); cudaFree(b->d_priorF);
  cudaFree(b->d_st_in); cudaFree(b->d_en_in);
  for (int k = 0; k < 2; k++) {
    cudaFree(b->d_st_new[k]); cudaFree(b->d_en_new[k]); cudaFree(b->d_en_wo[k]); cudaFree(b->d_cpt[k]); cudaFree(b->d_jpjd[k]);
    cudaFree(b->d_pout[k]); cudaFree(b->d_result[k]); cudaFreeHost(b->h_result[k]);
  }
  cudaFree(b->d_step); cudaFree(b->d_resub_sums); cudaFree(b->d_flush);
  cudaFree(b->d_part); cudaFree(b->d_wg); cudaFree(b->d_hdig); cudaFree(b->d_hdi_solve); cudaFree(b->d_bar);
  cudaFreeHost(b->h_up); cudaFreeHost(b->h_adj); cudaFreeHost(b->h_scratch); cudaFreeHost(b->h_en_newest);
  for (int i = 0; i < 4; i++) if (b->ev[i]) cudaEventDestroy(b->ev[i]);
  if (b->nccl_comm) dmv::nccl_destroy(b->nccl_comm);
  cudaFree(b->d_act); cudaFreeHost(b->h_act);
  cudaFree(b->d_marg); cudaFree(b->d_marg_mask); cudaFree(b->d_marg_rtz); cudaFree(b->d_marg_result);
  cudaFreeHost(b->h_marg_result);
  for (int r = 0; r < XCHG_MAXR; r++)
    if (b->xchg_map[r] && b->xchg_map[r] != b->xchg_own) cudaIpcCloseMemHandle(b->xchg_map[r]);
  cudaFree(b->xchg_own);
  if (b->stream) cudaStreamDestroy(b->stream);
  delete b;
  return DMV_OK;
}

int dmv_ba_set_params(dmv_ba* b, const dmv_ba_params* p) {
  if (!b || !p) return set_error(DMV_ERR_INVALID, "null argument");
  b->prm = *p;
  return DMV_OK;
}

int dmv_ba_upload_frame(dmv_ba* b, int slot, const float* dI) {
  if (!b || !dI || slot < 0 || slot >= b->cfg.max_frames) return set_error(DMV_ERR_INVALID, "bad slot/pointer");
  CK(cudaSetDevice(b->device));
  const size_t npx = (size_t)b->cfg.w * b->cfg.h;
  std::memcpy(b->h_scratch, dI, npx * 3 * sizeof(float));
  CK(cudaMemcpyAsync(b->d_stage_img, b->h_scratch, npx * 3 * sizeof(float), cudaMemcpyHostToDevice, b->stream));
  launch_repack(b->d_stage_img, b->d_img[slot], (int)npx, b->stream);
  b->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(b->stream));
  return DMV_OK;
}

int dmv_ba_upload_image(dmv_ba* b, int slot, const float* image) {
  if (!b || !image || slot < 0 || slot >= b->cfg.max_frames) return set_error(DMV_ERR_INVALID, "bad slot/pointer");
  CK(cudaSetDevice(b->device));
  const size_t npx = (size_t)b->cfg.w * b->cfg.h;
  std::memcpy(b->h_scratch, image, npx * sizeof(float));
  CK(cudaMemcpyAsync(b->d_stage_img, b->h_scratch, npx * sizeof(float), cudaMemcpyHostToDevice, b->stream));
  launch_make_dI(b->d_stage_img, b->d_img[slot], b->cfg.w, b->cfg.h, b->stream);
  b->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(b->stream));
  return DMV_OK;
}

// FrameHessian::dI of a frame that is ALREADY resident in a coarse-tracker handle (uploaded once when the frame arrived, pyramid built on
// the device): the BA slot takes a device-to-device copy of its level-0 plane (same float4 texel layout) — no second H2D, no second
// makeImages.  Stream-ordered behind whatever the tracker handle still has in flight.
extern "C" int dmv_ct_level0_plane(dmv_ct* c, const void** plane, int* w, int* h, int* device, cudaStream_t* stream);
int dmv_ba_adopt_frame(dmv_ba* b, int slot, dmv_ct* ct) {
  if (!b || !ct || slot < 0 || slot >= b->cfg.max_frames) return set_error(DMV_ERR_INVALID, "bad slot/handle");
  const void* plane = nullptr;
  int w = 0, h = 0, dev = 0;
  cudaStream_t cs = nullptr;
  int rc = dmv_ct_level0_plane(ct, &plane, &w, &h, &dev, &cs);
  if (rc != DMV_OK) return rc;
  if (w != b->cfg.w || h != b->cfg.h) return set_error(DMV_ERR_INVALID, "image size mismatch (%dx%d vs %dx%d)", w, h, b->cfg.w, b->cfg.h);
  if (dev != b->device) return set_error(DMV_ERR_INVALID, "the tracker handle lives on device %d, the BA handle on %d", dev, b->device);
  CK(cudaSetDevice(b->device));
  CK(cudaEventRecord(b->ev[0], cs));                 // the tracker's upload + pyramid kernels
  CK(cudaStreamWaitEvent(b->stream, b->ev[0], 0));
  CK(cudaMemcpyAsync(b->d_img[slot], plane, sizeof(float4) * (size_t)w * h, cudaMemcpyDeviceToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return DMV_OK;
}

int dmv_ba_set_window(dmv_ba* b, int nf, const int* slots) {
  if (!b || nf < 2 || nf > b->cfg.max_frames) return set_error(DMV_ERR_INVALID, "nf out of range");
  for (int f = 0; f < nf; f++) {
    const int s = slots ? slots[f] : f;
    if (s < 0 || s >= b->cfg.max_frames) return set_error(DMV_ERR_INVALID, "slot out of range");
    b->slots[f] = s;
  }
  b->nf = nf;
  b->N = 8 * nf + 4;
  b->NW = (b->N + 1 + 3) & ~3;
  b->T = b->NW / 4;
  b->ntiles = b->T * (b->T + 1) / 2;
  b->have_adj = b->have_state = b->have_tentative = b->have_committed = false;
  b->npts = b->nres = b->nchunks = 0;
  return DMV_OK;
}

int dmv_ba_set_points(dmv_ba* b, int npts, const int32_t* host, const float* u, const float* v, const float* idepth, const float* idepth_zero,
                      const float* color8, const float* weights8, const float* priorF) {
  if (!b || !host || !u || !v || !idepth || !color8 || !weights8) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->nf < 2) return set_error(DMV_ERR_STATE, "dmv_ba_set_window first");
  if (npts < 1 || npts > b->cfg.max_points) return set_error(DMV_ERR_INVALID, "npts %d exceeds capacity %d", npts, b->cfg.max_points);
  for (int i = 0; i < npts; i++) {
    if (host[i] < 0 || host[i] >= b->nf) return set_error(DMV_ERR_INVALID, "point %d: host %d out of range", i, host[i]);
    if (i > 0 && host[i] < host[i - 1]) return set_error(DMV_ERR_INVALID, "points must be ordered by host frame (EnergyFunctional::allPoints order)");
  }
  CK(cudaSetDevice(b->device));
  b->npts = npts;
  b->host_of_point.assign(host, host + npts);
  // one thread per residual (P = 32, fewest instructions) pays off once the window no longer fits one wave of 16-point chunks (measured at
  // 7 KF / 8000 points: 54 vs 68 us per step); below that the 4-lanes-per-residual shape (P = 16) has the shorter critical path (29.6 vs 37.9 us)
  if (b->P_auto) b->P = (npts > 16 * b->sms) ? 32 : 16;
  {
    int p = 0, c = 0;
    for (int h = 0; h < MAXF; h++) {
      b->host_start[h] = p;
      b->chunk_beg[h] = c;
      int cnt = 0;
      while (p < npts && host[p] == h) { p++; cnt++; }
      c += (cnt + b->P - 1) / b->P;
    }
    b->host_start[MAXF] = npts;
    b->chunk_beg[MAXF] = c;
    b->nchunks = c;
  }
  if (b->nchunks > b->max_chunks) return set_error(DMV_ERR_INVALID, "too many chunks");
  // one pinned staging block, the copies queued back to back, ONE synchronisation (was: seven blocking copies from pageable memory)
  float* s = b->h_scratch;   // >= 8 * MAXF * mp floats
  const size_t n = (size_t)npts;
  float *s_uv = s, *s_id = s + 2 * n, *s_idz = s + 3 * n, *s_col = s + 4 * n, *s_w = s + 12 * n, *s_pr = s + 20 * n;
  for (int i = 0; i < npts; i++) { s_uv[2 * i] = u[i]; s_uv[2 * i + 1] = v[i]; }
  std::memcpy(s_id, idepth, sizeof(float) * n);
  if (idepth_zero) std::memcpy(s_idz, idepth_zero, sizeof(float) * n);
  std::memcpy(s_col, color8, sizeof(float) * 8 * n);
  std::memcpy(s_w, weights8, sizeof(float) * 8 * n);
  if (priorF) std::memcpy(s_pr, priorF, sizeof(float) * n);
  b->id_cur = b->id_bak = 0;
  b->zero_alias = (idepth_zero == nullptr);
  CK(cudaMemcpyAsync(b->d_uv, s_uv, sizeof(float2) * n, cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemcpyAsync(b->d_idepth[0], s_id, sizeof(float) * n, cudaMemcpyHostToDevice, b->stream));
  if (idepth_zero) CK(cudaMemcpyAsync(b->d_idepth_zero, s_idz, sizeof(float) * n, cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemcpyAsync(b->d_color, s_col, sizeof(float) * 8 * n, cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemcpyAsync(b->d_weights, s_w, sizeof(float) * 8 * n, cudaMemcpyHostToDevice, b->stream));
  if (priorF) CK(cudaMemcpyAsync(b->d_priorF, s_pr, sizeof(float) * n, cudaMemcpyHostToDevice, b->stream));
  else CK(cudaMemsetAsync(b->d_priorF, 0, sizeof(float) * n, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->nres = 0;
  b->hdi_solve_n = 0;
  b->en_newest_valid = false;
  b->have_tentative = b->have_committed = false;
  return DMV_OK;
}

int dmv_ba_set_residuals(dmv_ba* b, int nres, const int32_t* point, const int32_t* target, const int32_t* state_state, const float* state_energy) {
  if (!b || !point || !target || nres < 0) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->npts < 1) return set_error(DMV_ERR_STATE, "dmv_ba_set_points first");
  CK(cudaSetDevice(b->device));
  const size_t ns = (size_t)MAXF * b->mp;
  b->h_st_in.assign(ns, (uint8_t)RES_NONE);
  b->h_en_in.assign(ns, 0.f);
  b->res_slot.resize(nres);
  for (int i = 0; i < nres; i++) {
    const int p = point[i], t = target[i];
    if (p < 0 || p >= b->npts || t < 0 || t >= b->nf) return set_error(DMV_ERR_INVALID, "residual %d out of range", i);
    if (t == b->host_of_point[p]) return set_error(DMV_ERR_INVALID, "residual %d targets its own host frame", i);
    const size_t slot = (size_t)t * b->mp + p;
    if (b->h_st_in[slot] != RES_NONE) return set_error(DMV_ERR_INVALID, "duplicate residual (point %d, target %d)", p, t);
    const int st = state_state ? state_state[i] : RES_IN;
    if (st < 0 || st > 2) return set_error(DMV_ERR_INVALID, "residual %d: bad state %d", i, st);
    b->h_st_in[slot] = (uint8_t)st;
    b->h_en_in[slot] = state_energy ? state_energy[i] : 0.f;
    b->res_slot[i] = (int)slot;
  }
  b->nres = nres;
  b->st_in_clean = true;
  for (int i = 0; i < nres; i++)
    if (b->h_st_in[b->res_slot[i]] != RES_IN || b->h_en_in[b->res_slot[i]] != 0.f) { b->st_in_clean = false; break; }
  CK(cudaMemcpyAsync(b->d_st_in, b->h_st_in.data(), ns, cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemcpyAsync(b->d_en_in, b->h_en_in.data(), ns * sizeof(float), cudaMemcpyHostToDevice, b->stream));
  for (int k = 0; k < 2; k++) CK(cudaMemsetAsync(b->d_st_new[k], 0xff, ns, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->have_tentative = b->have_committed = false;
  return DMV_OK;
}

int dmv_ba_set_adjoints(dmv_ba* b, const double* adHost, const double* adTarget) {
  if (!b || !adHost || !adTarget) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->nf < 2) return set_error(DMV_ERR_STATE, "dmv_ba_set_window first");
  CK(cudaSetDevice(b->device));
  const int nf = b->nf;
  BAAdj* A = b->h_adj;
  std::memset(A, 0, sizeof(BAAdj));
  for (int h = 0; h < nf; h++)
    for (int t = 0; t < nf; t++) {
      const double* ah = adHost + (size_t)(h + t * nf) * 64;
      const double* at = adTarget + (size_t)(h + t * nf) * 64;
      const int d = h * nf + t;
      for (int k = 0; k < 64; k++) { A->adHost[d][k] = ah[k]; A->adHostF[d][k] = (float)ah[k]; }
      for (int k = 0; k < 8; k++) {
        for (int c = 0; c < 8; c++)
          if (c != k && at[k * 8 + c] != 0.0) return set_error(DMV_ERR_INVALID, "adTarget[%d,%d] is not diagonal (EnergyFunctional.cpp:L66-84 makes it diagonal)", h, t);
        A->adTdiag[d][k] = at[k * 8 + k];
        A->adTdiagF[d][k] = (float)at[k * 8 + k];
      }
    }
  CK(cudaMemcpyAsync(b->d_adj, A, sizeof(BAAdj), cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->have_adj = true;
  return DMV_OK;
}

int dmv_ba_stage_state(dmv_ba* b, const dmv_ba_state* st) {
  if (!st->precalc || !st->frameEnergyTH) return set_error(DMV_ERR_INVALID, "precalc / frameEnergyTH required");
  BAIter& it = b->h_up->it;
  const int nf = b->nf;
  std::memcpy(it.calib, st->calib, sizeof(it.calib));
  for (int f = 0; f < nf; f++) it.TH[f] = st->frameEnergyTH[f];
  std::memcpy(it.precalc, st->precalc, sizeof(float) * 32 * nf * nf);
  if (st->idepth) CK(cudaMemcpyAsync(b->d_idepth[b->id_cur], st->idepth, sizeof(float) * b->npts, cudaMemcpyHostToDevice, b->stream));
  if (st->idepth_zero) {
    CK(cudaMemcpyAsync(b->d_idepth_zero, st->idepth_zero, sizeof(float) * b->npts, cudaMemcpyHostToDevice, b->stream));
    b->zero_alias = false;
  }
  b->have_state = true;
  return DMV_OK;
}

int dmv_ba_set_state(dmv_ba* b, const dmv_ba_state* st) {
  if (!b || !st) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->npts < 1) return set_error(DMV_ERR_STATE, "dmv_ba_set_points first");
  CK(cudaSetDevice(b->device));
  int rc = dmv_ba_stage_state(b, st);
  if (rc != DMV_OK) return rc;
  // pageable idepth sources: make the async copies complete before returning
  CK(cudaStreamSynchronize(b->stream));
  return DMV_OK;
}

static int enqueue_linearize(dmv_ba* b) {
  dmv_ba_fill_descriptor(b);
  dmv_ba_next_exchange(b);
  // the kernel writes the final blob into the pinned host mirror itself, unless a NCCL all-reduce still follows it
  const bool zero_copy = !(b->nccl_comm && !b->xchg_on);
  double* hres = b->h_result[b->tent];
  hres[(size_t)b->N * b->N + b->N + (size_t)b->ntiles * 16 + (ACC_MISC - 1)] = 0.0;  // error flag: written by the device on a timeout only
  if (zero_copy) b->h_up->win.result_host = hres;
  else  // the NCCL all-reduce sums the device copy of the slot: it must not carry a stale value (e.g. from a window of another size)
    CK(cudaMemsetAsync(b->d_result[b->tent] + (size_t)b->N * b->N + b->N + (size_t)b->ntiles * 16 + (ACC_MISC - 1), 0, sizeof(double), b->stream));
  HostUpload& U = *b->h_up;
  if (b->timing) CK(cudaEventRecord(b->ev[0], b->stream));
  CK(launch_fused_kernel(U.win, U.it, false, b->stream, &b->bar_count));  // whole linearisation: residuals -> H_top, b_top, [H_sc | b_sc]
  b->en_newest_valid = true;
  b->launches += 1;
  if (b->timing) CK(cudaEventRecord(b->ev[1], b->stream));
  {
    int rc = dmv_ba_enqueue_exchange(b);
    if (rc != DMV_OK) return rc;
  }
  if (!zero_copy)
    CK(cudaMemcpyAsync(b->h_result[b->tent], b->d_result[b->tent], sizeof(double) * result_doubles(b->N, b->ntiles), cudaMemcpyDeviceToHost, b->stream));
  if (b->timing) CK(cudaEventRecord(b->ev[3], b->stream));
  return DMV_OK;
}

int dmv_ba_finish_linearize(dmv_ba* b, dmv_ba_lin_result* out, double sums[3]) {
  if (b->h_up->it.have_x) { b->id_cur = 1 - b->id_bak; b->zero_alias = true; }  // the fused step wrote idepth_backup + step
  CK(cudaStreamSynchronize(b->stream));
  const double* tail = b->h_result[b->tent] + (b->N * b->N + b->N) + b->ntiles * 16;
  if (out) { out->energy = tail[0]; out->n_in = (int)tail[1]; out->n_oob = (int)tail[2]; out->n_outlier = (int)tail[3]; }
  if (sums) { sums[0] = tail[4]; sums[1] = tail[5]; sums[2] = tail[6]; }
  if (b->timing) {
    cudaEventElapsedTime(&b->last_ms[0], b->ev[0], b->ev[3]);
    cudaEventElapsedTime(&b->last_ms[1], b->ev[0], b->ev[1]);
    b->last_ms[2] = 0.f;
    cudaEventElapsedTime(&b->last_ms[3], b->ev[1], b->ev[3]);
  }
  if (tail[ACC_MISC - 1] != 0.0) return set_error(DMV_ERR_TIMEOUT, "grid barrier / peer exchange timed out inside ba_fused_kernel (a rank or CTA went missing)");
  b->have_tentative = true;
  return DMV_OK;
}

int dmv_ba_check_ready(dmv_ba* b) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  if (b->npts < 1 || b->nres < 0) return set_error(DMV_ERR_STATE, "points/residuals not set");
  if (!b->have_adj) return set_error(DMV_ERR_STATE, "dmv_ba_set_adjoints first");
  if (!b->have_state) return set_error(DMV_ERR_STATE, "dmv_ba_set_state first");
  return DMV_OK;
}

int dmv_ba_linearize(dmv_ba* b, dmv_ba_lin_result* out) {
  int rc = dmv_ba_check_ready(b);
  if (rc != DMV_OK) return rc;
  CK(cudaSetDevice(b->device));
  b->h_up->it.have_x = 0;
  rc = enqueue_linearize(b);
  if (rc != DMV_OK) return rc;
  return dmv_ba_finish_linearize(b, out, nullptr);
}

void dmv_ba_stage_x(dmv_ba* b, const double* x) {
  // EnergyFunctional::resubstituteF_MT (EnergyFunctional.cpp:L272-283): xAd[h*nf+t] = x_h^T adHostF + x_t^T adTargetF in float
  BAIter& it = b->h_up->it;
  const int nf = b->nf;
  const BAAdj* A = b->h_adj;
  for (int i = 0; i < 4; i++) it.xc[i] = (float)x[i];
  for (int h = 0; h < nf; h++)
    for (int t = 0; t < nf; t++) {
      const int d = h * nf + t;
      for (int c = 0; c < 8; c++) {
        float a = 0.f;
        for (int k = 0; k < 8; k++) a += (float)x[4 + 8 * h + k] * A->adHostF[d][k * 8 + c];
        const float bb = (float)x[4 + 8 * t + c] * A->adTdiagF[d][c];
        it.xAd[d][c] = a + bb;
      }
    }
  it.have_x = 1;
}

int dmv_ba_resubstitute(dmv_ba* b, const double* x, float* step_out, int apply, double sums[3]) {
  int rc = dmv_ba_check_ready(b);
  if (rc != DMV_OK) return rc;
  if (!x) return set_error(DMV_ERR_INVALID, "x is null");
  if (!b->have_committed) return set_error(DMV_ERR_STATE, "no committed linearisation (linearize + apply_res first)");
  CK(cudaSetDevice(b->device));
  dmv_ba_stage_x(b, x);
  dmv_ba_fill_descriptor(b);
  CK(cudaMemsetAsync(b->d_resub_sums, 0, sizeof(double) * 4, b->stream));
  launch_resub_kernel(b->h_up->win, b->h_up->it, apply, b->d_resub_sums, b->stream);
  b->launches += 1;
  CK(cudaGetLastError());
  double tail[8] = {0};
  CK(cudaMemcpyAsync(tail + 4, b->d_resub_sums, sizeof(double) * 3, cudaMemcpyDeviceToHost, b->stream));
  if (step_out) CK(cudaMemcpyAsync(step_out, b->d_step, sizeof(float) * b->npts, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  if (sums) { sums[0] = tail[4]; sums[1] = tail[5]; sums[2] = tail[6]; }
  if (apply) { b->id_cur = 1 - b->id_bak; b->zero_alias = true; }
  b->h_up->it.have_x = 0;
  return DMV_OK;
}

int dmv_ba_gn_step(dmv_ba* b, const double* x, const dmv_ba_state* st, dmv_ba_lin_result* out, double sums[3]) {
  if (!b || !st) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->npts < 1) return set_error(DMV_ERR_STATE, "points not set");
  if (!b->have_adj) return set_error(DMV_ERR_STATE, "dmv_ba_set_adjoints first");
  if (x && !b->have_committed) return set_error(DMV_ERR_STATE, "no committed linearisation to resubstitute");
  CK(cudaSetDevice(b->device));
  int rc = dmv_ba_stage_state(b, st);
  if (rc != DMV_OK) return rc;
  if (x) dmv_ba_stage_x(b, x); else b->h_up->it.have_x = 0;
  rc = enqueue_linearize(b);
  if (rc != DMV_OK) return rc;
  rc = dmv_ba_finish_linearize(b, out, sums);
  b->h_up->it.have_x = 0;
  return rc;
}

int dmv_ba_backup_points(dmv_ba* b) {
  if (!b || b->npts < 1) return set_error(DMV_ERR_STATE, "points not set");
  b->id_bak = b->id_cur;  // ping-pong: the next step writes the other buffer, nothing is copied
  return DMV_OK;
}
int dmv_ba_restore_points(dmv_ba* b) {
  if (!b || b->npts < 1) return set_error(DMV_ERR_STATE, "points not set");
  b->id_cur = b->id_bak;
  b->zero_alias = true;   // loadSateBackup: setIdepthZero(idepth_backup) (FullSystemOptimize.cpp:L380)
  return DMV_OK;
}
int dmv_ba_get_idepth(dmv_ba* b, float* idepth, float* idepth_zero) {
  if (!b || b->npts < 1) return set_error(DMV_ERR_STATE, "points not set");
  CK(cudaSetDevice(b->device));
  CK(cudaStreamSynchronize(b->stream));
  if (idepth) CK(cudaMemcpy(idepth, b->d_idepth[b->id_cur], sizeof(float) * b->npts, cudaMemcpyDeviceToHost));
  if (idepth_zero) CK(cudaMemcpy(idepth_zero, b->zero_alias ? b->d_idepth[b->id_cur] : b->d_idepth_zero, sizeof(float) * b->npts, cudaMemcpyDeviceToHost));
  return DMV_OK;
}

int dmv_ba_apply_res(dmv_ba* b) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  if (!b->have_tentative) return set_error(DMV_ERR_STATE, "no tentative linearisation to commit");
  b->tent = 1 - b->tent;
  b->have_committed = true;
  b->have_tentative = false;
  return DMV_OK;
}

static void unpack_system(const dmv_ba* b, const double* r, double* H_A, double* b_A, double* H_sc, double* b_sc, int* resInA);

int dmv_ba_accumulate(dmv_ba* b, double* H_A, double* b_A, double* H_sc, double* b_sc, int* resInA) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  if (!b->have_committed) return set_error(DMV_ERR_STATE, "no committed linearisation (linearize + apply_res first)");
  unpack_system(b, b->h_result[1 - b->tent], H_A, b_A, H_sc, b_sc, resInA);
  // AccumulatedSCHessian::addPoint is also what writes EFPoint::HdiF / PointHessian::idepth_hessian (AccumulatedSCHessian.cpp:L42-50): keep
  // the HdiF of THIS linearisation on the device (strided device-to-device copy on the handle's stream, no synchronisation) — later
  // linearisations overwrite the per-point output buffers, dmv_ba_get_solve_HdiF() still returns these
  CK(cudaSetDevice(b->device));
  CK(cudaMemcpy2DAsync(b->d_hdi_solve, sizeof(float), b->d_pout[1 - b->tent] + 6, 8 * sizeof(float), sizeof(float), b->npts, cudaMemcpyDeviceToDevice, b->stream));
  b->hdi_solve_n = b->npts;
  return DMV_OK;
}

int dmv_ba_get_solve_HdiF(dmv_ba* b, float* HdiF) {
  if (!b || !HdiF) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->hdi_solve_n != b->npts || b->npts < 1) return set_error(DMV_ERR_STATE, "no dmv_ba_accumulate since the points were set");
  CK(cudaSetDevice(b->device));
  CK(cudaMemcpyAsync(HdiF, b->d_hdi_solve, sizeof(float) * b->npts, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return DMV_OK;
}

// result blob -> dense top system + Schur complement (shared by dmv_ba_accumulate and dmv_ba_marginalize_points)
static void unpack_system(const dmv_ba* b, const double* r, double* H_A, double* b_A, double* H_sc, double* b_sc, int* resInA) {
  const int N = b->N, T = b->T;
  if (H_A) {
    std::memcpy(H_A, r, sizeof(double) * N * N);
    for (int i = 4; i < N; i++)  // the device fills H[frame,C]; mirror into H[C,frame] (AccumulatedTopHessian.h:L127-130)
      for (int c = 0; c < 4; c++) H_A[(size_t)c * N + i] = H_A[(size_t)i * N + c];
  }
  if (b_A) std::memcpy(b_A, r + (size_t)N * N, sizeof(double) * N);
  const double* sc = r + (size_t)N * N + N;  // raw upper-triangular 4x4 Gram tiles of [H_sc | b_sc] (ba_fused.cu, phase E)
  auto gram = [&](int rr, int cc) {
    if (cc < N && rr > cc) std::swap(rr, cc);
    const int ti = rr >> 2, tj = cc >> 2;
    const int tile = ti * T - (ti * (ti - 1)) / 2 + (tj - ti);
    return sc[(size_t)tile * 16 + (rr & 3) * 4 + (cc & 3)];
  };
  if (H_sc)
    for (int i = 0; i < N; i++)
      for (int j = 0; j < N; j++) H_sc[(size_t)i * N + j] = gram(i, j);
  if (b_sc)
    for (int i = 0; i < N; i++) b_sc[i] = gram(i, N);
  if (resInA) *resInA = (int)sc[(size_t)b->ntiles * 16 + 1];
}

int dmv_ba_reset_oob(dmv_ba* b) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  if (b->npts < 1) return set_error(DMV_ERR_STATE, "points/residuals not set");
  CK(cudaSetDevice(b->device));
  const size_t ns = (size_t)MAXF * b->mp;
  if (!b->st_in_clean) {  // otherwise the input arrays already say "IN, energy 0" for every residual: switching back to them is the reset
    for (int i = 0; i < b->nres; i++) { b->h_st_in[b->res_slot[i]] = (uint8_t)RES_IN; b->h_en_in[b->res_slot[i]] = 0.f; }
    CK(cudaStreamSynchronize(b->stream));
    CK(cudaMemcpy(b->d_st_in, b->h_st_in.data(), ns, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_en_in, b->h_en_in.data(), ns * sizeof(float), cudaMemcpyHostToDevice));
    b->st_in_clean = true;
  }
  b->have_tentative = b->have_committed = false;
  return DMV_OK;
}

int dmv_ba_drop_residuals(dmv_ba* b, int n, const int32_t* res_idx) {
  if (!b || n < 0 || (n > 0 && !res_idx)) return set_error(DMV_ERR_INVALID, "null argument");
  if (n == 0) return DMV_OK;
  CK(cudaSetDevice(b->device));
  std::vector<char> gone(b->nres, 0);
  for (int i = 0; i < n; i++) {
    if (res_idx[i] < 0 || res_idx[i] >= b->nres) return set_error(DMV_ERR_INVALID, "res_idx[%d] = %d out of range", i, res_idx[i]);
    gone[res_idx[i]] = 1;
  }
  // once per keyframe, <= 64 KB per array: round-trip the state arrays instead of a scatter kernel
  const size_t ns = (size_t)MAXF * b->mp;
  CK(cudaStreamSynchronize(b->stream));
  std::vector<uint8_t> st(ns);
  for (int k = 0; k < 2; k++) {
    CK(cudaMemcpy(st.data(), b->d_st_new[k], ns, cudaMemcpyDeviceToHost));
    for (int i = 0; i < b->nres; i++) if (gone[i]) st[b->res_slot[i]] = (uint8_t)RES_NONE;
    CK(cudaMemcpy(b->d_st_new[k], st.data(), ns, cudaMemcpyHostToDevice));
  }
  int w = 0;
  for (int i = 0; i < b->nres; i++) {
    if (gone[i]) { b->h_st_in[b->res_slot[i]] = (uint8_t)RES_NONE; b->h_en_in[b->res_slot[i]] = 0.f; }
    else b->res_slot[w++] = b->res_slot[i];
  }
  b->nres = w;
  b->res_slot.resize(w);
  CK(cudaMemcpy(b->d_st_in, b->h_st_in.data(), ns, cudaMemcpyHostToDevice));
  return DMV_OK;
}

int dmv_ba_marginalize_points(dmv_ba* b, const dmv_ba_marg_args* a) {
  int rc = dmv_ba_check_ready(b);
  if (rc != DMV_OK) return rc;
  if (!a || a->n < 0 || (a->n > 0 && !a->point) || !a->adHTdeltaF) return set_error(DMV_ERR_INVALID, "null argument");
  CK(cudaSetDevice(b->device));
  const int nf = b->nf, N = b->N;
  const size_t nres_d = result_doubles(N, b->ntiles), nslots = (size_t)MAXF * b->mp;
  if (!b->d_marg) {
    CK(cudaMalloc(&b->d_marg, sizeof(BAMarg)));
    CK(cudaMalloc(&b->d_marg_mask, b->mp));
    CK(cudaMalloc(&b->d_marg_rtz, sizeof(float) * 8 * nslots));
    const size_t maxres = result_doubles(8 * MAXF + 4, ((2 * MAXF + 2) * (2 * MAXF + 3)) / 2);
    CK(cudaMalloc(&b->d_marg_result, sizeof(double) * maxres));
    CK(cudaHostAlloc(&b->h_marg_result, sizeof(double) * maxres, cudaHostAllocDefault));
  }
  // tables
  BAMarg M;
  std::memset(&M, 0, sizeof(M));
  for (int h = 0; h < nf; h++)
    for (int t = 0; t < nf; t++) std::memcpy(M.adHTdelta[h * nf + t], a->adHTdeltaF + (size_t)(h + t * nf) * 8, sizeof(float) * 8);
  std::memcpy(M.cDelta, a->cDeltaF, sizeof(M.cDelta));
  M.priorFac = a->idepthFixPriorMargFac;
  std::vector<uint8_t> mask(b->mp, 0);
  for (int i = 0; i < a->n; i++) {
    if (a->point[i] < 0 || a->point[i] >= b->npts) return set_error(DMV_ERR_INVALID, "point[%d] = %d out of range", i, a->point[i]);
    mask[a->point[i]] = 1;
  }
  CK(cudaMemcpyAsync(b->d_marg, &M, sizeof(M), cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemcpyAsync(b->d_marg_mask, mask.data(), b->mp, cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemsetAsync(b->d_marg_rtz, 0, sizeof(float) * 8 * nslots, b->stream));
  // descriptor: the production one with a private result blob and no fused step.  On a sharded window every rank marginalises ITS flagged points
  // (n may be 0) and the partial M / Msc are summed over the ranks like any other linearisation (EnergyFunctional.cpp:L678-742 is a sum over
  // points): every rank must make this call at the same place of its launch sequence; all end with the identical full M, Msc
  b->h_up->it.have_x = 0;
  dmv_ba_fill_descriptor(b);
  dmv_ba_next_exchange(b);
  BAWinDev& W = b->h_up->win;
  W.result = b->d_marg_result;
  W.result_host = nullptr;
  W.en_wo_newest_host = nullptr;
  W.marg = b->d_marg; W.marg_mask = b->d_marg_mask; W.marg_rtz = b->d_marg_rtz;
  CK(cudaMemsetAsync(b->d_marg_result + nres_d - 1, 0, sizeof(double), b->stream));   // error slot: written by the device on a timeout only
  CK(launch_fused_kernel(W, b->h_up->it, true, b->stream, &b->bar_count));
  b->launches += 1;
  if (b->nccl_comm && !b->xchg_on) {
    const int rcx = dmv::nccl_allreduce_double(b->nccl_comm, b->d_marg_result, (int)nres_d, b->stream);
    if (rcx != DMV_OK) return rcx;
  }
  CK(cudaMemcpyAsync(b->h_marg_result, b->d_marg_result, sizeof(double) * nres_d, cudaMemcpyDeviceToHost, b->stream));
  std::vector<uint8_t> st(nslots);
  std::vector<float> rtz;
  CK(cudaMemcpyAsync(st.data(), b->d_st_new[b->tent], nslots, cudaMemcpyDeviceToHost, b->stream));
  if (a->res_toZeroF) {
    rtz.resize(8 * nslots);
    CK(cudaMemcpyAsync(rtz.data(), b->d_marg_rtz, sizeof(float) * 8 * nslots, cudaMemcpyDeviceToHost, b->stream));
  }
  CK(cudaStreamSynchronize(b->stream));
  b->have_tentative = false;  // the tentative buffers now hold the flagged points' re-linearisation only
  if (b->h_marg_result[nres_d - 1] != 0.0)
    return set_error(DMV_ERR_TIMEOUT, "grid barrier / peer exchange timed out inside ba_fused_kernel (marginalisation launch)");
  unpack_system(b, b->h_marg_result, a->M, a->Mb, a->Msc, a->Mbsc, nullptr);
  if (a->resInM) *a->resInM = (int)b->h_marg_result[(size_t)N * N + N + (size_t)b->ntiles * 16 + 1];
  std::vector<int> good(b->mp, 0);
  for (int i = 0; i < b->nres; i++) {
    const int slot = b->res_slot[i], p = slot % b->mp;
    const bool lin = mask[p] && st[slot] == RES_IN;
    if (lin) good[p]++;
    if (a->isLinearized) a->isLinearized[i] = lin ? 1 : 0;
    if (a->res_toZeroF)
      for (int c = 0; c < 8; c++) a->res_toZeroF[(size_t)i * 8 + c] = lin ? rtz[(size_t)slot * 8 + c] : 0.f;
  }
  if (a->ngoodRes)
    for (int i = 0; i < a->n; i++) a->ngoodRes[i] = good[a->point[i]];
  return DMV_OK;
}

static int fetch_f(dmv_ba* b, const float* dsrc, size_t n) {
  if (n > b->scratch_floats) return set_error(DMV_ERR_INVALID, "scratch too small");
  CK(cudaMemcpyAsync(b->h_scratch, dsrc, n * sizeof(float), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return DMV_OK;
}

int dmv_ba_get_residual_outputs(dmv_ba* b, int32_t* newState, float* newEnergy, float* newEnergyWithOutlier, float* cpt3, float* JpJdF8) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  if (!b->have_tentative && !b->have_committed) return set_error(DMV_ERR_STATE, "linearize first");
  CK(cudaSetDevice(b->device));
  const int k = b->have_tentative ? b->tent : 1 - b->tent;  // most recent linearisation
  const size_t ns = (size_t)MAXF * b->mp;
  int rc;
  if (newState) {
    std::vector<uint8_t> tmp(ns);
    CK(cudaMemcpy(tmp.data(), b->d_st_new[k], ns, cudaMemcpyDeviceToHost));
    for (int i = 0; i < b->nres; i++) newState[i] = tmp[b->res_slot[i]];
  }
  if (newEnergy) {
    if ((rc = fetch_f(b, b->d_en_new[k], ns)) != DMV_OK) return rc;
    for (int i = 0; i < b->nres; i++) newEnergy[i] = b->h_scratch[b->res_slot[i]];
  }
  if (newEnergyWithOutlier) {
    if ((rc = fetch_f(b, b->d_en_wo[k], ns)) != DMV_OK) return rc;
    for (int i = 0; i < b->nres; i++) newEnergyWithOutlier[i] = b->h_scratch[b->res_slot[i]];
  }
  if (cpt3) {
    if ((rc = fetch_f(b, b->d_cpt[k], 3 * ns)) != DMV_OK) return rc;
    for (int i = 0; i < b->nres; i++)
      for (int c = 0; c < 3; c++) cpt3[3 * i + c] = b->h_scratch[c * ns + b->res_slot[i]];
  }
  if (JpJdF8) {
    if ((rc = fetch_f(b, b->d_jpjd[k], 8 * ns)) != DMV_OK) return rc;
    for (int i = 0; i < b->nres; i++)
      for (int c = 0; c < 8; c++) JpJdF8[8 * i + c] = b->h_scratch[(size_t)b->res_slot[i] * 8 + c];
  }
  return DMV_OK;
}

int dmv_ba_get_target_energies(dmv_ba* b, int target, float* out, int cap, int* n) {
  if (!b || !out || !n || target < 0 || target >= b->nf) return set_error(DMV_ERR_INVALID, "bad argument");
  if (!b->have_tentative && !b->have_committed) return set_error(DMV_ERR_STATE, "linearize first");
  CK(cudaSetDevice(b->device));
  const int k = b->have_tentative ? b->tent : 1 - b->tent;
  const float* src = b->h_scratch;
  if (target == b->nf - 1 && b->en_newest_valid) {
    src = b->h_en_newest;   // the kernel streamed these into pinned host memory itself; every launch is followed by a stream synchronisation
  } else {
    int rc = fetch_f(b, b->d_en_wo[k] + (size_t)target * b->mp, b->npts);
    if (rc != DMV_OK) return rc;
  }
  int c = 0;
  for (int p = 0; p < b->npts && c < cap; p++)
    if (b->h_st_in[(size_t)target * b->mp + p] != RES_NONE && src[p] >= 0.f) out[c++] = src[p];
  *n = c;
  return DMV_OK;
}

int dmv_ba_get_point_outputs(dmv_ba* b, float* Hdd, float* bd, float* Hcd4, float* HdiF, float* bdSumF) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  if (!b->have_tentative && !b->have_committed) return set_error(DMV_ERR_STATE, "linearize first");
  CK(cudaSetDevice(b->device));
  const int k = b->have_tentative ? b->tent : 1 - b->tent;
  int rc = fetch_f(b, b->d_pout[k], (size_t)8 * b->npts);
  if (rc != DMV_OK) return rc;
  for (int p = 0; p < b->npts; p++) {
    const float* r = b->h_scratch + (size_t)8 * p;
    if (Hdd) Hdd[p] = r[0];
    if (bd) bd[p] = r[1];
    if (Hcd4) { Hcd4[4 * p] = r[2]; Hcd4[4 * p + 1] = r[3]; Hcd4[4 * p + 2] = r[4]; Hcd4[4 * p + 3] = r[5]; }
    if (HdiF) HdiF[p] = r[6];
    if (bdSumF) bdSumF[p] = r[7];
  }
  return DMV_OK;
}

int dmv_ba_last_timing(dmv_ba* b, float ms[4]) {
  if (!b || !ms) return set_error(DMV_ERR_INVALID, "null argument");
  for (int i = 0; i < 4; i++) ms[i] = b->last_ms[i];
  return DMV_OK;
}

int dmv_ba_kernel_launch_count(dmv_ba* b, long long* n) {
  if (!b || !n) return set_error(DMV_ERR_INVALID, "null argument");
  *n = b->launches;
  return DMV_OK;
}

int dmv_nccl_unique_id(void* id128) { return dmv::nccl_unique_id(id128); }

int dmv_ba_comm_init(dmv_ba* b, int nranks, int rank, const void* id) {
  if (!b || !id || nranks < 1 || rank < 0 || rank >= nranks) return set_error(DMV_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(b->device));
  if (nranks == 1) return DMV_OK;
  int rc = dmv::nccl_init(&b->nccl_comm, nranks, rank, id);
  if (rc != DMV_OK) return rc;
  b->nranks = nranks; b->rank = rank;
  return DMV_OK;
}

}  // extern "C"

// ---- peer-memory exchange set-up (CUDA IPC): export this rank's inbox, import everybody's
extern "C" int dmv_ba_p2p_export(dmv_ba* b, void* ipc_handle64) {
  if (!b || !ipc_handle64) return set_error(DMV_ERR_INVALID, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CK(cudaSetDevice(b->device));
  if (!b->xchg_own) {
    const int maxT = (8 * MAXF + 4 + 1 + 3) / 4, maxTiles = maxT * (maxT + 1) / 2;
    b->xchg_pitch = (result_doubles(8 * MAXF + 4, maxTiles) + 7) & ~7;
    const size_t bytes = (size_t)2 * XCHG_MAXR * b->xchg_pitch * sizeof(uint4);
    CK(cudaMalloc(&b->xchg_own, bytes));
    CK(cudaMemset(b->xchg_own, 0, bytes));
    CK(cudaDeviceSynchronize());
  }
  cudaIpcMemHandle_t hdl;
  CK(cudaIpcGetMemHandle(&hdl, b->xchg_own));
  std::memcpy(ipc_handle64, &hdl, 64);
  return DMV_OK;
}

extern "C" int dmv_ba_p2p_import(dmv_ba* b, int nranks, int rank, const void* ipc_handles) {
  if (!b || !ipc_handles || nranks < 1 || nranks > XCHG_MAXR || rank < 0 || rank >= nranks) return set_error(DMV_ERR_INVALID, "bad argument (1..%d ranks)", XCHG_MAXR);
  if (!b->xchg_own) return set_error(DMV_ERR_STATE, "dmv_ba_p2p_export first");
  CK(cudaSetDevice(b->device));
  for (int r = 0; r < nranks; r++) {
    if (r == rank) { b->xchg_map[r] = b->xchg_own; continue; }
    cudaIpcMemHandle_t hdl;
    std::memcpy(&hdl, static_cast<const char*>(ipc_handles) + (size_t)r * 64, 64);
    CK(cudaIpcOpenMemHandle(&b->xchg_map[r], hdl, cudaIpcMemLazyEnablePeerAccess));
  }
  b->nranks = nranks; b->rank = rank;
  b->xchg_on = nranks > 1;
  b->xchg_seq = 0;
  return DMV_OK;
}

// FullSystem::optimizeImmaturePoint for a batch of immature points (ip_trace.cu: ip_activate_kernel)
extern "C" int dmv_ba_activate_points(dmv_ba* b, const dmv_ba_activate_args* a) {
  if (!b || !a) return set_error(DMV_ERR_INVALID, "null argument");
  if (b->nf < 2 || !b->have_state) return set_error(DMV_ERR_STATE, "dmv_ba_set_window + dmv_ba_set_state first");
  if (a->n < 0 || (a->n > 0 && (!a->host || !a->u || !a->v || !a->color8 || !a->weights8 || !a->energyTH || !a->idepth_min || !a->idepth_max || !a->RT ||
                                !a->status || !a->idepth || !a->res_state)))
    return set_error(DMV_ERR_INVALID, "incomplete dmv_ba_activate_args");
  if (a->n == 0) return DMV_OK;
  const int n = a->n, nf = b->nf;
  for (int i = 0; i < n; i++)
    if (a->host[i] < 0 || a->host[i] >= nf) return set_error(DMV_ERR_INVALID, "point %d: host %d out of range", i, a->host[i]);
  CK(cudaSetDevice(b->device));
  if (n > b->act_cap) {
    cudaFree(b->d_act); cudaFreeHost(b->h_act);
    b->act_cap = std::max(n, 2048);
    const size_t words = (size_t)MAXF * MAXF * 14 + (size_t)(24 + MAXF) * b->act_cap;
    CK(cudaMalloc(&b->d_act, sizeof(float) * words));
    CK(cudaMallocHost(&b->h_act, sizeof(float) * words));
  }
  const size_t cap = b->act_cap;
  float* hb = b->h_act;
  float* d = b->d_act;
  // layout (words): RT[64*12] | aff[64*2] | host | u | v | color*8 | weights*8 | energyTH | idmin | idmax | status | idepth | res_state*MAXF
  const size_t o_rt = 0, o_aff = (size_t)MAXF * MAXF * 12, o_host = (size_t)MAXF * MAXF * 14, o_u = o_host + cap, o_v = o_u + cap, o_col = o_v + cap,
               o_wgt = o_col + 8 * cap, o_eth = o_wgt + 8 * cap, o_min = o_eth + cap, o_max = o_min + cap, o_st = o_max + cap, o_id = o_st + cap, o_rs = o_id + cap;
  std::memcpy(hb + o_rt, a->RT, sizeof(float) * 12 * nf * nf);
  const BAIter& it = b->h_up->it;
  for (int k = 0; k < nf * nf; k++) { hb[o_aff + 2 * k] = it.precalc[k][24]; hb[o_aff + 2 * k + 1] = it.precalc[k][25]; }  // PRE_aff_mode
  std::memcpy(hb + o_host, a->host, 4 * (size_t)n); std::memcpy(hb + o_u, a->u, 4 * (size_t)n); std::memcpy(hb + o_v, a->v, 4 * (size_t)n);
  std::memcpy(hb + o_col, a->color8, 32 * (size_t)n); std::memcpy(hb + o_wgt, a->weights8, 32 * (size_t)n); std::memcpy(hb + o_eth, a->energyTH, 4 * (size_t)n);
  std::memcpy(hb + o_min, a->idepth_min, 4 * (size_t)n); std::memcpy(hb + o_max, a->idepth_max, 4 * (size_t)n);
  CK(cudaMemcpyAsync(d, hb, sizeof(float) * o_st, cudaMemcpyHostToDevice, b->stream));
  IPActArgs A;
  A.n = n; A.nf = nf; A.w = b->cfg.w; A.h = b->cfg.h; A.minObs = a->minObs; A.GNIts = 3;  // setting_GNItsOnPointActivation
  A.fxl = it.calib[0]; A.fyl = it.calib[1]; A.cxl = it.calib[2]; A.cyl = it.calib[3]; A.fxli = it.calib[4]; A.fyli = it.calib[5];
  A.huberTH = b->prm.huberTH; A.minIdepthH_act = 100.f;                                      // setting_minIdepthH_act
  for (int f = 0; f < MAXF; f++) A.img[f] = f < nf ? b->d_img[b->slots[f]] : nullptr;
  A.RT = d + o_rt; A.aff = d + o_aff; A.host = reinterpret_cast<const int*>(d + o_host);
  A.u = d + o_u; A.v = d + o_v; A.color = d + o_col; A.weights = d + o_wgt; A.energyTH = d + o_eth; A.idepth_min = d + o_min; A.idepth_max = d + o_max;
  A.status = reinterpret_cast<int*>(d + o_st); A.idepth = d + o_id; A.res_state = reinterpret_cast<int*>(d + o_rs);
  launch_ip_activate(A, b->stream);
  b->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(hb + o_st, d + o_st, sizeof(float) * (2 * cap + (size_t)nf * n), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  std::memcpy(a->status, hb + o_st, 4 * (size_t)n); std::memcpy(a->idepth, hb + o_id, 4 * (size_t)n);
  std::memcpy(a->res_state, hb + o_rs, 4 * (size_t)n * nf);
  return DMV_OK;
}

extern "C" int dmv_ba_io_bytes(dmv_ba* b, long long* h2d, long long* d2h) {
  if (!b || !h2d || !d2h) return set_error(DMV_ERR_INVALID, "null argument");
  *h2d = (long long)sizeof(HostUpload);                        // descriptor + per-iteration tables, carried as kernel parameters
  *d2h = (long long)sizeof(double) * result_doubles(b->N, b->ntiles);     // H_A, b_A, H_sc, b_sc, energy + counters
  return DMV_OK;
}

extern "C" int dmv_ba_set_timing(dmv_ba* b, int enable) {
  if (!b) return set_error(DMV_ERR_INVALID, "null handle");
  b->timing = enable != 0;
  return DMV_OK;
}

