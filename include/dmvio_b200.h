/* dmvio_b200.h — C ABI of the B200-native DM-VIO photometric hot path.
 *
 * Drop-in boundary (SURVEY.md §8b).  Plain C, opaque handles, int status codes, caller-owned host
 * buffers, one CUDA stream per handle, no global mutable state: a BA handle (mapper thread) and a
 * coarse-tracker handle (tracker thread) never share anything.  Every entry point names the reference
 * interface it replaces (paths relative to the reference's src/dso/).
 *
 * Conventions shared with the reference:
 *   - state vector order  [C(4) | frame0: trans3 rot3 a b | frame1 ...],  N = 8*nf + 4
 *     (OptimizationBackend/EnergyFunctional.cpp:L1019-1024)
 *   - pair index of adjoint-like tables:  h + t*nf   (AccumulatedTopHessian.cpp:L71)
 *   - pair index of precalc tables:       h*nf + t   (host->targetPrecalc[target], FullSystem.cpp:L1670-1680)
 *   - x returned by the solve is -step               (EnergyFunctional.cpp:L975)
 *   - residual states: 0 = IN, 1 = OOB, 2 = OUTLIER  (FullSystem/Residuals.h:L43); 255 = "no residual in this slot"
 *
 * All functions return DMV_OK (0) or a negative dmv_status.  dmv_last_error() gives a message for the
 * calling thread.  There is NO CPU fallback: without a CUDA device every create() fails with DMV_ERR_NO_DEVICE.
 */
#ifndef DMVIO_B200_H
#define DMVIO_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMV_MAX_FRAMES 8      /* setting_maxFrames = 7 (+1 while the new keyframe is being optimised), util/settings.cpp:L100 */
#define DMV_PATTERN 8         /* patternNum, util/settings.h:L227 */
#define DMV_PRECALC_FLOATS 32 /* KRKi[9] Kt[3] R0[9] t0[3] aff[2] b0 pad[5] */
#define DMV_MAX_PYR_LEVELS 6  /* PYR_LEVELS, util/settings.h:L52 */

typedef enum dmv_status {
  DMV_OK = 0,
  DMV_ERR_INVALID = -1,   /* bad argument / inconsistent sizes */
  DMV_ERR_NO_DEVICE = -2, /* no usable CUDA device: the product has no CPU path */
  DMV_ERR_CUDA = -3,      /* a CUDA runtime call failed (see dmv_last_error) */
  DMV_ERR_STATE = -4,     /* call order violated (e.g. accumulate before linearize+apply) */
  DMV_ERR_NCCL = -5,
  DMV_ERR_TIMEOUT = -6    /* a grid barrier or the peer exchange inside a kernel gave up waiting (lost rank / CTA) */
} dmv_status;

const char* dmv_last_error(void);
const char* dmv_version(void);
int dmv_device_count(void);

/* ------------------------------------------------------------------------------------------------
 * Bundle-adjustment handle  ==  the GPU side of EnergyFunctional + FullSystem::linearizeAll
 * ------------------------------------------------------------------------------------------------ */
typedef struct dmv_ba dmv_ba;

typedef struct dmv_ba_config {
  int w, h;           /* level-0 image size (wG[0], hG[0]) */
  int max_frames;     /* <= DMV_MAX_FRAMES */
  int max_points;     /* capacity of the active point set */
  int device;         /* CUDA device ordinal */
  int chunk_points;   /* points per thread block: 16 or 32; 0 = chosen per window (16 up to 16 x #SMs points, i.e. one wave; 32 beyond) */
} dmv_ba_config;

/* util/settings.cpp values read by the kernels (constant during a run) */
typedef struct dmv_ba_params {
  float huberTH;                /* setting_huberTH = 9 */
  float outlierTHSumComponent;  /* setting_outlierTHSumComponent = 50*50 */
  float affineOptModeA;         /* <0: JabF[0] is zeroed (Residuals.cpp:L229-242) */
  float affineOptModeB;
} dmv_ba_params;

int dmv_ba_create(const dmv_ba_config* cfg, dmv_ba** out);
int dmv_ba_destroy(dmv_ba* ba);
int dmv_ba_set_params(dmv_ba* ba, const dmv_ba_params* p);
void dmv_ba_default_params(dmv_ba_params* p);

/* FrameHessian::dI (HessianBlocks.h:L122): level-0 [I,dx,dy] AoS, w*h*3 floats, into image slot `slot`
 * (0 <= slot < max_frames).  Slots let frames stay resident across keyframes while window indices shift. */
int dmv_ba_upload_frame(dmv_ba* ba, int slot, const float* dI_aos3);
/* Same, but builds [I,dx,dy] on the device from the raw float image (FrameHessian::makeImages, HessianBlocks.cpp:L128-191, level 0). */
int dmv_ba_upload_image(dmv_ba* ba, int slot, const float* image_wh);
/* Same frame, no second upload: the level-0 [I,dx,dy] plane is copied device-to-device from the coarse-tracker handle in which the frame is
 * resident (dmv_ct_upload_new_image when it arrived; same device).  The reference shares one FrameHessian::dIp between tracker and mapper
 * (HessianBlocks.h:L122-123); here the frame crosses PCIe once and makeImages runs once. */
struct dmv_ct;
int dmv_ba_adopt_frame(dmv_ba* ba, int slot, struct dmv_ct* ct);

/* EnergyFunctional::makeIDX (EnergyFunctional.cpp:L998-1016): window frame index -> image slot */
int dmv_ba_set_window(dmv_ba* ba, int nf, const int* slots);

/* EFPoint/PointHessian fields read on the path (HessianBlocks.h:L413-508, EnergyFunctionalStructs.h:L104-137).
 * Points must be ordered by host frame index (that is EnergyFunctional::allPoints' order).
 * color8/weights8: npts*8.  priorF/deltaF may be NULL (zeros). */
int dmv_ba_set_points(dmv_ba* ba, int npts, const int32_t* host, const float* u, const float* v, const float* idepth,
                      const float* idepth_zero, const float* color8, const float* weights8, const float* priorF);

/* The active (non-linearised) PointFrameResiduals of the window: (point, target) pairs, at most one per pair,
 * with PointFrameResidual::state_state / state_energy (Residuals.h:L64-84).  state_state/state_energy may be NULL (all IN / 0). */
int dmv_ba_set_residuals(dmv_ba* ba, int nres, const int32_t* point, const int32_t* target, const int32_t* state_state,
                         const float* state_energy);

/* EnergyFunctional::setAdjointsF (EnergyFunctional.cpp:L48-108): adHost/adTarget, nf*nf 8x8 row-major doubles, index h + t*nf */
int dmv_ba_set_adjoints(dmv_ba* ba, const double* adHost, const double* adTarget);

/* Per-iteration state == FullSystem::setPrecalcValues (FrameFramePrecalc::set, HessianBlocks.cpp:L193-223) + CalibHessian values +
 * FrameHessian::frameEnergyTH.  idepth (npts) may be NULL: keep the device copy (e.g. after dmv_ba_resubstitute(apply=1)).
 * idepth_zero likewise.  deltaF (npts) = idepth - idepth_zero for the prior shift (EnergyFunctional.cpp:L194); NULL => recomputed on device. */
typedef struct dmv_ba_state {
  float calib[8];          /* fxl fyl cxl cyl fxli fyli cxli cyli (CalibHessian::value_scaledf / value_scaledi) */
  const float* precalc;    /* nf*nf*DMV_PRECALC_FLOATS, index h*nf + t */
  const float* frameEnergyTH; /* nf */
  const float* idepth;     /* npts or NULL */
  const float* idepth_zero;/* npts or NULL */
} dmv_ba_state;
int dmv_ba_set_state(dmv_ba* ba, const dmv_ba_state* st);

/* FullSystem::linearizeAll(false) (FullSystemOptimize.cpp:L150-218) fused with the *tentative* accumulateAF/SCF of the
 * next solveSystemF: evaluates every active residual at the current state, reduces the per-pair 13x13 blocks, the
 * per-point Hdd/bd/Hcd and the Schur complement, and assembles the dense system on the device (one launch).
 * Nothing becomes visible to dmv_ba_accumulate / dmv_ba_resubstitute until dmv_ba_apply_res().
 * out: energy = sum of PointFrameResidual::linearize() return values (stats[0]); n_in = #residuals with state_NewState==IN. */
typedef struct dmv_ba_lin_result {
  double energy;
  int n_in, n_oob, n_outlier;
} dmv_ba_lin_result;
int dmv_ba_linearize(dmv_ba* ba, dmv_ba_lin_result* out);

/* Per-residual outputs of the last linearize, in the order given to dmv_ba_set_residuals
 * (state_NewState, state_NewEnergy, state_NewEnergyWithOutlier, centerProjectedTo; Residuals.h:L64-84). Any pointer may be NULL. */
int dmv_ba_get_residual_outputs(dmv_ba* ba, int32_t* newState, float* newEnergy, float* newEnergyWithOutlier, float* centerProjectedTo3,
                                float* JpJdF8);

/* state_NewEnergyWithOutlier of the residuals whose target is frame `target` (input of FullSystem::setNewFrameEnergyTH,
 * FullSystemOptimize.cpp:L96-149): writes at most cap floats, returns the count in *n. Entries < 0 (not evaluated) are skipped. */
int dmv_ba_get_target_energies(dmv_ba* ba, int target, float* out, int cap, int* n);

/* PointFrameResidual::applyRes(true) + EFResidual::takeDataF for all active residuals (FullSystemOptimize.cpp:L90-94):
 * commits the tentative linearisation (buffer swap; no kernel). */
int dmv_ba_apply_res(dmv_ba* ba);

/* The accumulate half of EnergyFunctional::solveSystemF (EnergyFunctional.cpp:L853-860): accumulateAF_MT + accumulateSCF_MT of the
 * committed linearisation.  H_A/H_sc: N*N row-major doubles, b_A/b_sc: N.  (accumulateLF_MT's priors are host data; the host adapter adds them.)
 * resInA = AccumulatedTopHessianSSE::nres[0]. */
int dmv_ba_accumulate(dmv_ba* ba, double* H_A, double* b_A, double* H_sc, double* b_sc, int* resInA);

/* Per-point results of the committed accumulation: EFPoint::{Hdd_accAF, bd_accAF, Hcd_accAF, HdiF, bdSumF} (EnergyFunctionalStructs.h:L117-135).
 * Any pointer may be NULL. */
int dmv_ba_get_point_outputs(dmv_ba* ba, float* Hdd_accAF, float* bd_accAF, float* Hcd_accAF4, float* HdiF, float* bdSumF);
/* EFPoint::HdiF as AccumulatedSCHessian::addPoint left it during the last solveSystemF (AccumulatedSCHessian.cpp:L42-50; idepth_hessian =
 * 1 / HdiF): the values of the linearisation the last dmv_ba_accumulate() returned, kept on the device while later linearisations
 * (rejected steps, the tail's linearizeAll(true)) overwrite the per-point outputs.  FullSystem::flagPointsForRemoval reads it (FullSystem.cpp:L840-850). */
int dmv_ba_get_solve_HdiF(dmv_ba* ba, float* HdiF);

/* EnergyFunctional::resubstituteF_MT (EnergyFunctional.cpp:L267-321): x = N doubles (= -step).  step_out (npts) may be NULL.
 * apply != 0 additionally performs the point part of FullSystem::doStepFromBackup (FullSystemOptimize.cpp:L264-272):
 * idepth = idepth_backup + step, idepth_zero likewise (DM-VIO), on the device copy; sums[0] = sum step^2, sums[1] = sum |idepth_backup|, sums[2] = npts. */
int dmv_ba_resubstitute(dmv_ba* ba, const double* x, float* step_out, int apply, double sums[3]);
/* FullSystem::backupState / loadSateBackup for the point depths held on the device (FullSystemOptimize.cpp:L322-388) */
int dmv_ba_backup_points(dmv_ba* ba);
int dmv_ba_restore_points(dmv_ba* ba);
int dmv_ba_get_idepth(dmv_ba* ba, float* idepth, float* idepth_zero);

/* Fused GN iteration (one host<->device round trip): resubstitute(x) + point step + set_state + linearize.
 * x may be NULL (first linearisation).  Equivalent to dmv_ba_resubstitute(x, apply=1) ; dmv_ba_set_state(st) ; dmv_ba_linearize(). */
int dmv_ba_gn_step(dmv_ba* ba, const double* x, const dmv_ba_state* st, dmv_ba_lin_result* out, double sums[3]);

/* Point activation: FullSystem::optimizeImmaturePoint (FullSystem/FullSystemOptPoint.cpp:L51-205) with ImmaturePoint::linearizeResidual
 * (FullSystem/ImmaturePoint.cpp:L498-565) for n immature points against every other keyframe of the window, as
 * FullSystem::activatePointsMT_Reductor does (FullSystem.cpp:L586-602).  Uses the frames, calibration and PRE_aff_mode of the last
 * dmv_ba_set_state / dmv_ba_gn_step.  RT: nf*nf*12 floats, index h*nf+t: PRE_RTll (row-major) | PRE_tTll of FrameFramePrecalc (current state).
 * out: status 1 = activate (the caller creates the PointHessian with idepth and one residual per res_state == 0), 0 = not well
 * constrained (keep as immature point), -1 = outlier (delete); idepth = optimised inverse depth; res_state[i*nf+f]: 0 IN, 1 OOB, 2 OUTLIER,
 * 255 = no residual.  Bit-identical to the CPU code (see dmv_ct_trace_points). */
typedef struct dmv_ba_activate_args {
  int n;
  const int32_t* host;
  const float *u, *v, *color8, *weights8, *energyTH, *idepth_min, *idepth_max;
  const float* RT;
  int minObs;               /* 1 in activatePointsMT_Reductor */
  int32_t* status;
  float* idepth;
  int32_t* res_state;
} dmv_ba_activate_args;
int dmv_ba_activate_points(dmv_ba* ba, const dmv_ba_activate_args* a);

/* PointFrameResidual::resetOOB for every residual of the window, as FullSystem::optimize does when it collects activeResiduals
 * (FullSystem/FullSystemOptimize.cpp:L431-448; FullSystem/Residuals.h:L91-98): state IN, energy 0.  Discards the tentative and the committed
 * linearisation (the next dmv_ba_linearize / dmv_ba_gn_step starts from these states). */
int dmv_ba_reset_oob(dmv_ba* ba);

/* Residuals leave the window: the deletion loop of FullSystem::linearizeAll(fixLinearization = true) (FullSystem/FullSystemOptimize.cpp:L196-214 ->
 * EnergyFunctional::dropResidual, OptimizationBackend/EnergyFunctional.cpp:L500-520) for residuals that did not end up IN.  res_idx: indices in
 * the current dmv_ba_set_residuals order; the remaining residuals keep their relative order (per-residual outputs shrink accordingly).  The
 * committed linearisation stays valid (a non-active residual contributes nothing to it). */
int dmv_ba_drop_residuals(dmv_ba* ba, int n, const int32_t* res_idx);

/* Point marginalisation at keyframe creation, one launch pair for the whole flagged set:
 *   - the compute of FullSystem::flagPointsForRemoval for each flagged point (FullSystem/FullSystem.cpp:L826-838): PointFrameResidual::resetOOB,
 *     linearize, applyRes(true), EFResidual::fixLinearizationF (OptimizationBackend/EnergyFunctionalStructs.cpp:L88-114) -> res_toZeroF;
 *   - EnergyFunctional::marginalizePointsF (OptimizationBackend/EnergyFunctional.cpp:L678-742): priorF *= idepthFixPriorMargFac,
 *     AccumulatedTopHessian::addPoint<2>, AccumulatedSCHessian::addPoint(p, shiftPriorToZero = false), stitch without priors.
 * The caller decides WHICH points (PointHessian::isOOB / isInlierNew / idepth_hessian > setting_minIdepthH_marg are host bookkeeping) and finishes
 * with HM += setting_margWeightFac * (M - Msc), bM += setting_margWeightFac * (Mb - Mbsc), then re-uploads the window without the points.
 * Uses the frames / calibration / depths of the last dmv_ba_set_state or dmv_ba_gn_step.  adHTdeltaF: nf*nf*8 floats, entry [h + t*nf]
 * (EnergyFunctional::setDeltaF, EnergyFunctional.cpp:L175-198); cDeltaF: calibration value - value_zero.  Any output may be NULL.
 * M/Msc: N*N row-major, N = 8 nf + 4.  res_toZeroF [nres*8] / isLinearized [nres] follow the dmv_ba_set_residuals order (zero for residuals
 * that were not linearised); ngoodRes [n] follows `point`.  Invalidates the tentative linearisation; the committed one is untouched.
 * Sharded handles (dmv_ba_comm_init / dmv_ba_p2p_import): not supported, returns DMV_ERR_STATE (marginalise per rank and sum on the host). */
typedef struct dmv_ba_marg_args {
  int32_t n;
  const int32_t* point;          /* [n] indices in dmv_ba_set_points order */
  const float* adHTdeltaF;
  float cDeltaF[4];
  float idepthFixPriorMargFac;   /* 600*600 (util/settings.cpp:L68) */
  double *M, *Mb, *Msc, *Mbsc;
  int32_t* resInM;
  int32_t* ngoodRes;
  float* res_toZeroF;
  uint8_t* isLinearized;
} dmv_ba_marg_args;
int dmv_ba_marginalize_points(dmv_ba* ba, const dmv_ba_marg_args* a);

/* Multi-GPU (SURVEY.md §8e): points are sharded over ranks, images/tables replicated.  After dmv_ba_comm_init every
 * dmv_ba_linearize / dmv_ba_gn_step / dmv_ba_marginalize_points all-reduces the system (and energy / counters) over NCCL so that all ranks
 * hold identical H,b; every rank must make the same sequence of these calls (dmv_ba_marginalize_points with its own flagged points, possibly none).
 * nccl_unique_id: 128 bytes from ncclGetUniqueId() on rank 0, distributed by the caller. */
int dmv_nccl_unique_id(void* id128);
int dmv_ba_comm_init(dmv_ba* ba, int nranks, int rank, const void* nccl_unique_id);

/* The same exchange without NCCL, over NVLink/NVSwitch peer memory (CUDA IPC, one process per GPU of one node, <= 8 ranks):
 * every rank exports its inbox (64-byte cudaIpcMemHandle_t), the caller all-gathers the handles (any transport: MPI,
 * torch.distributed, a file) and every rank imports all of them.  From then on the all-reduce happens INSIDE THE LINEARISATION KERNEL:
 * the lanes that produce a result entry push it to every peer as a 16-byte flag-carrying packet, later wait (bounded: DMV_ERR_TIMEOUT) for the
 * peers' packets of the same entry and add them in rank order (bit-identical H,b on all ranks; no extra launch, no fence round trip).
 * Takes precedence over a NCCL communicator if both are set; nranks = 1 in dmv_ba_p2p_import switches it off again.
 * No reference counterpart (the reference is single-node CPU). */
int dmv_ba_p2p_export(dmv_ba* ba, void* ipc_handle64);
int dmv_ba_p2p_import(dmv_ba* ba, int nranks, int rank, const void* ipc_handles /* nranks*64 bytes, rank order */);

/* ---- batched windows (SURVEY.md section 8d "batched variant"): B independent windows, each an ordinary BA handle on the same device with
 * the same chunk_points, linearised by ONE launch.  No reference counterpart (FullSystem::optimize handles one window); per window the
 * results are bit-identical to dmv_ba_gn_step on that handle. */
typedef struct dmv_ba_batch dmv_ba_batch;
int dmv_ba_batch_create(dmv_ba* const* handles, int n, dmv_ba_batch** out);   /* n <= 64; the handles stay owned by the caller */
int dmv_ba_batch_destroy(dmv_ba_batch* batch);
/* dmv_ba_gn_step on every handle: x[i] may be NULL (x itself may be NULL), st[i] as for dmv_ba_gn_step; out (n entries) and sums3 (3 n doubles)
 * may be NULL.  Afterwards: dmv_ba_apply_res / dmv_ba_accumulate / ... per handle as usual. */
int dmv_ba_batch_gn_step(dmv_ba_batch* batch, const double* const* x, const dmv_ba_state* const* st, dmv_ba_lin_result* out, double* sums3);
int dmv_ba_batch_set_timing(dmv_ba_batch* batch, int enable);
int dmv_ba_batch_last_kernel_ms(dmv_ba_batch* batch, float* ms);   /* CUDA-event time of the last batched launch (after set_timing(1)) */

/* instrumentation (cheap, always present): CUDA-event timing of the last linearize / gn_step on the handle's stream, milliseconds:
 * [0] = total device time of the call, [1] = ba_fused_kernel, [2] = 0, [3] = what follows the kernel (NCCL all-reduce / D2H copy) */
int dmv_ba_last_timing(dmv_ba* ba, float ms[4]);
int dmv_ba_kernel_launch_count(dmv_ba* ba, long long* n);
/* enable/disable the CUDA-event timing of dmv_ba_linearize / dmv_ba_gn_step (off by default) */
int dmv_ba_set_timing(dmv_ba* ba, int enable);
/* bytes copied host->device and device->host by one dmv_ba_gn_step / dmv_ba_linearize call */
int dmv_ba_io_bytes(dmv_ba* ba, long long* h2d, long long* d2h);
/* The measurement-only entry points (dmv_ba_bench_device, dmv_ba_bench_e2e, ...) live in dmvio_b200_bench.h / csrc/ba_bench.cu and
 * are compiled in only with BENCH=1. */

/* ------------------------------------------------------------------------------------------------
 * Coarse-tracker handle  ==  the GPU side of CoarseTracker (FullSystem/CoarseTracker.{h,cpp})
 * ------------------------------------------------------------------------------------------------ */
typedef struct dmv_ct dmv_ct;
typedef struct dmv_ct_config {
  int w, h;
  int levels;      /* pyrLevelsUsed */
  int max_points;  /* capacity of pc_* per level */
  int device;
} dmv_ct_config;

int dmv_ct_create(const dmv_ct_config* cfg, dmv_ct** out);
int dmv_ct_destroy(dmv_ct* ct);
/* CoarseTracker::makeK (CoarseTracker.cpp:L105-134): per-level intrinsics */
int dmv_ct_set_K(dmv_ct* ct, int level, float fx, float fy, float cx, float cy);
/* pc_u/pc_v/pc_idepth/pc_color of one level (result of makeCoarseDepthL0, CoarseTracker.cpp:L249-293) */
int dmv_ct_set_ref(dmv_ct* ct, int level, int n, const float* pc_u, const float* pc_v, const float* pc_idepth, const float* pc_color);
/* CoarseTracker::setCoarseTrackingRef -> makeCoarseDepthL0 (CoarseTracker.cpp:L138-295, L524-538) on the device: builds pc_* of EVERY level from the
 * keyframe's IN residuals that target it: per residual centerProjectedTo = (Ku, Kv, new_idepth) and its point's HdiF (CoarseTracker.cpp:L148-158).
 * The reference frame (lastRef->dIp) is the frame currently resident in the handle (upload it first with dmv_ct_upload_new_image /
 * dmv_ct_upload_new of every level); afterwards a new frame may be uploaded for tracking.  pc_n_out (levels entries, may be NULL) = pc_n[].
 * Bit-identical lists (values and order) to the CPU code. */
int dmv_ct_make_coarse_depth(dmv_ct* ct, int n, const float* Ku, const float* Kv, const float* new_idepth, const float* HdiF, int32_t* pc_n_out);
/* download pc_u / pc_v / pc_idepth / pc_color of one level (any pointer may be NULL; *n = pc_n[level]) */
int dmv_ct_get_ref(dmv_ct* ct, int level, int* n, float* pc_u, float* pc_v, float* pc_idepth, float* pc_color);
/* newFrame->dIp[level] (w_l*h_l*3 floats AoS) */
int dmv_ct_upload_new(dmv_ct* ct, int level, const float* dIp_aos3);
/* builds the whole pyramid of the new frame on the device from the raw image (FrameHessian::makeImages) */
int dmv_ct_upload_new_image(dmv_ct* ct, const float* image_wh);
/* settings read by calcRes: setting_huberTH */
int dmv_ct_set_huber(dmv_ct* ct, float huberTH);

/* CoarseTracker::calcRes (L361-517) fused with calcGSSSE (L299-356) for one pose:
 *   RKi = R * Ki[lvl] (row-major 3x3 float), t (3), affLL = AffLight::fromToVecExposure(...) (2),
 *   a_gs = affLL[0] (first argument `a` of calcGSSSE), b0 = lastRef_aff_g2l.b, cutoffTH.
 * out: res6 = Vec6 of calcRes; if want_gs: H (8x8 row-major) and b (8) exactly as calcGSSSE returns them
 * (divided by the 4-padded warped count, SCALE_* applied); n_warped = buf_warped_n (padded). */
int dmv_ct_calc_res_gs(dmv_ct* ct, int level, const float RKi[9], const float t[3], const float affLL[2], float b0, float cutoffTH,
                       int want_gs, double res6[6], double H[64], double b[8], int* n_warped);
/* CoarseTracker::trackNewestCoarse (CoarseTracker.cpp:L539-770, visual-only branch L639-683) as ONE persistent launch: the whole
 * Levenberg-Marquardt loop over the pyramid levels (calcRes + calcGSSSE per evaluation, 8x8 LDLT, SE3 update, accept/reject, cutoff
 * doubling, level repeat) runs on the device; the host gets the tracked pose back.  Same semantics as driving dmv_ct_calc_res_gs from the
 * host loop: R,t = lastToNew_out (refToNew, row-major), a,b = aff_g2l_out; on an aborted track (NaN residual or > 1.5*minResForAbort)
 * trackingGood = 0, status = 2 and R,t,a,b are returned unchanged, like the reference's early `return false`.
 * Runs on one thread-block cluster and takes any reference-point count up to max_points per level. */
typedef struct dmv_ct_track_args {
  double R[9], t[3];          /* in: initial refToNew */
  double a, b;                /* in: initial aff_g2l of the new frame */
  double ref_a, ref_b;        /* lastRef_aff_g2l */
  float ref_exposure, new_exposure; /* lastRef->ab_exposure, newFrame->ab_exposure */
  float coarseCutoffTH;       /* setting_coarseCutoffTH = 20 */
  float affineOptModeA, affineOptModeB;
  int coarsestLvl;
  double minResForAbort[5];   /* NaN = never abort */
} dmv_ct_track_args;
typedef struct dmv_ct_track_result {
  double R[9], t[3], a, b;
  double lastResiduals[5];    /* CoarseTracker::lastResiduals */
  double flowIndicators[3];   /* CoarseTracker::lastFlowIndicators */
  int trackingGood, iterations, evaluations, status;
} dmv_ct_track_result;
int dmv_ct_track(dmv_ct* ct, const dmv_ct_track_args* in, dmv_ct_track_result* out);

/* ------------------------------------------------------------------------------------------------
 * Immature-point tracing  ==  ImmaturePoint::traceOn (FullSystem/ImmaturePoint.cpp:L77-437) for all immature points of ONE host
 * frame against the newest frame, i.e. one iteration of the host loop of FullSystem::traceNewCoarse (FullSystem.cpp:L554-575).
 * Runs on the coarse-tracker handle: the frame traced against is the one last given to dmv_ct_upload_new_image / dmv_ct_upload_new
 * (level 0), which is resident there anyway.  Results are BIT-IDENTICAL to the reference's CPU code (the kernel is compiled without
 * FMA contraction and keeps the reference's operation order).
 * ------------------------------------------------------------------------------------------------ */
typedef struct dmv_ip_settings {   /* util/settings.cpp:L79, L178-187 */
  float maxPixSearch;              /* setting_maxPixSearch = 0.027 */
  float trace_stepsize;            /* 1.0 */
  float trace_GNThreshold;         /* 0.1 */
  float trace_extraSlackOnTH;      /* 1.2 */
  float trace_slackInterval;       /* 1.5 */
  float trace_minImprovementFactor;/* 2 */
  float huberTH;                   /* setting_huberTH = 9 */
  int trace_GNIterations;          /* 3 */
  int minTraceTestRadius;          /* 2 */
} dmv_ip_settings;
void dmv_ip_default_settings(dmv_ip_settings* s);
/* ImmaturePoint fields (ImmaturePoint.h:L56-90), structure of arrays over the n points of one host frame.
 * in: u, v, color[8], weights[8], gradH (Mat22f row-major), energyTH.   in/out: idepth_min, idepth_max, quality,
 * lastTraceStatus (ImmaturePointStatus: 0 GOOD, 1 OOB, 2 OUTLIER, 3 SKIPPED, 4 BADCONDITION, 5 UNINITIALIZED), lastTraceUV, lastTracePixelInterval. */
typedef struct dmv_ip_points {
  int n;
  const float *u, *v, *color8, *weights8, *gradH4, *energyTH;
  float *idepth_min, *idepth_max, *quality;
  int32_t* lastTraceStatus;
  float *lastTraceUV2, *lastTracePixelInterval;
} dmv_ip_points;
/* ImmaturePoint::ImmaturePoint (ImmaturePoint.cpp:L34-63) for n integer pixels (u, v) of the frame resident in the handle (the frame that
 * just became a keyframe, FullSystem::makeNewTraces, FullSystem.cpp:L1640-1665): pattern colours, weights (setting_outlierTHSumComponent = 50*50),
 * gradH (row-major 2x2), energyTH (= 8 * setting_outlierTH * setting_overallEnergyTHWeight^2 = 1152); ok[i] = 0 where a colour is not finite
 * (energyTH = NaN, the caller drops the point like the reference).  Bit-identical to the CPU code. */
int dmv_ct_init_points(dmv_ct* ct, int n, const int32_t* u, const int32_t* v, float* color8, float* weights8, float* gradH4, float* energyTH, int32_t* ok);
/* hostToFrame_KRKi (row-major 3x3), hostToFrame_Kt, hostToFrame_affine exactly as traceNewCoarse computes them (FullSystem.cpp:L557-561).
 * settings may be NULL (defaults). */
int dmv_ct_trace_points(dmv_ct* ct, const dmv_ip_points* pts, const float KRKi[9], const float Kt[3], const float aff[2], const dmv_ip_settings* settings);
/* The same for the immature points of SEVERAL host keyframes at once (the whole loop of FullSystem::traceNewCoarse, FullSystem.cpp:L554-575):
 * sets[k] = the points hosted by keyframe k, tables14 = per host [KRKi 9 | Kt 3 | aff 2]; one upload, one launch, one download. */
int dmv_ct_trace_points_multi(dmv_ct* ct, int nsets, const dmv_ip_points* sets, const float* tables14, const dmv_ip_settings* settings);

/* ------------------------------------------------------------------------------------------------
 * Pixel selection for new keyframes  ==  PixelSelector::makeMaps (FullSystem/PixelSelector2.cpp:L94-454) and FullSystem::makeNewTraces
 * (FullSystem.cpp:L1640-1665) on the frame resident in the coarse-tracker handle: the frame last given to dmv_ct_upload_new_image, or to
 * dmv_ct_upload_new for levels 0, 1 and 2 (the same contract as dmv_ct_init_points).  absSquaredGrad of levels 0..2 is computed from the
 * resident {I, dx, dy} planes.  Results are BIT-IDENTICAL to the reference's CPU code and identical from call to call.
 * The selector's state (PixelSelector::currentPotential) travels through the call: the caller owns it, as FullSystem owns pixelSelector.
 * DMV_ERR_INVALID: w or h not divisible by 16, fewer than 3 levels, density <= 0, currentPotential < 1; DMV_ERR_STATE: no frame resident.
 * ------------------------------------------------------------------------------------------------ */
typedef struct dmv_ps_settings {       /* util/settings.cpp:L167-170 */
  float minGradHistCut;                /* 0.5 */
  float minGradHistAdd;                /* 7 */
  float gradDownweightPerLevel;        /* 0.75 */
  int selectDirectionDistribution;     /* 1 */
} dmv_ps_settings;
void dmv_ps_default_settings(dmv_ps_settings* s);
typedef struct dmv_ps_args {
  float density;          /* numWant: setting_desiredImmatureDensity (makeNewTraces) or densities[0]*w*h (CoarseInitializer::setFirst) */
  int recursionsLeft;     /* 1 */
  float thFactor;         /* 1 (makeNewTraces), 2 (setFirst) */
  int currentPotential;   /* PixelSelector::currentPotential before the call (3 for a new selector) */
  const float* B256;      /* CalibHessian::B for the gamma weighting of absSquaredGrad; NULL = HCalib == 0 / setting_gammaWeightsPixelSelect == 0 */
  const dmv_ps_settings* settings;     /* NULL = defaults */
} dmv_ps_args;
typedef struct dmv_ps_result { int numHaveSub; int currentPotential; } dmv_ps_result;  /* makeMaps' return value; the potential after the call */
/* PixelSelector::makeMaps(fh, map_out, density, recursionsLeft, false, thFactor).  map_out: w*h floats of 0/1/2/4 (may be NULL). */
int dmv_ct_select_pixels(dmv_ct* ct, const dmv_ps_args* a, float* map_out, dmv_ps_result* r);
/* FullSystem::makeNewTraces: makeMaps, then an ImmaturePoint (as dmv_ct_init_points) for every selected pixel with x, y in
 * [patternPadding+1, dim-patternPadding-2), in raster order; points whose energyTH is not finite are dropped, as the reference does.
 * Out: *n points of u, v, type (the map value), color8, weights8, gradH4 (row-major 2x2), energyTH.  If more than cap points are kept, only
 * *n (the count needed) is written and DMV_ERR_INVALID is returned. */
int dmv_ct_make_new_traces(dmv_ct* ct, const dmv_ps_args* a, int cap, int* n, int32_t* u, int32_t* v, float* type,
                           float* color8, float* weights8, float* gradH4, float* energyTH, dmv_ps_result* r);

/* enable/disable the CUDA-event timing of dmv_ct_calc_res_gs (off by default); dmv_ct_last_timing()[0] = kernel milliseconds */
int dmv_ct_set_timing(dmv_ct* ct, int enable);
int dmv_ct_last_timing(dmv_ct* ct, float ms[4]);
int dmv_ct_kernel_launch_count(dmv_ct* ct, long long* n);
int dmv_ct_last_point_evaluations(dmv_ct* ct, double* n);   /* sum over the last dmv_ct_track's evaluations of the level's reference-point count */

/* ------------------------------------------------------------------------------------------------
 * Coarse-initialiser handle  ==  the GPU side of CoarseInitializer::calcResAndGS (FullSystem/CoarseInitializer.{h,cpp})
 * The rest of CoarseInitializer::trackFrame (doStep, applyStep, optReg, propagateUp/Down, the 8x8 solve; L85-281, L650-965) is scalar
 * per-point host code that runs once per sequence and stays with the caller: it owns the Pnt arrays and passes their live fields per call.
 * ------------------------------------------------------------------------------------------------ */
typedef struct dmv_ci dmv_ci;
typedef struct dmv_ci_config {
  int w, h;
  int levels;      /* pyrLevelsUsed */
  int max_points;  /* capacity of points[lvl] (numPoints[0] is the largest) */
  int device;
} dmv_ci_config;
int dmv_ci_create(const dmv_ci_config* cfg, dmv_ci** out);
int dmv_ci_destroy(dmv_ci* ci);
/* CoarseInitializer::makeK (CoarseInitializer.cpp:L967-999) */
int dmv_ci_set_K(dmv_ci* ci, int level, float fx, float fy, float cx, float cy);
/* firstFrame->dIp[level] / newFrame->dIp[level] (w_l*h_l*3 floats AoS) */
int dmv_ci_upload_first(dmv_ci* ci, int level, const float* dIp_aos3);
int dmv_ci_upload_new(dmv_ci* ci, int level, const float* dIp_aos3);
/* the constant fields of points[level] (Pnt::u, v, outlierTH; CoarseInitializer.h:L44-82), set by setFirst (L804-889) */
int dmv_ci_set_points(dmv_ci* ci, int level, int n, const float* u, const float* v, const float* outlierTH);

typedef struct dmv_ci_eval_args {
  int level;
  float RKi[9];          /* (refToNew.rotationMatrix() * Ki[lvl]).cast<float>(), row-major (L341) */
  double t_d[3];         /* refToNew.translation() */
  double t_log[3];       /* refToNew.log().head<3>() (L601) */
  float r2new_aff[2];    /* exp(refToNew_aff.a), refToNew_aff.b (L343) */
  float huberTH;         /* setting_huberTH */
  float alphaK, alphaW, couplingWeight;             /* CoarseInitializer members (CoarseInitializer.h:L107-111) */
  double weightZeroPriorX, weightZeroPriorY;        /* setting_weightZeroPriorDSOInitX / Y (L606-611) */
  /* live per-point fields of points[level], n entries (n as given to dmv_ci_set_points) */
  const float* idepth_new;
  const uint8_t* isGood;
  const float* energy2;   /* Pnt::energy, 2 per point */
  const float* iR;
  /* per-point results (any may be NULL): Pnt::isGood_new, energy_new (2 per point), maxstep, lastHessian_new and the JbBuffer_new rows
   * (10 per point) as L562-586 leave them.  maxstep / lastHessian_new / JbBuffer_new are meaningful for isGood_new points only. */
  uint8_t* isGood_new;
  float* energy_new2;
  float* maxstep;
  float* lastHessian_new;
  float* JbBuffer_new10;
} dmv_ci_eval_args;
typedef struct dmv_ci_eval_result {
  float H[64], b[8], Hsc[64], bsc[8];   /* H_out, b_out, H_out_sc, b_out_sc (row-major) */
  float res3[3];                        /* Vec3f(E.A, alphaEnergy, E.num) */
  float alphaOpt;
  int n_good_new;
} dmv_ci_eval_result;
/* CoarseInitializer::calcResAndGS (CoarseInitializer.cpp:L333-625) as ONE launch */
int dmv_ci_calc_res_and_gs(dmv_ci* ci, const dmv_ci_eval_args* args, dmv_ci_eval_result* out);
int dmv_ci_kernel_launch_count(dmv_ci* ci, long long* n);

#ifdef __cplusplus
}
#endif
#endif /* DMVIO_B200_H */
