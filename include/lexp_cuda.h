/* lexp_cuda.h -- C-ABI of the B200-native unary-cost engine for Local Expansion Stereo.
 *
 * This is the drop-in boundary for ONE path of t-taniai/LocalExpStereo: the per-cell
 * slanted-plane unary cost evaluation + guided-filter aggregation.  Every entry point
 * names the reference interface it replaces (paths relative to
 * /root/reference/LocalExpansionStereo/).  Plain C types only; no torch / OpenCV types.
 * All functions return 0 on success and a negative lexp_status on failure;
 * lexp_last_error() returns a thread-local message.  There is NO CPU fallback: every
 * evaluation runs hand-written sm_100a kernels, or fails.
 *
 * Threading: a context may be used from several host threads (the reference calls the
 * virtuals from OpenMP threads, FastGCStereo.h:30-49).  Device work is serialised internally;
 * concurrent lexp_eval_cell calls are combined into batched launches (lexp_combine_stats).
 */
#ifndef LEXP_CUDA_H_
#define LEXP_CUDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define LEXP_API __declspec(dllexport)
#else
#define LEXP_API __attribute__((visibility("default")))
#endif

typedef enum lexp_status {
    LEXP_OK = 0,
    LEXP_ERR_INVALID = -1, /* bad argument / precondition violated        */
    LEXP_ERR_CUDA = -2,    /* CUDA runtime error (message in last_error)   */
    LEXP_ERR_STATE = -3,   /* images / volume not uploaded yet             */
    LEXP_ERR_NOMEM = -4
} lexp_status;

/* cv::Rect layout (x, y, width, height), image coordinates. */
typedef struct lexp_rect { int x, y, width, height; } lexp_rect;

/* struct Plane {a,b,c,v}  (Plane.h:4-8); d(x,y) = a*x + b*y + c (Plane.h:51-58). */
typedef struct lexp_plane { float a, b, c, v; } lexp_plane;

/* Subset of `struct Parameters` (StereoEnergy.h:13-40) + the CostVolumeEnergy constructor
 * arguments (CostVolumeEnergy.h:16) that the unary path uses. */
typedef struct lexp_params {
    int height, width;  /* image size (imL.rows, imL.cols)                                    */
    int ndisp;          /* D = vol.size[0]; volume is float[D][H][W] (main.cpp:353-354)        */
    int windR;          /* Parameters::windR; guided-filter box radius R = windR/2 (CostVolumeEnergy.h:30) */
    float eps;          /* Parameters::filter_param1 (GF regulariser, main.cpp:73: 1e-4)       */
    float th_col;       /* Parameters::th_col (truncation, CostVolumeEnergy.h:96)              */
    float min_disp;     /* MIN_DISPARITY (0 in main.cpp)                                       */
    float max_disp;     /* MAX_DISPARITY (= ndisp-1 in main.cpp:385-386)                       */
    int device;         /* CUDA device ordinal                                                  */
    int energy_kind;    /* 0: CostVolumeEnergy (CostVolumeEnergy.h:6-184); 1: NaiveStereoEnergy (StereoEnergy.h:629-764), no volume */
    float alpha;        /* Parameters::alpha   (NaiveStereoEnergy only, StereoEnergy.h:659-664)   */
    float th_grad;      /* Parameters::th_grad (NaiveStereoEnergy only)                            */
    int reserved[4];
} lexp_params;

typedef struct lexp_ctx lexp_ctx;   /* replaces a CostVolumeEnergy instance (CostVolumeEnergy.h:6-184) */
typedef struct lexp_plan lexp_plan; /* device-side work list for a fixed set of (filterRect, targetRect) */

LEXP_API const char* lexp_last_error(void);
LEXP_API int lexp_version(void);

/* CostVolumeEnergy::CostVolumeEnergy(imL, imR, volL, volR, params, MAX, MIN) -- CostVolumeEnergy.h:16-43.
 * Split in three so that volumes may already live on the device. */
LEXP_API int lexp_create(const lexp_params* params, lexp_ctx** out_ctx);
LEXP_API int lexp_destroy(lexp_ctx* ctx);

/* Guide image of view `mode` (0 = left, 1 = right): uint8 BGR, `step_bytes` per row (cv::Mat::step).
 * Runs the one-time guided-filter statistics on the device
 * (FastGuidedImageFilter<double>(im, windR/2, eps, 1/255): CostVolumeEnergy.h:30-31, GuidedFilter.h:58-102). */
LEXP_API int lexp_set_image(lexp_ctx* ctx, int mode, const uint8_t* bgr_host, ptrdiff_t step_bytes);

/* vol[mode] = float[D][H][W] contiguous (CostVolumeEnergy.h:20-21).  Both calls re-lay the volume out
 * into a context-owned blocked copy in HBM (4-pixel blocks, disparity contiguous) and scan it for
 * NaN/Inf; the caller's buffer (host, or device for _device) is not referenced after the call returns. */
LEXP_API int lexp_set_volume_host(lexp_ctx* ctx, int mode, const float* vol_host);
LEXP_API int lexp_set_volume_device(lexp_ctx* ctx, int mode, const float* vol_device);

/* The same with the reference's volume preparation (main.cpp:146-199, 353-370) fused into the one re-layout pass:
 *   LEXP_VOL_FILL             fillOutOfView(vol, mode, 0) (main.cpp:146-176): columns that look outside the other view repeat the
 *                             first valid one (view 0: x < d takes x = d; view 1: x > W-1-d takes x = W-1-d);
 *   LEXP_VOL_RIGHT_FROM_LEFT  (mode must be 1) `vol` is the LEFT volume as loaded (im0.acrt, not yet filled); the context's view-1
 *                             volume becomes fillOutOfView(convertVolumeL2R(fillOutOfView(vol, 0)), 1) (main.cpp:356-365), i.e.
 *                             volR[d][y][x] = volL[d][y][min(x + d, W-1)] -- no second volume on the host, no im1.acrt.
 * The host variant uploads in slabs of disparities (LEXP_UPLOAD_SLAB_MB, default 512): no second full-size device copy. */
#define LEXP_VOL_PLAIN 0
#define LEXP_VOL_FILL 1
#define LEXP_VOL_RIGHT_FROM_LEFT 2
LEXP_API int lexp_set_volume_host_ex(lexp_ctx* ctx, int mode, const float* vol_host, int transform);
LEXP_API int lexp_set_volume_device_ex(lexp_ctx* ctx, int mode, const float* vol_device, int transform);

/* Debug / parity: copy the 9 statistics planes [mean_r,g,b, inv_rr,rg,rb,gg,gb,bb] (float[9][H][W]) to the host. */
LEXP_API int lexp_get_stats(lexp_ctx* ctx, int mode, float* out9_host);

/* StereoEnergy::ComputeUnaryPotential / ComputeUnaryPotentialWithoutCheck (StereoEnergy.h:625-626,
 * CostVolumeEnergy.h:55-183) for ONE cell.  `costs` is the pointer the reference passes as
 * `costs.data` -- element (filterRect.y, filterRect.x) of the caller's cost image, row pitch
 * `costs_step_bytes` (cv::Mat::step).  Only costs(targetRect - filterRect.tl()) is written
 * (CostVolumeEnergy.h:169-171,180-182).  Blocking.  with_check != 0 selects ComputeUnaryPotential. */
LEXP_API int lexp_eval_cell(lexp_ctx* ctx, int mode, const lexp_rect* filter_rect, const lexp_rect* target_rect,
                            const lexp_plane* plane, float* costs, ptrdiff_t costs_step_bytes, int with_check);

/* One batched step = the independent cells of one disjoint group with one proposal each
 * (the `#pragma omp parallel for` body at FastGCStereo.h:30-49).  `cost_image` is element (0,0)
 * of the caller's H x W cost image (proposalCost, FastGCStereo.h:25); call i writes
 * cost_image(target_rects[i]).  Host pointers; blocking. */
LEXP_API int lexp_eval_batch(lexp_ctx* ctx, int mode, int n, const lexp_rect* filter_rects,
                             const lexp_rect* target_rects, const lexp_plane* planes, float* cost_image,
                             ptrdiff_t cost_step_bytes, int with_check);

/* Plans: the rects of a (layer, group) never change (LayerManager.h:14-24), only the planes do.
 * A plan tiles every call into CTA work items once and keeps them in HBM. */
LEXP_API int lexp_plan_create(lexp_ctx* ctx, int n, const lexp_rect* filter_rects, const lexp_rect* target_rects,
                              lexp_plan** out_plan);
LEXP_API int lexp_plan_destroy(lexp_plan* plan);
LEXP_API int lexp_plan_num_calls(const lexp_plan* plan);
LEXP_API int lexp_plan_num_items(const lexp_plan* plan);
/* Sum over calls of filterRect pixels (= "evals" of one step), of targetRect pixels, and the
 * algorithmic bytes 20*F + 36*A + 4*S of SURVEY.md section 8(d). */
LEXP_API int lexp_plan_work(const lexp_plan* plan, int64_t* sum_filter_px, int64_t* sum_target_px,
                            int64_t* algorithmic_bytes);

/* Asynchronous evaluation on the context stream; outputs stay in HBM.
 * planes: n planes, on the host (planes_on_device == 0; copied H2D, 16 B each) or on the device.
 * d_cost_image: device pointer to element (0,0) of an H x W float image with row pitch step_bytes. */
LEXP_API int lexp_plan_eval_device(lexp_ctx* ctx, lexp_plan* plan, int mode, const lexp_plane* planes,
                                   int planes_on_device, float* d_cost_image, ptrdiff_t step_bytes, int with_check);
/* Same, but call i writes its targetRect as a contiguous tile (row pitch = targetRect.width) at
 * d_tiles + offset_i, offset_i = sum of targetRect areas of calls 0..i-1 (the layout that is
 * all-gathered between GPUs on the cell-shard path). */
LEXP_API int lexp_plan_eval_device_tiles(lexp_ctx* ctx, lexp_plan* plan, int mode, const lexp_plane* planes,
                                         int planes_on_device, float* d_tiles, int with_check);
/* Host planes in, the per-call contiguous tiles of lexp_plan_eval_device_tiles out into HOST memory (sum of the targetRect
 * areas floats); blocking.  Zero-copy when `tiles` lies in a buffer registered with lexp_host_register, else one contiguous
 * D2H copy.  For a loop restructured step-wise: the fusion of cell i (FastGCStereo.h:52-60) wraps tile i in a cv::Mat header. */
LEXP_API int lexp_plan_eval_host_tiles(lexp_ctx* ctx, lexp_plan* plan, int mode, const lexp_plane* planes, float* tiles,
                                       int with_check);
/* Same, host in / host out (planes H2D, compact tiles D2H, scattered into cost_image); blocking. */
LEXP_API int lexp_plan_eval_host(lexp_ctx* ctx, lexp_plan* plan, int mode, const lexp_plane* planes,
                                 float* cost_image, ptrdiff_t cost_step_bytes, int with_check);

/* Page-lock and map a host buffer (e.g. the caller's cost image, cv::Mat::data) so that the batched host entry
 * points write results straight into it from the kernel over PCIe (zero-copy) instead of staging through a
 * pinned bounce buffer + CPU scatter.  Optional; unregister before freeing the buffer. */
LEXP_API int lexp_host_register(void* ptr, size_t bytes);
LEXP_API int lexp_host_unregister(void* ptr);

LEXP_API int lexp_sync(lexp_ctx* ctx);
/* cudaStream_t of the context (so a caller can order its own device work / events after ours). */
LEXP_API void* lexp_stream(lexp_ctx* ctx);
/* Run all subsequent work of this context on the caller's stream (e.g. torch's current stream, or a stream that is
 * being captured into a CUDA graph: lexp_plan_eval_device* issue only graph-capturable work).  Does not synchronise. */
LEXP_API int lexp_set_stream(lexp_ctx* ctx, void* cuda_stream);
/* Opt in to overlapping launches (programmatic dependent launch) for lexp_plan_eval_device[_tiles] with planes_on_device != 0: a launch
 * may then start -- and read its plane array -- while the context's previous launches are still running (it fills their partly empty
 * last wave; outputs stay ordered).  The caller guarantees that the plane arrays are complete before the PREVIOUS launch of the context was
 * issued (e.g. all proposal steps generated up front).  Off by default; launches whose planes come from the host never overlap; the
 * PatchMatch phase orders itself by flags and always overlaps. */
LEXP_API int lexp_set_overlap(lexp_ctx* ctx, int on);
/* number of kernels this context has launched so far (bench.py's gpu_launches). */
LEXP_API int64_t lexp_launch_count(const lexp_ctx* ctx);
/* Concurrent lexp_eval_cell calls (the OpenMP loop of FastGCStereo.h:30-49, one blocking call per cell and thread) are
 * combined: calls that arrive while the device is busy are evaluated together in one batched launch.  Returns how many
 * such launches there were and how many calls they served (calls that found the device idle are not counted). */
LEXP_API int lexp_combine_stats(const lexp_ctx* ctx, int64_t* batches, int64_t* calls);

/* ---- PatchMatch phase on the device: FastGCStereo::run's `pmInit` iterations (FastGCStereo.h:143-157), i.e.
 * localExpansionMovesForLayer_CPU with doGC == false (FastGCStereo.h:22-72): per cell and proposal
 *     label = proposer->getNextProposal();  ComputeUnaryPotential(...);  mask = currentCost > proposalCost;
 *     proposalCost.copyTo(currentCost, mask);  currentLabeling.setTo(label, mask);                     (:45-60)
 * with currentCost_[mode] / currentLabeling_[mode] (PMStereoBase.h) resident in HBM, the proposal drawn on the device
 * (ExpansionProposer Proposer.h:69-75, RandomProposer :120-148; cv::RNG-compatible streams, one per cell and step) and the
 * update fused into the epilogue of the unary-cost kernel: nothing crosses PCIe between steps.  The proposal steps of a
 * cell are ordered by per-cell completion counters, so consecutive launches overlap on the device. */
#define LEXP_PROP_LIST 0       /* planes supplied by the caller (host list replay; the RansacProposer slot) */
#define LEXP_PROP_EXPANSION 1  /* ExpansionProposer::getNextProposal */
#define LEXP_PROP_RANDOM 2     /* RandomProposer::getNextProposal, m = outerIter + iter */
#define LEXP_PM_INIT 1         /* flags: unconditional write of cost and label (initCurrentFast, FastGCStereo.h:105-113) */
/* (Re)start the state of view `mode`: currentCost = cost (NULL: +INFINITY, FastGCStereo.h:137), currentLabeling = labeling
 * (NULL: zeros); host arrays float[H][W] / lexp_plane[H][W]. */
LEXP_API int lexp_pm_begin(lexp_ctx* ctx, int mode, const float* cost_host, const lexp_plane* labeling_host);
/* Copy the state back (either pointer may be NULL); blocking. */
LEXP_API int lexp_pm_get(lexp_ctx* ctx, int mode, float* cost_host, lexp_plane* labeling_host);
/* Device pointers of the state (for callers that keep working on the device: multi-GPU exchange, disparity maps). */
LEXP_API int lexp_pm_device_state(lexp_ctx* ctx, int mode, float** d_cost, lexp_plane** d_labeling);
/* unitRegion of every call of the plan (where its proposers draw, LayerManager.h:117-121) and a global id per cell (seeds
 * the cell's random streams; NULL: 0..n-1).  Required before lexp_plan_pm_step. */
LEXP_API int lexp_plan_set_units(lexp_plan* plan, const lexp_rect* unit_rects, const int* cell_ids);
/* Zero the per-cell completion counters of all plans of the context (asynchronous).  Call once before the steps of an
 * initialisation or of an iteration are issued (never between its groups: all launches of an iteration are chained by
 * programmatic dependent launch and may overlap). */
LEXP_API int lexp_pm_reset_sync(lexp_ctx* ctx);
/* One proposal step for all cells of the plan (asynchronous, on the context stream).  step_index = 0, 1, ... within the
 * group visit (the steps of a group must be issued in order; lexp_pm_reset_sync between two visits of the same group).  kind / m: LEXP_PROP_*;
 * seed: random stream of this (view, iteration, layer, group, step).  planes: LEXP_PROP_LIST only.  d_planes_out: optional
 * device array [ncalls] receiving the plane every call evaluated.  Always with the validity check (ComputeUnaryPotential). */
LEXP_API int lexp_plan_pm_step(lexp_ctx* ctx, lexp_plan* plan, int mode, int step_index, int kind, int m, uint64_t seed,
                               const lexp_plane* planes, int planes_on_device, lexp_plane* d_planes_out, int flags);

/* ---- multi-GPU cell shard of the PatchMatch phase (SURVEY.md section 8e): one context (process) per GPU, every rank holds the
 * read-only inputs and a full copy of currentCost_ / currentLabeling_, and evaluates its share of the cells of every group.  The
 * exchange is fused into the kernel: the epilogue stores every accepted update into ALL copies (peer memory over NVLink /
 * NVSwitch), and ranks meet at group boundaries through epoch flags written into peer memory by the last work item of a group's
 * last step and polled by the first step of the next group.  No host round trip and no library collective on the data path
 * (NCCL is only used by the caller to broadcast the inputs once).
 * lexp_pm_ipc_export: after lexp_pm_begin; writes LEXP_PM_IPC_BYTES bytes (CUDA IPC handles of cost, labeling, flags) that the caller
 * all-gathers; lexp_pm_ipc_connect: maps the peers' state (handles = world x LEXP_PM_IPC_BYTES, rank order).  lexp_pm_connect_local:
 * the same for contexts living in one process (tests; also multi-device single-process callers). */
#define LEXP_PM_IPC_BYTES 192
#define LEXP_PM_MAX_PEERS 8
LEXP_API int lexp_pm_ipc_export(lexp_ctx* ctx, int mode, void* handles_out);
LEXP_API int lexp_pm_ipc_connect(lexp_ctx* ctx, int mode, int rank, int world, const void* all_handles);
LEXP_API int lexp_pm_connect_local(lexp_ctx* ctx, int mode, int rank, int world, lexp_ctx* const* peer_contexts);
/* lexp_plan_pm_step with the group-boundary protocol.  Consecutive groups overlap spatially, so the first step of a group must
 * not start before the previous group has finished -- on this device and, on the multi-GPU cell shard, on the peers.  Since the
 * launches of an iteration may overlap on the device, this is done with flags too.  Groups are numbered by epochs that only grow; the
 * epochs passed here are RELATIVE to a per-context device counter (the epoch base) that lexp_pm_advance_epoch advances in stream
 * order -- so the launches of one iteration can be captured into a CUDA graph and replayed.  publish_epoch != 0 (last step of
 * a group): when the launch completes, flags[rank] = base + publish_epoch is stored on every copy.  wait_mask / wait_epochs
 * (int[LEXP_PM_MAX_PEERS]; first step of a group): every work item first waits until flags[r] >= base + wait_epochs[r] for every
 * rank r in wait_mask -- the last earlier group each rank owned cells of (<= 0 for groups of the previous iteration). */
LEXP_API int lexp_plan_pm_step_ex(lexp_ctx* ctx, lexp_plan* plan, int mode, int step_index, int kind, int m, uint64_t seed,
                                  const lexp_plane* planes, int planes_on_device, lexp_plane* d_planes_out, int flags,
                                  int publish_epoch, const int* wait_epochs, unsigned wait_mask);
/* epoch base += delta (= the number of groups issued since the last call), asynchronous on the context stream. */
LEXP_API int lexp_pm_advance_epoch(lexp_ctx* ctx, int mode, int delta);

/* ---- The whole PatchMatch phase as one object: what a maintainer calls instead of the pmInit loop of FastGCStereo::run
 * (FastGCStereo.h:143-157).  It owns one plan per (layer, group) of LayerManager::addLayer(unit_sizes[l]) (LayerManager.h:88-185),
 * the proposer list of every layer as (kind, K) pairs in the order of main.cpp:391-397 (LEXP_PROP_EXPANSION / LEXP_PROP_RANDOM; a
 * LEXP_PROP_LIST slot is not allowed here -- use lexp_plan_pm_step for replays), and the epoch bookkeeping of the group boundaries.
 * rank / world: the multi-GPU cell shard (0 / 1 on a single GPU); connect the contexts first (lexp_pm_ipc_connect). */
typedef struct lexp_pm_sweep lexp_pm_sweep;
LEXP_API int lexp_pm_sweep_create(lexp_ctx* ctx, int mode, int n_layers, const int* unit_sizes, const int* n_proposers,
                                  const int* proposer_kind, const int* proposer_K, int rank, int world, lexp_pm_sweep** out);
LEXP_API int lexp_pm_sweep_destroy(lexp_pm_sweep* sweep);
/* number of unit regions of layer 0 (= labels lexp_pm_sweep_init expects) */
LEXP_API int lexp_pm_sweep_num_init_labels(const lexp_pm_sweep* sweep);
/* initCurrentFast (FastGCStereo.h:101-113) with one label per unit region of layer 0 (all of them, in LayerManager order; a rank of
 * a cell shard evaluates its share).  lexp_pm_begin first.  Asynchronous. */
LEXP_API int lexp_pm_sweep_init(lexp_pm_sweep* sweep, const lexp_plane* labels_host);
/* One pm iteration over all layers (FastGCStereo.h:147-157, doGC == false): every cell of every group visited with its layer's
 * proposers, RandomProposer with m = iteration + iter and its early stop (Proposer.h:149-152).  Asynchronous; returns the number
 * of kernel launches issued through *n_launches (may be NULL). */
LEXP_API int lexp_pm_sweep_iteration(lexp_pm_sweep* sweep, int iteration, uint64_t seed, int* n_launches);

/* ---- Pairwise terms and the expansion move on the device (SURVEY.md section 8 f-2 / f-3): the graph-cut iterations of
 * FastGCStereo::run (FastGCStereo.h:171-184, localExpansionMovesForLayer_CPU with doGC == true) on the same device-resident state as
 * the PatchMatch phase (lexp_pm_begin / lexp_pm_get).
 *
 * lexp_set_smoothness: Parameters::lambda / omega / th_smooth / epsilon (StereoEnergy.h:14-39; defaults 1, 10, 1, 0.01 as
 * main.cpp:73 paramsGF).  The coefficient maps smoothnessCoeff[mode][k] of StereoEnergy::initSmoothnessCoeff (StereoEnergy.h:131-163)
 * are (re)built on the device when first needed after this call or after lexp_set_image.
 * lexp_get_smooth_coeff: the eight maps without their margin, float[8][H][W] in the reference's neighbour order (StereoEnergy.h:47-56). */
LEXP_API int lexp_set_smoothness(lexp_ctx* ctx, float lambda, float omega, float th_smooth, float epsilon);
LEXP_API int lexp_get_smooth_coeff(lexp_ctx* ctx, int mode, float* out8_host);
/* StereoEnergy::computeSmoothnessTermsExpansion(currentLabeling_m, label1, region, cost00, cost01, cost10, onlyForward = true, mode)
 * (StereoEnergy.h:398-453) for n (region, proposal) pairs at once, on the current labeling of view `mode` (lexp_pm_begin).  out_host:
 * per call, back to back, float[3][4][region.height][region.width] = cost00, cost01, cost10 for the forward neighbours NB_GE, NB_EG,
 * NB_LG, NB_GG (the only ones the reference fills with onlyForward).  Blocking. */
LEXP_API int lexp_pairwise_terms(lexp_ctx* ctx, int mode, int n, const lexp_rect* regions, const lexp_plane* planes, float* out_host);
/* initCurrentFast for any energy kind (FastGCStereo.h:101-113): for every call of the plan, currentLabeling(targetRect) = planes[call] and
 * currentCost(targetRect) = its unary cost (ComputeUnaryPotential on the call's filterRect).  The cost-volume energy has the same step fused
 * into lexp_plan_pm_step(.., LEXP_PM_INIT); this form also serves the image-based energy (`-mode MiddV2`), whose iterations are all
 * graph-cut iterations.  Asynchronous, stream ordered (host planes are staged before the call returns). */
LEXP_API int lexp_plan_init_step(lexp_ctx* ctx, lexp_plan* plan, int mode, const lexp_plane* planes, int planes_on_device);
/* The reference's cost-volume file, raw float[ndisp][height][width] without a header (`loadMatBinary(.., "im0.acrt", volL, false)`,
 * main.cpp:353-358,364), streamed from disk in slabs through page-locked buffers with the volume preparation `transform`
 * (LEXP_VOL_*) fused in as for lexp_set_volume_host_ex: the 17 GB volume of the 4K configuration never exists in host memory. */
LEXP_API int lexp_set_volume_file(lexp_ctx* ctx, int mode, const char* path, int transform);
/* StereoEnergy::computeDisparities(currentLabeling_[mode]) (StereoEnergy.h:269-272): float[H][W] into host memory; blocking. */
LEXP_API int lexp_get_disparities(lexp_ctx* ctx, int mode, float* out_host);
/* cvutils::io::save_pfm_file (Utilities.hpp:84-137) for a 1-channel float image (disp0.pfm of main.cpp:319,410): byte-identical file. */
LEXP_API int lexp_save_pfm(const char* path, const float* image, int width, int height, ptrdiff_t step_bytes);
/* Energy of the current state of view `mode`, as the reference logs it (Evaluator / PMStereoBase.h:266): *data_term = sum of currentCost_,
 * *smoothness_term = StereoEnergy::computeSmoothnessCost(currentLabeling_m) (StereoEnergy.h:165-199).  Either pointer may be NULL.  Blocking. */
LEXP_API int lexp_energy(lexp_ctx* ctx, int mode, double* data_term, double* smoothness_term);
/* One proposal step of a group with the graph-cut move: for every call (cell) of the plan -- proposal (kind / m / seed / planes as
 * lexp_plan_pm_step), ComputeUnaryPotential on the cell's filterRect, then FastGCStereo::expansionMoveBK on its targetRect
 * (= sharedRegion): graph of FastGCStereo.h:424-549 from the unary costs, the pairwise terms and the boundary terms, its minimum cut,
 * and `copyTo / setTo` of cost and label where the proposal wins (FastGCStereo.h:53-59).  The cells of the plan must be pairwise
 * non-adjacent (a disjoint group of LayerManager, LayerManager.h:168-173).  lexp_plan_set_units first.  Asynchronous and stream ordered
 * for plans whose cells have at most LEXP_GC_BIG_NODES (default 32768) nodes: one CTA per cell; plans with larger cells (layer 2) run the
 * same steps as phase kernels over all SMs with two flags read back per decision -- that form returns when the moves are done.
 * d_planes_out: optional device array [ncalls] (the plane every call evaluated); d_flows_out: optional device array double[ncalls]
 * (the value expansionMoveBK returns: the minimum-cut energy of the move). */
LEXP_API int lexp_plan_gc_step(lexp_ctx* ctx, lexp_plan* plan, int mode, int kind, int m, uint64_t seed, const lexp_plane* planes,
                               int planes_on_device, lexp_plane* d_planes_out, double* d_flows_out);

/* One iteration of the main (graph-cut) loop of FastGCStereo::run (FastGCStereo.h:171-184) over the schedule of a sweep object
 * (lexp_pm_sweep_create with world == 1): lexp_plan_gc_step for every proposal step of every group.  Asynchronous. */
LEXP_API int lexp_pm_sweep_gc_iteration(lexp_pm_sweep* sweep, int iteration, uint64_t seed, int* n_steps);

/* LayerManager::addLayer (LayerManager.h:44-185): cell geometry of one layer.
 * Call with rect pointers == NULL to query counts.  group_of[r] = (i%4)*4 + (j%4) (LayerManager.h:168-173). */
LEXP_API int lexp_layer_geometry(int width, int height, int windR, int unit_size, int* height_blocks,
                                 int* width_blocks, lexp_rect* unit_regions, lexp_rect* shared_regions,
                                 lexp_rect* filter_regions, int* group_of);

#ifdef __cplusplus
}
#endif
#endif /* LEXP_CUDA_H_ */
