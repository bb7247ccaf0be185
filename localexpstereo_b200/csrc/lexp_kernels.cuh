// lexp_kernels.cuh -- hand-written sm_100a kernels of the unary-cost hot path.
//
// K0  lexp_stats_*      one-time guided-filter statistics       (GuidedFilter.h:58-102)
// K1+K2+K3 fused        lexp_fused_kernel: plane-cost sampling + truncation
//                       (CostVolumeEnergy.h:69-98), guided filter filter_raw
//                       (GuidedFilter.h:142-247) with the sub-region window counts of
//                       createSubregionFilter (GuidedFilter.h:301-326), validity mask
//                       (StereoEnergy.h:577-610, CostVolumeEnergy.h:176-183).
// File:line citations are relative to /root/reference/LocalExpansionStereo/.
//
// Design (DESIGN.md section 3): one CTA = one output tile (<= 64 columns) of one (cell, plane) call.  The CTA streams
// top-to-bottom over the rows of the tile's dependency cone (tile +- 2R) in chunks of kCH rows.  Four warp teams form a
// producer/consumer pipeline; each hand-off is a double-buffered shared-memory row buffer guarded by a pair of named
// barriers (bar.arrive / bar.sync), all intermediates stay in shared memory / registers:
//   A (4 warps, thread = column): gather p = min(lerp(V, plane), th) from the blocked volume (register batch of kG rows,
//       one batch of loads in flight), products {p, I0 p, I1 p, I2 p}, running column sums over 2R+1 rows
//       (thread-private ring of the rows to subtract later)              -> hb1
//       NAIVE: the raw cost comes from the warped other view instead (NaiveStereoEnergy, StereoEnergy.h:694-754)
//   H (2 warps, thread = run of 8 columns): horizontal window sums: warp 0 hb1 -> ho1, warp 1 hb2 -> ho2
//   C (3 warps, thread = column): (a, b) from the stage-1 box sums and the precomputed
//       statistics, running column sums of {a0, a1, a2, b}                -> hb2
//   E (2 warps, thread = column): q = (Bb + Ba.I) / N, validity mask, store.
// float4 quantities are held as two packed f32x2 registers and added with Blackwell's
// FADD2 (add.rn.f32x2): two FP32 adds per issue slot.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lexp {

constexpr int kWarpsA = 4, kWarpsH = 2, kWarpsC = 3, kWarpsE = 2;
constexpr int kThreads = 32 * (kWarpsA + kWarpsH + kWarpsC + kWarpsE);  // 352
constexpr int kMaxVW = 32 * kWarpsA;   // virtual tile width  ow + 4R
constexpr int kMaxW2 = 32 * kWarpsC;   // (a,b) columns       ow + 2R
constexpr int kMaxOW = 32 * kWarpsE;   // output columns
constexpr int kRun = 8;                // columns per H task
constexpr int kCH = 2;                 // rows per pipeline chunk
// ---- measured design choices (B200, profiles/r2_variants.md) ---------------------------------------------------------------
// Row table: the byte offset of a volume row inside the blocked layout, (y / 4) * block-row pitch + (y % 4) * 16, is looked up
//   in a per-tile shared-memory table (16-byte units, filled in the prologue next to the plane's b*y + c) instead of being
//   recomputed with 64-bit multiplies for every row of every column: ~19 -> ~5 address instructions per gathered row in team A,
//   17.56 -> 17.26 ms per sweep.
// Programmatic dependent launch (PDL): every thread signals `griddepcontrol.launch_dependents` at the top of the kernel, so the
//   NEXT batched evaluation of the stream (launched with the programmatic-stream-serialization attribute, lexp_capi.cu) may
//   occupy CTA slots as soon as all CTAs of this one are resident: it fills the partly empty last wave and hides the launch gap
//   and its own prologue + 4R warm-up rows.  Consecutive launches write overlapping parts of the same cost image (the steps of a
//   group), so team E executes `griddepcontrol.wait` (previous grids complete, their writes visible) before its first store;
//   nothing else written by a previous launch is read.  17.56 -> 15.49 ms per sweep (the 240 launches of a sweep replayed as one
//   CUDA graph).
// ---- build-time switch -----------------------------------------------------------------------------------------------------
// LEXP_TRACE: diagnosis build.  Every warp accumulates the clock cycles it spends waiting for its input link (consume_begin) and
//   for a free output buffer (produce_begin) and writes {total, wait_in, wait_out, chunks} at the end; lexp_capi.cu averages
//   them per team after every launch (LEXP_TRACE_FILE).  Shows directly which team the pipeline waits for.  Not a product build.
#ifndef LEXP_TRACE
#define LEXP_TRACE 0
#endif
constexpr int kMinCtas = 2;           // resident CTAs per SM the kernel is compiled for (register cap 65536 / (kMinCtas * kThreads))
constexpr int kG = 6;                 // rows per gather batch of team A (one batch of loads in flight)
constexpr float kCostInvalid = 1000000.0f;  // StereoEnergy.h:45
constexpr int kMaxPeers = 8;                // GPUs of one NVSwitch domain that share a PatchMatch-phase state

struct __align__(16) Item {  // one CTA work item (64 B)
    int fx, fy, fw, fh;      // filterRect of the call
    int ox0, oy0, ow, oh;    // output tile (image coordinates), inside targetRect
    int call;                // index of the call (plane / compact slot)
    int compact_off;         // float offset of the tile's first pixel in the compact output
    int compact_stride;      // = targetRect.width
    int flags;               // bit0: targetRect is 1x1 (IsValiLabel fast path, StereoEnergy.h:579-583)
    int pad[4];
};

struct Plane4 { float a, b, c, v; };

// per-call (= per cell) data of the device-side PatchMatch phase (FastGCStereo.h:22-72 with doGC == false)
struct __align__(16) CallInfo {
    int ux, uy, uw, uh;      // unitRegion of the cell: where the proposers draw their source pixel (Proposer.h:38-45,69-75)
    int n_done_per_step;     // completion signals one proposal step of this cell produces (its work items x kWarpsE)
    int cell_id;             // global id of the cell (seeds its random stream; independent of how cells are sharded over GPUs)
    int n_items;             // work items (tiles) of the cell = tickets drawn per proposal step
    int pad;
};
// per-call synchronisation record of a group (zeroed before the group's first step)
struct __align__(16) CellSync {
    int done;                // completion signals so far (all steps)
    int ticket;              // work items that have started so far (all steps): the first one of a step draws the proposal
    int ready;               // = step + 1 once `plane` holds the proposal of that step
    int pad;
    Plane4 plane;            // the proposal of the current step, shared by all work items of the cell
};

struct KParams {
    const float* __restrict__ vol;      // blocked cost volume float[Hb][Wb][D][4 rows][4 px], Hb = ceil(H/4), Wb = ceil(W/4) (lexp_relayout_volume)
    int Wb;
    const uchar4* __restrict__ guide;   // uchar4[H][W] = (c0,c1,c2,0), OpenCV BGR order
    const float4* __restrict__ statA;   // float4[H][W] = {mean0, mean1, mean2, inv00}
    const float4* __restrict__ statB;   // float4[H][W] = {inv01, inv02, inv11, inv12}
    const float* __restrict__ statC;    // float [H][W] =  inv22
    const Item* __restrict__ items;
    const Plane4* __restrict__ planes;
    float* __restrict__ out;
    long long out_pitch;                // floats per row (image mode)
    int out_compact;                    // 1: per-call contiguous tiles, 0: H x W image
    int H, W, D;
    float th_col, min_disp, max_disp;
    int with_check;
    int R;                              // guided-filter box radius (windR / 2)
    // NaiveStereoEnergy (StereoEnergy.h:629-764): image-based raw cost instead of the cost volume
    const float4* __restrict__ exi_own;   // ExI[mode]      float4[H][W] = {c0,c1,c2 * (1-alpha), alpha * Sobel_x(gray)}
    const float4* __restrict__ exi_other; // ExI[1 - mode]
    float thresh_color, thresh_gradient;  // StereoEnergy.h:663-664
    int mode;                             // 0: left reference view, 1: right
    int fast_ok;                        // MIN == 0, MAX == D-1, th_col >= 0 and the volume holds no NaN/Inf
    // ---- device-side PatchMatch phase (pm_mode != 0): proposal -> unary cost -> `mask = cur > prop; copy; setTo`
    // (FastGCStereo.h:34-60 with doGC == false) without leaving the device
    int smem_plane_off;                 // byte offset of a 16-byte slot at the end of the launch's dynamic shared memory
    int pm_mode;                        // 0: unary costs only (out); 1: fused update of cur_cost / cur_label; 2: initialisation (unconditional write, :105-113)
    int prop_kind;                      // 0: planes[call] (host list / RANSAC slot), 1: ExpansionProposer, 2: RandomProposer
    int prop_m;                         // RandomProposer: m = outerIter + iter (Proposer.h:124)
    int step_index;                     // proposal step within the group: the cell's previous steps must have completed
    unsigned long long seed;            // random stream of this (view, iteration, layer, group, step); hashed with the cell id
    float* __restrict__ cur_cost;       // float [H][W]   currentCost_[mode]
    float4* __restrict__ cur_label;     // float4[H][W]   currentLabeling_[mode] (Plane = 4 floats, Plane.h:4-8)
    const CallInfo* __restrict__ calls; // [ncalls]
    CellSync* cell_sync;                // [ncalls] completion counters / proposal hand-over of the group (zeroed before its first step)
    Plane4* planes_out;                 // [ncalls] the plane each call evaluated in this step (optional: replay / logging)
    // ---- multi-GPU cell shard of the PatchMatch phase (SURVEY.md 8e): every rank holds a full copy of the state; an accepted update
    // is stored into ALL copies by the kernel itself (peer memory over NVLink), ranks meet at group boundaries through epoch flags
    int n_copies;                       // copies of the state the epilogue writes (1: only this device's)
    float* copy_cost[kMaxPeers];        // [n_copies] currentCost_ of this rank (entry 0) and of its peers (P2P-mapped)
    float4* copy_label[kMaxPeers];      // [n_copies]
    int* copy_flags[kMaxPeers];         // [n_copies] epoch flags int[kMaxPeers] of every copy: flags[r] = last group rank r completed
    int my_rank;
    // epochs are relative to *epoch_base (a device counter the host advances once per iteration): the launches of an iteration
    // can then be replayed as a CUDA graph while the epochs keep growing
    const int* epoch_base;
    int* err_flag;                      // set to 1 if a wait for a peer gave up (the host then reports an error instead of hanging)
    int publish_epoch;                  // != 0: the last work item of this launch stores flags[my_rank] = base + publish_epoch on every copy
    int wait_epochs[kMaxPeers];         // every work item first waits until flags[r] >= base + wait_epochs[r] for all ranks r in wait_mask
    unsigned wait_mask;
    int* launch_done;                   // completion counter of this launch (zeroed with the group's CellSync records)
#if LEXP_TRACE
    long long* trace;                   // [items][kThreads / 32][4]
#endif
};

// largest output-tile width the team sizes allow for box radius R
__host__ __device__ inline int max_tile_ow(int R) {
    int a = kMaxVW - 4 * R, b = kMaxW2 - 2 * R, c = kMaxOW;
    int m = a < b ? a : b;
    return m < c ? m : c;
}
__host__ __device__ __forceinline__ int sidx(int x) { return x + (x >> 3); }  // 1 pad slot per 8 columns
__host__ __device__ inline int srow_stride(int vw) {
    int s = sidx(vw + kRun + 7) + 1;
    return s + ((12 - (s & 7)) & 7);  // == 4 (mod 8) float4 units: the 2 rows x 4 runs of a quarter-warp hit 8 bank groups
}
__host__ __device__ inline size_t fused_smem_bytes(int vw, int oh, int R) {
    const int K = 2 * R + 1;
    const int vh = oh + 4 * R;
    const int rows = 8 * kCH * srow_stride(vw);
    return (size_t)((K * vw + 1) / 2 + K * (vw - 2 * R) + rows + 3 * ((vh + 3) / 4) + 3) * 16 + 16;  // + 6 doubles (NAIVE: inverse affine map) + the plane slot (PatchMatch phase) at the very end
}

// ---- packed f32x2 helpers (sm_100: FADD2 / FFMA2) --------------------------------------------
typedef unsigned long long u64;
struct __align__(16) F4 { u64 lo, hi; };  // lo = (x, y), hi = (z, w)
#ifndef LEXP_EMU
__device__ __forceinline__ u64 pk2(float a, float b) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void up2(u64 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
#define LEXP_LOADS_LANDED(...) asm volatile("" : __VA_ARGS__ :: "memory")
#define LEXP_DYNAMIC_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define LEXP_NOINLINE __noinline__
#else  // host emulation of the same operations (tests/emu/, test infrastructure only)
inline u64 pk2(float a, float b) { return (u64)__float_as_uint(a) | ((u64)__float_as_uint(b) << 32); }
inline void up2(u64 v, float& a, float& b) { a = __uint_as_float((unsigned)v); b = __uint_as_float((unsigned)(v >> 32)); }
inline u64 add2(u64 a, u64 b) { float a0, a1, b0, b1; up2(a, a0, a1); up2(b, b0, b1); return pk2(__fadd_rn(a0, b0), __fadd_rn(a1, b1)); }
inline u64 sub2(u64 a, u64 b) { float a0, a1, b0, b1; up2(a, a0, a1); up2(b, b0, b1); return pk2(__fsub_rn(a0, b0), __fsub_rn(a1, b1)); }
#define LEXP_LOADS_LANDED(...) ((void)0)
#define LEXP_DYNAMIC_SMEM(name) unsigned char* name = emu::dyn_smem()
#define LEXP_NOINLINE
#endif
__device__ __forceinline__ F4 f4add(F4 a, F4 b) { return F4{add2(a.lo, b.lo), add2(a.hi, b.hi)}; }
__device__ __forceinline__ F4 f4sub(F4 a, F4 b) { return F4{sub2(a.lo, b.lo), sub2(a.hi, b.hi)}; }
__device__ __forceinline__ F4 f4zero() { return F4{0ull, 0ull}; }

// ---- named barriers: pairwise producer/consumer hand-off between warp teams ------------------------
// link L (0: A->H1 via hb1, 1: H1->C via ho1, 2: C->H2 via hb2, 3: H2->E via ho2), buffer parity b:
//   FULL  id = 4 L + b       producer bar.arrive after writing, consumer bar.sync before reading
//   EMPTY id = 4 L + 2 + b   consumer bar.arrive after reading, producer bar.sync before overwriting (chunk >= 2)
#ifndef LEXP_EMU
__device__ __forceinline__ void bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
#else
inline void bar_sync(int id, int nthreads) { emu::barrier(id, nthreads, true); }
inline void bar_arrive(int id, int nthreads) { emu::barrier(id, nthreads, false); }
#endif
__device__ __forceinline__ void produce_begin(int link, int c, int nthreads) { if (c >= 2) bar_sync(4 * link + 2 + (c & 1), nthreads); }
__device__ __forceinline__ void produce_end(int link, int c, int nthreads) { bar_arrive(4 * link + (c & 1), nthreads); }
__device__ __forceinline__ void consume_begin(int link, int c, int nthreads) { bar_sync(4 * link + (c & 1), nthreads); }
__device__ __forceinline__ void consume_end(int link, int c, int nChunks, int nthreads) { if (c + 2 < nChunks) bar_arrive(4 * link + 2 + (c & 1), nthreads); }
#if LEXP_TRACE  // timed versions: `(name)(...)` calls the function, not the macro
#define consume_begin(link, c, n) do { const unsigned t__ = (unsigned)clock64(); (consume_begin)(link, c, n); tr_wait_in += (unsigned)clock64() - t__; } while (0)
#define produce_begin(link, c, n) do { const unsigned t__ = (unsigned)clock64(); (produce_begin)(link, c, n); tr_wait_out += (unsigned)clock64() - t__; } while (0)
// cycles until a register filled by an earlier global load is readable (the MOV stalls on the scoreboard)
#ifndef LEXP_EMU
#define LEXP_TRACE_LOAD_WAIT(reg32) do { const unsigned t__ = (unsigned)clock64(); unsigned d__; asm volatile("mov.b32 %0, %1;" : "=r"(d__) : "r"(reg32)); \
                                         tr_wait_ld += (unsigned)clock64() - t__; } while (0)
#else
#define LEXP_TRACE_LOAD_WAIT(reg32) do { tr_wait_ld += 0u * (unsigned)(reg32); } while (0)
#endif
#else
#define LEXP_TRACE_LOAD_WAIT(reg32) ((void)0)
#endif
constexpr int kLinkAH = 32 * (4 + 1), kLinkHC = 32 * (1 + 3), kLinkCH = 32 * (3 + 1), kLinkHE = 32 * (1 + 2);  // threads per link

// Inverse affine map (dst pixel of the filterRect -> source pixel of the other view) of NaiveStereoEnergy
// (StereoEnergy.h:704-729), computed the way the reference does: the three float corner correspondences, then
// cv::getAffineTransform (6x6 system, Gaussian elimination with partial pivoting in double) and the inversion at the top of
// cv::warpAffine -- same operations in the same order as oracle/_ref, every product and sum rounded separately (no FMA
// contraction), so the 10-bit fixed-point source coordinates are bit-identical to the reference's.  One thread per CTA.
__device__ LEXP_NOINLINE void naive_inverse_affine(const Item it, const Plane4 pl, int mode, double* iM) {
    const float sign = mode ? -1.0f : 1.0f;
    const float x00 = (float)it.fx, y00 = (float)it.fy;
    const float x11 = __fadd_rn(x00, (float)it.fw), y11 = __fadd_rn(y00, (float)it.fh);
    auto gz = [&](float x, float y) { return __fadd_rn(__fadd_rn(__fmul_rn(pl.a, x), __fmul_rn(pl.b, y)), pl.c); };  // Plane.h:51-54
    float sx[3], sy[3];
    sx[0] = __fsub_rn(x00, __fmul_rn(sign, gz(x00, y00))); sy[0] = y00;   // :714-719
    sx[1] = __fsub_rn(x00, __fmul_rn(sign, gz(x00, y11))); sy[1] = y11;
    sx[2] = __fsub_rn(x11, __fmul_rn(sign, gz(x11, y00))); sy[2] = y00;
    if (pl.v != 0.0f) { sy[0] = __fadd_rn(sy[0], pl.v); sy[1] = __fadd_rn(sy[1], pl.v); sy[2] = __fadd_rn(sy[2], pl.v); }  // :720-725
    const double dx[3] = {0.0, 0.0, (double)__fsub_rn(x11, x00)}, dy[3] = {0.0, (double)__fsub_rn(y11, y00), 0.0};   // :711-713
    double a[6][7];
    for (int i = 0; i < 3; i++) {
        a[i][0] = sx[i]; a[i][1] = sy[i]; a[i][2] = 1.0; a[i][3] = 0.0; a[i][4] = 0.0; a[i][5] = 0.0; a[i][6] = dx[i];
        a[i + 3][0] = 0.0; a[i + 3][1] = 0.0; a[i + 3][2] = 0.0; a[i + 3][3] = sx[i]; a[i + 3][4] = sy[i]; a[i + 3][5] = 1.0; a[i + 3][6] = dy[i];
    }
    double M[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    bool singular = false;
    for (int c = 0; c < 6 && !singular; c++) {
        int piv = c;
        for (int r = c + 1; r < 6; r++) if (fabs(a[r][c]) > fabs(a[piv][c])) piv = r;
        if (fabs(a[piv][c]) < 2.220446049250313e-16) { singular = true; break; }
        if (piv != c) for (int k = 0; k < 7; k++) { const double t = a[c][k]; a[c][k] = a[piv][k]; a[piv][k] = t; }
        const double d = __ddiv_rn(-1.0, a[c][c]);
        for (int r = c + 1; r < 6; r++) {
            const double f = __dmul_rn(a[r][c], d);
            for (int k = c + 1; k < 7; k++) a[r][k] = __dadd_rn(a[r][k], __dmul_rn(f, a[c][k]));
        }
    }
    if (!singular) {
        for (int r = 5; r >= 0; r--) {
            double s = a[r][6];
            for (int k = r + 1; k < 6; k++) s = __dsub_rn(s, __dmul_rn(a[r][k], M[k]));
            M[r] = __ddiv_rn(s, a[r][r]);
        }
    }
    // cv::warpAffine without WARP_INVERSE_MAP inverts M in double
    double D = __dsub_rn(__dmul_rn(M[0], M[4]), __dmul_rn(M[1], M[3]));
    D = D != 0.0 ? __ddiv_rn(1.0, D) : 0.0;
    const double A11 = __dmul_rn(M[4], D), A22 = __dmul_rn(M[0], D);
    iM[0] = A11; iM[1] = __dmul_rn(M[1], -D); iM[3] = __dmul_rn(M[3], -D); iM[4] = A22;
    iM[2] = __dsub_rn(__dmul_rn(-iM[0], M[2]), __dmul_rn(iM[1], M[5]));
    iM[5] = __dsub_rn(__dmul_rn(-iM[3], M[2]), __dmul_rn(iM[4], M[5]));
}

// ---- device-side proposers of the PatchMatch phase ------------------------------------------------------------------------
// cv::RNG (OpenCV core: multiply-with-carry, 64-bit state) -- the generator behind cv::theRNG() that the reference's proposers
// draw from (Proposer.h:40,132,147; Utilities.hpp:254-261).  Same integer recurrence and the same float / double conversions,
// every floating-point operation rounded separately, so a stream started from the same state yields the same proposals.
struct CvRng {
    u64 state;
    __device__ unsigned next() {
        state = (u64)(unsigned)state * 4164903690ull + (u64)(unsigned)(state >> 32);
        return (unsigned)state;
    }
    __device__ int uniform_int(int a, int b) { return a == b ? a : (int)(next() % (unsigned)(b - a) + (unsigned)a); }
    __device__ float uniform_float(float a, float b) {
        const float r = __fmul_rn((float)next(), 2.32830643653869629E-10f);
        return __fadd_rn(__fmul_rn(r, __fsub_rn(b, a)), a);
    }
    __device__ double uniform_double(double a, double b) {
        const unsigned t = next();
        const u64 w = ((u64)t << 32) | (u64)next();
        const double r = __dmul_rn(__ull2double_rn(w), 5.4210108624275221700372640043497e-20);
        return __dadd_rn(__dmul_rn(r, __dsub_rn(b, a)), a);
    }
};
// Start state of the random stream of one (cell, proposal step): the reference draws from a per-thread cv::theRNG() whose
// assignment to cells is arbitrary; here every (launch seed, cell id) pair gets its own stream (splitmix64 finaliser), so the
// result does not depend on scheduling or on how cells are sharded over GPUs.  Restated by oracle.pm_rng_state.
__host__ __device__ inline u64 pm_rng_state(u64 seed, int cell_id) {
    u64 z = seed + 0x9E3779B97F4A7C15ull * (u64)(unsigned)(cell_id + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z = z ^ (z >> 31);
    return z ? z : 0xffffffffull;   // cv::RNG(0) starts from 0xffffffff
}
// One proposal of ExpansionProposer (Proposer.h:69-75: the current label of a random pixel of the unitRegion) or of
// RandomProposer (Proposer.h:120-148: that label with its disparity at the pixel and its normal perturbed), MAX_VDISPARITY = 0.
// Executed by one thread of the CTA; kept out of line so that it does not weigh on the register allocation of the pipeline.
struct ProposeArgs {   // by value: a reference to the kernel parameters would force them into a stack frame
    u64 seed; const float4* cur_label; int W, prop_kind, prop_m; float min_disp, max_disp;
};
__device__ LEXP_NOINLINE float4 pm_propose(const ProposeArgs P, const int ux, const int uy, const int uw, const int uh, const int cell_id) {
    CvRng rng{pm_rng_state(P.seed, cell_id)};
    const int n = rng.uniform_int(0, uw * uh);                          // selectRandomPixelInRect (:38-45)
    const int sx = ux + n % uw, sy = uy + n / uw;
    const float4 in4 = __ldcg(P.cur_label + (size_t)sy * P.W + sx);   // L2: written by other SMs, possibly by a launch still running
    const Plane4 in{in4.x, in4.y, in4.z, in4.w};
    if (P.prop_kind == 1) return in4;                                    // ExpansionProposer (:69-75)
    const float fx = (float)sx, fy = (float)sy;
    float zs = __fadd_rn(__fadd_rn(__fmul_rn(in.a, fx), __fmul_rn(in.b, fy)), in.c);   // Plane::GetZ (Plane.h:51-54)
    const float scale = exp2f(-(float)(P.prop_m + 1));                                 // pow(0.5f, m + 1): exact
    const float dz = __fmul_rn(__fsub_rn(P.max_disp, P.min_disp), scale);              // :107-110
    const float minz = fmaxf(P.min_disp, __fsub_rn(zs, dz)), maxz = fminf(P.max_disp, __fadd_rn(zs, dz));
    zs = rng.uniform_float(minz, maxz);                                                 // :132
    const float nr = exp2f(-(float)P.prop_m);                                           // randomNmax * pow(0.5f, m) (:143)
    const double theta = rng.uniform_double(0.0, 3.14159265358979323846);               // getRandomUnitVector (Utilities.hpp:254-261)
    const double phi = rng.uniform_double(0.0, __dmul_rn(3.14159265358979323846, 2.0));
    const double cT = cos(theta), sT = sin(theta), cP = cos(phi), sP = sin(phi);
    const float r0 = (float)__dmul_rn(sT, cP), r1 = (float)__dmul_rn(sT, sP), r2 = (float)cT;
    // Plane::GetNormal (Plane.h:42-50): sqrt in double, then cast to float
    const float gnz = (float)__ddiv_rn(1.0, sqrt(__dadd_rn(__dadd_rn(1.0, (double)__fmul_rn(in.a, in.a)), (double)__fmul_rn(in.b, in.b))));
    const float gnx = __fmul_rn(-in.a, gnz), gny = __fmul_rn(-in.b, gnz);
    const float v0 = __fadd_rn(gnx, __fmul_rn(r0, nr)), v1 = __fadd_rn(gny, __fmul_rn(r1, nr)), v2 = __fadd_rn(gnz, __fmul_rn(r2, nr));  // :144
    double dd = __dmul_rn((double)v0, (double)v0);                                      // nv.ddot(nv), then nv / sqrt(.) = nv * (1 / sqrt(.))  (:146)
    dd = __dadd_rn(dd, __dmul_rn((double)v1, (double)v1));
    dd = __dadd_rn(dd, __dmul_rn((double)v2, (double)v2));
    const double inv = __ddiv_rn(1.0, sqrt(dd));
    const float nx = (float)__dmul_rn((double)v0, inv), ny = (float)__dmul_rn((double)v1, inv), nz = (float)__dmul_rn((double)v2, inv);
    float4 out;                                                                         // Plane::CreatePlane (Plane.h:23-31)
    out.x = __fdiv_rn(-nx, nz);
    out.y = __fdiv_rn(-ny, nz);
    out.z = __fsub_rn(__fsub_rn(zs, __fmul_rn(out.x, fx)), __fmul_rn(out.y, fy));
    out.w = in.v;
    return out;
}
// acquire load / polling of a completion counter written by CTAs of earlier launches that may still be running (PDL)
__device__ __forceinline__ int ld_acquire_sys(const int* p) {   // a flag written by another GPU
#ifndef LEXP_EMU
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
#else
    return *reinterpret_cast<const volatile int*>(p);
#endif
}
__device__ __forceinline__ void st_release_sys(int* p, int v) {
#ifndef LEXP_EMU
    asm volatile("st.release.sys.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
#else
    *reinterpret_cast<volatile int*>(p) = v;
#endif
}
__device__ __forceinline__ int ld_acquire(const int* p) {
#ifndef LEXP_EMU
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
#else
    return *reinterpret_cast<const volatile int*>(p);
#endif
}

// Cost-volume samples: plain read-only loads.  Measured on B200 (profiles/r1_experiments.md): letting them allocate in
// L1 (the d0 / d0+1 samples of a 4-pixel block share 128-byte lines) beats L1::no_allocate + L2 evict-first by 8 %.
__device__ __forceinline__ float ldg_stream(const float* p) { return __ldg(p); }

template <int R_T, bool NAIVE, bool PM>
__global__ void __launch_bounds__(kThreads, kMinCtas) lexp_fused_kernel(const KParams P) {
    const int R = R_T > 0 ? R_T : P.R;
    const int K = 2 * R + 1;
    LEXP_DYNAMIC_SMEM(smem_raw);
    F4* smem = reinterpret_cast<F4*>(smem_raw);

#ifndef LEXP_EMU
    asm volatile("griddepcontrol.launch_dependents;");
#endif
#if LEXP_TRACE
    unsigned tr_wait_in = 0, tr_wait_out = 0, tr_wait_ld = 0;  // 32-bit cycle counts: a work item runs for ~1e5 cycles
    const unsigned tr_t0 = (unsigned)clock64();
#endif
    const Item it = P.items[blockIdx.x];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    Plane4 pl;
    if (!PM) pl = P.planes[it.call];
    const int VW = it.ow + 4 * R;
    const int X0 = it.ox0 - 2 * R;
    const int W2 = VW - 2 * R;
    const int SW = srow_stride(VW);   // row stride of hb1 (stage-1 column sums, VW columns)
    const int SW2 = SW, SW3 = SW;
    const int fx1 = it.fx + it.fw, fy1 = it.fy + it.fh;
    // streamed rows y = ys + v, v in [0, VHs): the dependency cone of the tile, minus leading rows above
    // the filterRect (they are zero padding).  Rows >= fy1 are zero rows that flush the running sums.
    const int ys = max(it.oy0 - 2 * R, it.fy);
    const int VHs = it.oy0 + it.oh + 2 * R - ys;
    const int vReal = min(VHs, fy1 - ys);                    // rows [0, vReal) lie inside the filterRect
    const int vC0 = max(it.oy0 - R, it.fy) + R - ys;         // first v whose stage-1 centre row (y - R) is needed
    const int vC1 = min(VHs, fy1 + R - ys);                  // centre rows >= fy1 are zero rows
    const int vE0 = it.oy0 + 2 * R - ys;                     // first v whose stage-2 centre row (y - 2R) is an output row

    uint2* ring1 = reinterpret_cast<uint2*>(smem);   // [K][VW] {p, packed guide}: the products are recomputed when a row leaves the window
    F4* ring2 = smem + (K * VW + 1) / 2;              // [K][W2]
    F4* hb1 = ring2 + K * W2;              // [2][CH][SW] stage-1 column sums   (index: column - X0)
    F4* ho1 = hb1 + 2 * kCH * SW;          // [2][CH][SW2] stage-1 box sums     (index: column - X0 - R)
    F4* hb2 = ho1 + 2 * kCH * SW2;         // [2][CH][SW2] stage-2 column sums  (index: column - X0 - R)
    F4* ho2 = hb2 + 2 * kCH * SW2;         // [2][CH][SW3] stage-2 box sums     (index: column - X0 - 2R)
    float* s_invny = reinterpret_cast<float*>(ho2 + 2 * kCH * SW3);  // [VHs] 1 / (#rows of the window inside filterRect)
    float* s_dbase = s_invny + 4 * ((it.oh + 4 * R + 3) / 4);        // [VHs] b*y + c of the plane  (NAIVE: int X0 of the warp)
    int* s_Y0 = reinterpret_cast<int*>(s_dbase + 4 * ((it.oh + 4 * R + 3) / 4));  // [VHs] NAIVE: fixed-point source row
    double* s_iM = reinterpret_cast<double*>(s_Y0 + 4 * ((it.oh + 4 * R + 3) / 4));  // [6] NAIVE: inverse affine map of the call

    if (PM) {
        // PatchMatch phase.  (0) Group boundary: the previous group (this rank's and, on the multi-GPU cell shard, the peers') must
        // have finished -- its last launch stored an epoch flag when its last work item completed; all launches of an iteration are
        // chained by programmatic dependent launch, so this launch may have started long before.  (1) This cell's previous proposal
        // steps (all their work items) must have updated cur_cost / cur_label before the proposer reads a label and before this
        // step's own update (FastGCStereo.h:41-60 is sequential per cell): per-cell counters, written by CTAs of earlier launches
        // that may still be running.  (2) The proposal is drawn ONCE per (cell, step), by the first of the cell's work items to
        // arrive (ticket; tickets of the next step can only be taken after all of this step's, because of (1)), and handed to the
        // others through global memory: no work item of the step can write a label before the proposer has read its source label.
        // Warp 0 does this while the other warps zero the shared-memory rings.
        Plane4& s_pl = *reinterpret_cast<Plane4*>(smem_raw + P.smem_plane_off);   // last 16 bytes of the launch's dynamic shared memory
        if (tid == 0) {
            if (P.wait_mask) {
                const int base = *P.epoch_base;
                for (int r = 0; r < kMaxPeers; r++)
                    if ((P.wait_mask >> r) & 1u) {
                        unsigned polls = 0;   // a peer that never arrives (a crashed rank) must not hang this GPU: give up after ~10 s,
                        while (ld_acquire_sys(P.copy_flags[0] + r) < base + P.wait_epochs[r]) {   // and at once when somebody already has
#ifndef LEXP_EMU
                            __nanosleep(200);
#endif
                            if (++polls > (1u << 25) || ((polls & 1023u) == 0 && ld_acquire(P.err_flag))) { atomicExch(P.err_flag, 1); break; }
                        }
                    }
            }
            const CallInfo ci = P.calls[it.call];
            CellSync* cs = P.cell_sync + it.call;
            const int need = P.step_index * ci.n_done_per_step;
            for (unsigned polls = 0; ld_acquire(&cs->done) < need;) {   // bounded like every wait in this kernel: an ordering bug or a lost
#ifndef LEXP_EMU                                                        // peer must surface as an error (lexp_pm_get), never as a hung GPU
                __nanosleep(100);
#endif
                if (++polls > (1u << 25) || ((polls & 1023u) == 0 && ld_acquire(P.err_flag))) { atomicExch(P.err_flag, 1); break; }
            }
            const int ticket = atomicAdd(&cs->ticket, 1);
            Plane4 q;
            if (ticket == P.step_index * ci.n_items) {
                if (P.prop_kind) {
                    const float4 g = pm_propose(ProposeArgs{P.seed, P.cur_label, P.W, P.prop_kind, P.prop_m, P.min_disp, P.max_disp},
                                                ci.ux, ci.uy, ci.uw, ci.uh, ci.cell_id);
                    q = Plane4{g.x, g.y, g.z, g.w};
                } else q = P.planes[it.call];
                if (P.planes_out) P.planes_out[it.call] = q;
                if (ci.n_items > 1) {
                    __stcg(reinterpret_cast<float4*>(&cs->plane), make_float4(q.a, q.b, q.c, q.v));
                    __threadfence();
                    atomicExch(&cs->ready, P.step_index + 1);
                }
            } else {
                for (unsigned polls = 0; ld_acquire(&cs->ready) < P.step_index + 1;) {
#ifndef LEXP_EMU
                    __nanosleep(100);
#endif
                    if (++polls > (1u << 25) || ((polls & 1023u) == 0 && ld_acquire(P.err_flag))) { atomicExch(P.err_flag, 1); break; }
                }
                const float4 g = __ldcg(reinterpret_cast<const float4*>(&cs->plane));
                q = Plane4{g.x, g.y, g.z, g.w};
            }
            s_pl = q;
        }
        {   // zero-fill (the box filter is zero padded, GuidedFilter.h:43 BORDER_CONSTANT) by warps 1.. meanwhile
            const int total = (K * VW + 1) / 2 + K * W2 + 2 * kCH * (SW + 2 * SW2 + SW3);
            if (tid >= 32) for (int i = tid - 32; i < total; i += kThreads - 32) smem[i] = f4zero();
        }
        __syncthreads();
        pl = s_pl;
    }
    if (NAIVE) {
        if (tid == 0) naive_inverse_affine(it, pl, P.mode, s_iM);
        __syncthreads();
    }

    {   // zero-fill: the box filter is zero padded (GuidedFilter.h:43 BORDER_CONSTANT)
        const int total = (K * VW + 1) / 2 + K * W2 + 2 * kCH * (SW + 2 * SW2 + SW3);
        if (!PM) for (int i = tid; i < total; i += kThreads) smem[i] = f4zero();
        for (int v = tid; v < VHs; v += kThreads) {
            const int y = ys + v;
            s_invny[v] = 1.0f / (float)(min(y + R, fy1 - 1) - max(y - R, it.fy) + 1);  // GuidedFilter.h:324
            if (!NAIVE) {
                s_dbase[v] = __fadd_rn(__fmul_rn(pl.b, (float)y), pl.c);               // CostVolumeEnergy.h:73
                // row offset in the blocked volume, in 16-byte units (the s_Y0 slot is unused by the cost-volume energy)
                reinterpret_cast<unsigned*>(s_Y0)[v] = (unsigned)(y >> 2) * ((unsigned)P.Wb * (unsigned)P.D * 4u) + (unsigned)(y & 3);
            } else {
                // cv::warpAffine fixed-point row terms (AB_BITS = 10, round_delta = 16) for the inverse affine map of
                // StereoEnergy.h:704-729
                const double yr = (double)(y - it.fy);
                reinterpret_cast<int*>(s_dbase)[v] = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(s_iM[1], yr), s_iM[2]), 1024.0)) + 16;
                s_Y0[v] = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(s_iM[4], yr), s_iM[5]), 1024.0)) + 16;
            }
        }
    }
    __syncthreads();

    const int nChunks = (VHs + kCH - 1) / kCH;

    if (warp < kWarpsA) {
        // =========================================================================== team A
        if (NAIVE) {
            // NaiveStereoEnergy raw cost: bilinear sample of ExI[1-mode] at cv::warpAffine's fixed-point coordinates,
            // truncated L1 colour + gradient difference (StereoEnergy.h:729-741).  Straightforward (one chunk of loads
            // at a time): config 1 is the reference's small CPU-runnable case, not the throughput path.
            const int t = tid;
            const int XA = X0 + t;
            const bool colA = (t < VW) && XA >= it.fx && XA < fx1;
            const int adelta = __double2int_rn(__dmul_rn(__dmul_rn(s_iM[0], (double)(XA - it.fx)), 1024.0));
            const int bdelta = __double2int_rn(__dmul_rn(__dmul_rn(s_iM[3], (double)(XA - it.fx)), 1024.0));
            const float s255 = 1.0f / 255.0f;
            const int Wm1 = P.W - 1, Hm1 = P.H - 1;
            F4 acc = f4zero();
            int slot = 0;
            for (int c = 0; c < nChunks; c++) {
                F4 nwr[kCH];
                float pr[kCH];
                uint32_t gr[kCH];
#pragma unroll
                for (int r = 0; r < kCH; r++) {
                    const int v = c * kCH + r;
                    nwr[r] = f4zero(); pr[r] = 0.f; gr[r] = 0u;
                    if (colA && v < vReal) {
                        const int y = ys + v;
                        const int X = (reinterpret_cast<const int*>(s_dbase)[v] + adelta) >> 5, Y = (s_Y0[v] + bdelta) >> 5;
                        const int sx = X >> 5, sy = Y >> 5;
                        const float fxw = (float)(X & 31) * (1.0f / 32), fyw = (float)(Y & 31) * (1.0f / 32);
                        const int x0c = min(max(sx, 0), Wm1), x1c = min(max(sx + 1, 0), Wm1);
                        const int y0c = min(max(sy, 0), Hm1), y1c = min(max(sy + 1, 0), Hm1);
                        const float4 S00 = __ldg(P.exi_other + (size_t)y0c * P.W + x0c), S01 = __ldg(P.exi_other + (size_t)y0c * P.W + x1c);
                        const float4 S10 = __ldg(P.exi_other + (size_t)y1c * P.W + x0c), S11 = __ldg(P.exi_other + (size_t)y1c * P.W + x1c);
                        const float4 L = __ldg(P.exi_own + (size_t)y * P.W + XA);
                        const uint32_t g = __ldg(reinterpret_cast<const unsigned int*>(P.guide) + (size_t)y * P.W + XA);
                        const float w00 = __fmul_rn(1.0f - fyw, 1.0f - fxw), w01 = __fmul_rn(1.0f - fyw, fxw);
                        const float w10 = __fmul_rn(fyw, 1.0f - fxw), w11 = __fmul_rn(fyw, fxw);
                        auto bil = [&](float a, float b, float cc, float d) {  // remapBilinear: ((S00 w00 + S01 w01) + S10 w10) + S11 w11
                            return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a, w00), __fmul_rn(b, w01)), __fmul_rn(cc, w10)), __fmul_rn(d, w11));
                        };
                        const float r0 = bil(S00.x, S01.x, S10.x, S11.x), r1 = bil(S00.y, S01.y, S10.y, S11.y);
                        const float r2 = bil(S00.z, S01.z, S10.z, S11.z), r3 = bil(S00.w, S01.w, S10.w, S11.w);
                        const float col = __fadd_rn(__fadd_rn(fabsf(__fsub_rn(L.x, r0)), fabsf(__fsub_rn(L.y, r1))), fabsf(__fsub_rn(L.z, r2)));
                        const float p = __fadd_rn(fminf(P.thresh_color, col), fminf(P.thresh_gradient, fabsf(__fsub_rn(L.w, r3))));  // :737-740
                        const float ps = p * s255, nm = -8388608.0f * ps;
                        const float q0 = fmaf(__uint_as_float(__byte_perm(g, 0x4B000000u, 0x7440)), ps, nm);
                        const float q1 = fmaf(__uint_as_float(__byte_perm(g, 0x4B000000u, 0x7441)), ps, nm);
                        const float q2 = fmaf(__uint_as_float(__byte_perm(g, 0x4B000000u, 0x7442)), ps, nm);
                        nwr[r] = F4{pk2(p, q0), pk2(q1, q2)}; pr[r] = p; gr[r] = g;
                    }
                }
                produce_begin(0, c, kLinkAH);
                if (t < VW) {
                    F4* hb = hb1 + (c & 1) * kCH * SW + sidx(t);
#pragma unroll
                    for (int r = 0; r < kCH; r++) {
                        uint2* sl = ring1 + slot * VW + t;
                        const uint2 oldpg = *sl;
                        *sl = make_uint2(__float_as_uint(pr[r]), gr[r]);
                        const float po = __uint_as_float(oldpg.x);
                        const float pso = po * s255, nmo = -8388608.0f * pso;
                        const float o0 = fmaf(__uint_as_float(__byte_perm(oldpg.y, 0x4B000000u, 0x7440)), pso, nmo);
                        const float o1 = fmaf(__uint_as_float(__byte_perm(oldpg.y, 0x4B000000u, 0x7441)), pso, nmo);
                        const float o2 = fmaf(__uint_as_float(__byte_perm(oldpg.y, 0x4B000000u, 0x7442)), pso, nmo);
                        acc = f4add(acc, f4sub(nwr[r], F4{pk2(po, o0), pk2(o1, o2)}));
                        hb[r * SW] = acc;
                        slot = (slot + 1 == K) ? 0 : slot + 1;
                    }
                }
                produce_end(0, c, kLinkAH);
            }
        } else {
        const int t = tid;
        const int XA = X0 + t;
        const bool colA = (t < VW) && XA >= it.fx && XA < fx1;
        const float ax = __fmul_rn(pl.a, (float)XA);  // CostVolumeEnergy.h:76 (product rounded separately)
        const float th = P.th_col;
        const float s255 = 1.0f / 255.0f;
        // fast sampler: finite plane, MIN = 0, MAX = D-1, th >= 0, finite volume (checked at upload)
        // (finite bound on |a| W + |b| H + |c|: then a*x, b*y + c and their sum are finite for every pixel, so d is never NaN --
        //  an overflowing a*x = +inf against b*y + c = -inf would be, and the reference then returns COST_FOR_INVALID, :80)
        const bool fast = P.fast_ok && isfinite(fabsf(pl.a) * (float)P.W + fabsf(pl.b) * (float)P.H + fabsf(pl.c));
        const unsigned W4 = (unsigned)P.W * 4u;
        const int XAc = colA ? XA : it.fx;
        // blocked volume: element (d, y, x) lives at ((((y/4) * Wb + x/4) * D + d) * 4 + y%4) * 4 + x%4:
        // a 128-byte line holds 2 disparities of a 4x4 pixel block, so the rows of a gather batch share lines
        const char* vcol = reinterpret_cast<const char*>(P.vol) + ((size_t)(XAc >> 2) * P.D * 16 + (XAc & 3)) * 4;
#ifndef LEXP_EMU
        // keep the column base as ONE 64-bit pointer (otherwise: offset + uniform base, re-added per row)
        asm volatile("" : "+l"(vcol));
#endif
        const char* grow = reinterpret_cast<const char*>(P.guide) + ((size_t)ys * P.W + XAc) * 4;
        const float maxd = (float)(P.D - 1);
        F4 acc = f4zero();
        int slot = 0;
        // Gather batches of kG rows.  Exactly ONE batch of loads is in flight at any time: the hardware
        // scoreboard cannot tell older from younger loads, so a deeper register pipeline would stall on the
        // youngest load.  Order per batch: wait(batch b) -> issue(batch b+1) -> process(batch b).
        float lv0[kG], lv1[kG], lf1[kG];
        uint32_t lg[kG];
        // weight f1 and slice indices for plane disparity d
        //   fast: d < 0 -> V[0]; d >= D-1 -> (1-1) V[D-2] + 1 V[D-1] = V[D-1]; else lerp (:78-92)
        //   generic: f1 in [0,1] lerp | 2: COST_FOR_INVALID | 3: C = V[d0] | -1: outside filterRect
        auto weights = [&](float d, int& d0, int& d1) -> float {
            if (fast) {
                const float dc = fminf(fmaxf(d, 0.f), maxd);
                d0 = min(__float2int_rz(dc), P.D - 2);
                d1 = d0 + 1;
                return dc - (float)d0;
            }
            const int D0 = (int)(-P.min_disp);
            const bool lo = d < P.min_disp;                                    // :78
            const bool hi = !lo && d >= P.max_disp;                            // :79
            bool bad = !lo && !hi && (isnan(d) || isinf(d));                   // :80
            const float dd = (lo || hi || bad) ? 0.f : d;
            d0 = (int)dd + D0;                                                 // :83
            float ff = dd - floorf(dd);                                        // :85
            if (d0 + 1 >= P.D || d0 < 0) bad = true;                           // :87-90
            if (lo) { d0 = 0; ff = 3.f; }
            if (hi) { d0 = P.D - 1; ff = 3.f; }
            if (bad && !lo && !hi) { d0 = 0; ff = 2.f; }
            d1 = min(d0 + 1, P.D - 1);
            return ff;
        };
        int vi = 0;  // next virtual row to issue
        auto issue = [&]() {
#pragma unroll
            for (int j = 0; j < kG; j++) {
                lv0[j] = 0.f; lv1[j] = 0.f; lg[j] = 0u; lf1[j] = fast ? 0.f : -1.f;  // outside filterRect: zero
                if (colA && vi < vReal) {
                    int d0, d1;
                    const char* vrow = vcol + (size_t)reinterpret_cast<const unsigned*>(s_Y0)[vi] * 16;
                    if (fast) {  // the second sample is always the next disparity: 64 bytes further in the blocked layout
                        lf1[j] = weights(__fadd_rn(ax, s_dbase[vi]), d0, d1);  // :76
                        const float* p0 = reinterpret_cast<const float*>(vrow + (size_t)(unsigned)d0 * 64);
                        lv0[j] = ldg_stream(p0);
                        lv1[j] = ldg_stream(p0 + 16);
                    } else {
                        lf1[j] = weights(__fadd_rn(ax, s_dbase[vi]), d0, d1);
                        const float* p0 = reinterpret_cast<const float*>(vrow + (size_t)(unsigned)d0 * 64);
                        lv0[j] = ldg_stream(p0);
                        lv1[j] = ldg_stream(p0 + ((d1 - d0) << 4));  // d1 - d0 is 1, or 0 when the sampler clamps at D - 1
                    }
                    lg[j] = __ldg(reinterpret_cast<const unsigned int*>(grow));
                }
                vi++;
                grow += W4;
            }
        };

        issue();
        int c = 0;  // pipeline chunk
        while (c < nChunks) {
            LEXP_TRACE_LOAD_WAIT(lg[kG - 1]);  // the youngest load of the batch in flight
            float wp[kG];
            uint32_t wg[kG];
#pragma unroll
            for (int j = 0; j < kG; j++) {
                // consume point of the batch: every load must have landed before the next batch is issued
                LEXP_LOADS_LANDED("+f"(lv0[j]), "+f"(lv1[j]), "+r"(lg[j]));
                const float f1 = lf1[j];
                float C = __fadd_rn(__fmul_rn(1.0f - f1, lv0[j]), __fmul_rn(f1, lv1[j]));  // :92
                if (!fast) {
                    if (f1 > 2.5f) C = lv0[j];             // :78-79
                    else if (f1 > 1.5f) C = kCostInvalid;  // :80,:89
                }
                float p = (th < C) ? th : C;               // std::min (:96); fast & outside: min(0, th) = 0
                if (!fast && f1 < 0.f) p = 0.f;            // outside filterRect: zero padding
                wp[j] = p;
                wg[j] = lg[j];
            }
            issue();
#pragma unroll
            for (int cc = 0; cc < kG / kCH; cc++) {
                if (c < nChunks) {  // CTA-uniform
                    produce_begin(0, c, kLinkAH);
                    if (t < VW) {
                        F4* hb = hb1 + (c & 1) * kCH * SW + sidx(t);
#pragma unroll
                        for (int r = 0; r < kCH; r++) {
                            const int j = cc * kCH + r;
                            const float p = wp[j];
                            const uint32_t g = wg[j];
                            uint2* sl = ring1 + slot * VW + t;
                            const uint2 oldpg = *sl;
                            *sl = make_uint2(__float_as_uint(p), g);
                            // (2^23 + byte) * ps - 2^23 * ps = byte/255 * p   (GuidedFilter.h:62-65,151-169), for the entering row
                            // and again for the row that leaves the window (kept as {p, guide}: 8 instead of 16 bytes per pixel)
                            const float ps = p * s255, nm = -8388608.0f * ps;
                            const float q0 = fmaf(__uint_as_float(__byte_perm(g, 0x4B000000u, 0x7440)), ps, nm);
                            const float q1 = fmaf(__uint_as_float(__byte_perm(g, 0x4B000000u, 0x7441)), ps, nm);
                            const float q2 = fmaf(__uint_as_float(__byte_perm(g, 0x4B000000u, 0x7442)), ps, nm);
                            const float po = __uint_as_float(oldpg.x);
                            const float pso = po * s255, nmo = -8388608.0f * pso;
                            const float o0 = fmaf(__uint_as_float(__byte_perm(oldpg.y, 0x4B000000u, 0x7440)), pso, nmo);
                            const float o1 = fmaf(__uint_as_float(__byte_perm(oldpg.y, 0x4B000000u, 0x7441)), pso, nmo);
                            const float o2 = fmaf(__uint_as_float(__byte_perm(oldpg.y, 0x4B000000u, 0x7442)), pso, nmo);
                            const F4 nw = F4{pk2(p, q0), pk2(q1, q2)};
                            const F4 old = F4{pk2(po, o0), pk2(o1, o2)};
                            acc = f4add(acc, f4sub(nw, old));
                            hb[r * SW] = acc;  // column sum centred on row y - R
                            slot = (slot + 1 == K) ? 0 : slot + 1;
                        }
                    }
                    produce_end(0, c, kLinkAH);
                    c++;
                }
            }
        }
        }  // !NAIVE
    } else if (warp < kWarpsA + kWarpsH) {
        // =========================================================================== team H
        // out[i] = sum_{m=0}^{2R} in[i + m]: lane = (row r of the chunk, run k of 8 columns)
        const bool st2 = (warp == kWarpsA + 1);
        const int r = lane & (kCH - 1), k = lane / kCH;
        const int nruns = ((st2 ? it.ow : W2) + kRun - 1) / kRun;
        const int lin = st2 ? 2 : 0, lout = st2 ? 3 : 1;                 // input / output link
        const int nin = st2 ? kLinkCH : kLinkAH, nout = st2 ? kLinkHE : kLinkHC;
        const int vmin = st2 ? vE0 : vC0, vmax = st2 ? VHs : vC1;
        const F4* inb = st2 ? hb2 : hb1;
        F4* outb = st2 ? ho2 : ho1;
        for (int c = 0; c < nChunks; c++) {
            const int v = c * kCH + r;
            consume_begin(lin, c, nin);
            produce_begin(lout, c, nout);
            if (k < nruns && v >= vmin && v < vmax) {
                const F4* in = inb + ((c & 1) * kCH + r) * (st2 ? SW2 : SW) + 9 * k;
                F4* out = outb + ((c & 1) * kCH + r) * (st2 ? SW3 : SW2) + 9 * k;
                if (R_T > 0) {
                    F4 w[kRun - 1];
                    F4 s = in[0], s2 = in[1];  // two partial sums: halves the dependent FADD2 chain
                    w[0] = s; w[1] = s2;
#pragma unroll
                    for (int j = 2; j < 2 * R_T + 1; j++) {
                        const F4 x = in[j + (j >> 3)];
                        if (j < kRun - 1) w[j] = x;
                        if (j & 1) s2 = f4add(s2, x); else s = f4add(s, x);
                    }
                    s = f4add(s, s2);
                    out[0] = s;
#pragma unroll
                    for (int j = 1; j < kRun; j++) {
                        const int jn = 2 * R_T + j;
                        s = f4add(s, f4sub(in[jn + (jn >> 3)], w[j - 1]));
                        out[j] = s;
                    }
                } else {
                    F4 s = in[0];
                    for (int j = 1; j < K; j++) s = f4add(s, in[sidx(j)]);
                    out[0] = s;
                    for (int j = 1; j < kRun; j++) {
                        s = f4add(s, f4sub(in[sidx(2 * R + j)], in[sidx(j - 1)]));
                        out[j] = s;
                    }
                }
            }
            consume_end(lin, c, nChunks, nin);
            produce_end(lout, c, nout);
        }
    } else if (warp < kWarpsA + kWarpsH + kWarpsC) {
        // =========================================================================== team C
        const int t = tid - 32 * (kWarpsA + kWarpsH);
        const int XC = X0 + R + t;
        const bool colC = (t < W2) && XC >= it.fx && XC < fx1;
        float inv_nx = 0.f;
        if (colC) inv_nx = 1.0f / (float)(min(XC + R, fx1 - 1) - max(XC - R, it.fx) + 1);
        F4 acc = f4zero();
        int slot = 0;
        // one batch (= one chunk) of statistics loads in flight: wait(c) -> issue(c + 1) -> process(c)
        float4 sa[kCH], sb[kCH];
        float sc[kCH];
        // statistics of centre row yc = ys + v - R, issued chunk by chunk in order
        int vi = 0;
        const size_t pix0 = (size_t)(ys - R) * P.W + (colC ? XC : it.fx);  // rows above vC0 are never dereferenced
        const float4* pa = P.statA + pix0;
        const float4* pb = P.statB + pix0;
        const float* pc = P.statC + pix0;
        auto issue = [&]() {
#pragma unroll
            for (int r = 0; r < kCH; r++) {
                sa[r] = make_float4(0.f, 0.f, 0.f, 0.f); sb[r] = sa[r]; sc[r] = 0.f;
                if (colC && vi >= vC0 && vi < vC1) {
                    sa[r] = __ldg(pa);
                    sb[r] = __ldg(pb);
                    sc[r] = __ldg(pc);
                }
                vi++;
                pa += P.W; pb += P.W; pc += P.W;
            }
        };
        issue();
        for (int c = 0; c < nChunks; c++) {
            {
                LEXP_TRACE_LOAD_WAIT(__float_as_uint(sc[kCH - 1]));
                float4 ca[kCH], cb[kCH];
                float cc[kCH];
#pragma unroll
                for (int r = 0; r < kCH; r++) {
                    LEXP_LOADS_LANDED("+f"(sa[r].x), "+f"(sa[r].y), "+f"(sa[r].z), "+f"(sa[r].w), "+f"(sb[r].x), "+f"(sb[r].y),
                                      "+f"(sb[r].z), "+f"(sb[r].w), "+f"(sc[r]));
                    ca[r] = sa[r]; cb[r] = sb[r]; cc[r] = sc[r];
                }
                issue();
                consume_begin(1, c, kLinkHC);
                produce_begin(2, c, kLinkCH);
                if (t < W2) {
                    const F4* ho = ho1 + (c & 1) * kCH * SW2 + sidx(t);
                    F4* hb = hb2 + (c & 1) * kCH * SW2 + sidx(t);
#pragma unroll
                    for (int r = 0; r < kCH; r++) {
                        const int v = c * kCH + r;
                        if (v >= vC0 && v < VHs) {
                            F4 ab = f4zero();
                            if (colC && v < vC1) {
                                const float invN = inv_nx * s_invny[v - R];
                                const F4 B = ho[r * SW2];
                                float Bp, B0, B1, B2;
                                up2(B.lo, Bp, B0); up2(B.hi, B1, B2);
                                const float m0 = ca[r].x, m1 = ca[r].y, m2 = ca[r].z, i00 = ca[r].w;
                                const float i01 = cb[r].x, i02 = cb[r].y, i11 = cb[r].z, i12 = cb[r].w, i22 = cc[r];
                                const float mp = Bp * invN;                      // GuidedFilter.h:206
                                const float c0 = fmaf(B0, invN, -m0 * mp);       // :212-214
                                const float c1 = fmaf(B1, invN, -m1 * mp);
                                const float c2 = fmaf(B2, invN, -m2 * mp);
                                const float a0 = i00 * c0 + i01 * c1 + i02 * c2;  // :216-218
                                const float a1 = i01 * c0 + i11 * c1 + i12 * c2;
                                const float a2 = i02 * c0 + i12 * c1 + i22 * c2;
                                const float bb = mp - a0 * m0 - a1 * m1 - a2 * m2;  // :220
                                ab = F4{pk2(a0, a1), pk2(a2, bb)};
                            }
                            F4* sl = ring2 + slot * W2 + t;
                            const F4 old = *sl;
                            *sl = ab;
                            acc = f4add(acc, f4sub(ab, old));
                            hb[r * SW2] = acc;  // column sum centred on row y - 2R
                            slot = (slot + 1 == K) ? 0 : slot + 1;
                        }
                    }
                }
                consume_end(1, c, nChunks, kLinkHC);
                produce_end(2, c, kLinkCH);
            }
        }
    } else if (warp < kWarpsA + kWarpsH + kWarpsC + kWarpsE) {
        // =========================================================================== team E
        const int t = tid - 32 * (kWarpsA + kWarpsH + kWarpsC);
        const int XE = it.ox0 + t;
        const bool colE = t < it.ow;
        float inv_nx = 0.f;
        if (colE) inv_nx = 1.0f / (float)(min(XE + R, fx1 - 1) - max(XE - R, it.fx) + 1);
        const float s255 = 1.0f / 255.0f;
        const float xa = __fmul_rn((float)XE, pl.a);
        const float a5 = __fmul_rn(pl.a, 5.0f), b5 = __fmul_rn(pl.b, 5.0f);
        const float vz = __fmul_rn(0.0f, pl.v);
        // conservative tile-level validity: if the plane stays inside [MIN, MAX] by a margin over the whole
        // tile (+-5 px corners), every per-pixel test of StereoEnergy.h:577-610 passes and is skipped
        bool check = P.with_check != 0;
        if (check && isfinite(pl.a) && isfinite(pl.b) && isfinite(pl.c) && isfinite(pl.v)) {
            const float x0 = (float)it.ox0, x1 = (float)(it.ox0 + it.ow - 1), y0 = (float)it.oy0, y1 = (float)(it.oy0 + it.oh - 1);
            const float axl = fminf(pl.a * x0, pl.a * x1), axh = fmaxf(pl.a * x0, pl.a * x1);
            const float byl = fminf(pl.b * y0, pl.b * y1), byh = fmaxf(pl.b * y0, pl.b * y1);
            const float ext = 5.0f * (fabsf(pl.a) + fabsf(pl.b));
            const float mag = fabsf(axl) + fabsf(axh) + fabsf(byl) + fabsf(byh) + fabsf(pl.c) + ext;
            const float margin = 1e-5f * mag + 1e-30f;
            if (axl + byl + pl.c - ext - margin >= P.min_disp && axh + byh + pl.c + ext + margin <= P.max_disp) check = false;
        }
        uint32_t gq[kCH];
        float cq[kCH];   // PatchMatch phase: the pixel's current cost, prefetched with the guide (L2 only: other SMs wrote it)
        const bool pm_update = PM && P.pm_mode == 1;
        int vi = 0;
        const unsigned int* pg = reinterpret_cast<const unsigned int*>(P.guide) + (size_t)(ys - 2 * R) * P.W + (colE ? XE : it.ox0);
        auto issue = [&]() {
#pragma unroll
            for (int r = 0; r < kCH; r++) {
                gq[r] = 0u; cq[r] = 0.f;
                if (colE && vi >= vE0 && vi < VHs) {
                    gq[r] = __ldg(pg);
                    if (pm_update) cq[r] = __ldcg(P.cur_cost + (pg - reinterpret_cast<const unsigned int*>(P.guide)));
                }
                vi++;
                pg += P.W;
            }
        };
        issue();
        size_t cpix = (size_t)it.oy0 * P.W + XE;   // PatchMatch phase: pixel index of the next output row in cur_cost / cur_label
        float* orow;  // output pointer of row yq = ys + v - 2R at column XE
        long long ostride;
        if (P.out_compact) { orow = P.out + (size_t)it.compact_off + t; ostride = it.compact_stride; }
        else { orow = P.out + (size_t)it.oy0 * P.out_pitch + XE; ostride = P.out_pitch; }
        bool prior_grids_done = false;
        for (int c = 0; c < nChunks; c++) {
            {
                LEXP_TRACE_LOAD_WAIT(gq[kCH - 1]);
                uint32_t cg[kCH];
                float cc[kCH];
#pragma unroll
                for (int r = 0; r < kCH; r++) {
                    LEXP_LOADS_LANDED("+r"(gq[r]), "+f"(cq[r]));
                    cg[r] = gq[r]; cc[r] = cq[r];
                }
                issue();
                consume_begin(3, c, kLinkHE);
                if (colE) {
                    const F4* ho = ho2 + (c & 1) * kCH * SW3 + sidx(t);
#pragma unroll
                    for (int r = 0; r < kCH; r++) {
                        const int v = c * kCH + r;
                        if (v >= vE0 && v < VHs) {
                            const F4 S = ho[r * SW3];
                            float S0, S1, S2, Sb;
                            up2(S.lo, S0, S1); up2(S.hi, S2, Sb);
                            const uint32_t g = cg[r];
                            const float i0 = __uint_as_float(__byte_perm(g, 0x4B000000u, 0x7440)) - 8388608.0f;
                            const float i1 = __uint_as_float(__byte_perm(g, 0x4B000000u, 0x7441)) - 8388608.0f;
                            const float i2 = __uint_as_float(__byte_perm(g, 0x4B000000u, 0x7442)) - 8388608.0f;
                            const float dot = S0 * i0 + S1 * i1 + S2 * i2;
                            float q = fmaf(dot, s255, Sb) * (inv_nx * s_invny[v - 2 * R]);  // GuidedFilter.h:243
                            if (check) {  // StereoEnergy.h:577-610
                                const int yq = ys + v - 2 * R;
                                const float yb = __fmul_rn((float)yq, pl.b);
                                float ds = __fadd_rn(__fadd_rn(xa, yb), pl.c);
                                if (!(it.flags & 1)) ds = __fadd_rn(ds, vz);  // channelSum's 4th term (0 * v)
                                const float lo = P.min_disp, hi = P.max_disp;
                                const float dpp = __fadd_rn(__fadd_rn(ds, a5), b5), dpm = __fsub_rn(__fadd_rn(ds, a5), b5);
                                const float dmp = __fadd_rn(__fsub_rn(ds, a5), b5), dmm = __fsub_rn(__fsub_rn(ds, a5), b5);
                                const bool ok = ds >= lo && ds <= hi && dpp >= lo && dpp <= hi && dpm >= lo && dpm <= hi &&
                                                dmp >= lo && dmp <= hi && dmm >= lo && dmm <= hi;
                                if (!ok) q = kCostInvalid;  // CostVolumeEnergy.h:180-182
                            }
                            if (PM) {
                                // `updateMask = subCurrentCost > subProposalCost; copyTo; setTo` (FastGCStereo.h:56-60); NaN never
                                // updates.  Initialisation (pm_mode 2, :105-113) writes unconditionally.  Ordering against the cell's
                                // previous steps is by its completion counter (prologue), not by griddepcontrol.wait.
                                if (P.pm_mode == 2 || cc[r] > q) {
                                    P.cur_cost[cpix] = q;
                                    P.cur_label[cpix] = make_float4(pl.a, pl.b, pl.c, pl.v);
                                    for (int p = 1; p < P.n_copies; p++) {   // the peers' copies: plain stores over NVLink
                                        P.copy_cost[p][cpix] = q;
                                        P.copy_label[p][cpix] = make_float4(pl.a, pl.b, pl.c, pl.v);
                                    }
                                }
                                cpix += (size_t)P.W;
                            } else {
                                if (!prior_grids_done) {  // write-after-write order against the previous launch of the stream
#ifndef LEXP_EMU
                                    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
                                    prior_grids_done = true;
                                }
                                *orow = q;
                                orow += ostride;
                            }
                        }
                    }
                }
                consume_end(3, c, nChunks, kLinkHE);
            }
        }
        if (PM) {   // this work item's part of the proposal step is done: publish (release) to the cell's counter
            // the peers' copies only have to be complete when the group's epoch is published (last step of the group): the steps of a
            // cell in between run on this GPU and read its own copy, so a device-scope fence orders them (a system-scope fence waits for
            // the NVLink round trip of every remote store -- microseconds on the per-step critical path)
            if (P.n_copies > 1 && P.publish_epoch) __threadfence_system(); else __threadfence();
            __syncwarp();
            if (lane == 0) {
                atomicAdd(&P.cell_sync[it.call].done, 1);
                if (P.publish_epoch) {
                    // last step of a group on the multi-GPU cell shard: the warp that completes the launch tells every peer that this
                    // rank's updates of the group are in place (all stores above were fenced system-wide before their increments)
                    const int fin = atomicAdd(P.launch_done, 1) + 1;
                    if (fin == (int)gridDim.x * kWarpsE) {
                        __threadfence_system();
                        const int e = *P.epoch_base + P.publish_epoch;
                        for (int p = 0; p < P.n_copies; p++) st_release_sys(P.copy_flags[p] + P.my_rank, e);
                    }
                }
            }
        }
    }
#if LEXP_TRACE
    if (lane == 0 && P.trace) {
        long long* o = P.trace + ((size_t)blockIdx.x * (kThreads / 32) + warp) * 4;
        o[0] = (unsigned)clock64() - tr_t0; o[1] = tr_wait_in; o[2] = tr_wait_out; o[3] = nChunks | ((long long)tr_wait_ld << 32);
    }
#endif
}

// ---------------------------------------------------------------------------------------------
// K0: one-time guided-filter statistics, GuidedFilter.h:58-102 with T = double.
// Window sums of the 8-bit guide and of its pairwise products are integers: they are summed
// exactly in int32, and only the final normalisation / 3x3 inversion runs in FP64.
// ---------------------------------------------------------------------------------------------
__global__ void lexp_stats_rowsum(const uchar4* __restrict__ guide, int* __restrict__ rs, int H, int W, int R) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    int s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    const int xa = max(x - R, 0), xb = min(x + R, W - 1);
    for (int xx = xa; xx <= xb; xx++) {
        const uchar4 g = guide[(size_t)y * W + xx];
        const int c0 = g.x, c1 = g.y, c2 = g.z;
        s[0] += c0; s[1] += c1; s[2] += c2;
        s[3] += c0 * c0; s[4] += c0 * c1; s[5] += c0 * c2; s[6] += c1 * c1; s[7] += c1 * c2; s[8] += c2 * c2;
    }
    const size_t HW = (size_t)H * W;
#pragma unroll
    for (int k = 0; k < 9; k++) rs[k * HW + (size_t)y * W + x] = s[k];
}

__global__ void lexp_stats_finish(const int* __restrict__ rs, float4* __restrict__ statA, float4* __restrict__ statB,
                                  float* __restrict__ statC, int H, int W, int R, double eps) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    const size_t HW = (size_t)H * W;
    long long s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    const int ya = max(y - R, 0), yb = min(y + R, H - 1);
    for (int yy = ya; yy <= yb; yy++) {
#pragma unroll
        for (int k = 0; k < 9; k++) s[k] += rs[k * HW + (size_t)yy * W + x];
    }
    const double N = (double)((min(x + R, W - 1) - max(x - R, 0) + 1) * (yb - ya + 1));  // :69
    const double sc = 1.0 / 255.0;
    const double m0 = s[0] * sc / N, m1 = s[1] * sc / N, m2 = s[2] * sc / N;             // :70-72
    const double sc2 = sc * sc;
    const double v00 = s[3] * sc2 / N - m0 * m0 + eps, v01 = s[4] * sc2 / N - m0 * m1, v02 = s[5] * sc2 / N - m0 * m2;  // :79-84
    const double v11 = s[6] * sc2 / N - m1 * m1 + eps, v12 = s[7] * sc2 / N - m1 * m2, v22 = s[8] * sc2 / N - m2 * m2 + eps;
    double i00 = v11 * v22 - v12 * v12, i01 = v12 * v02 - v01 * v22, i02 = v01 * v12 - v11 * v02;  // :87-92
    double i11 = v00 * v22 - v02 * v02, i12 = v02 * v01 - v00 * v12, i22 = v00 * v11 - v01 * v01;
    const double det = i00 * v00 + i01 * v01 + i02 * v02;                                          // :94
    const size_t p = (size_t)y * W + x;
    statA[p] = make_float4((float)m0, (float)m1, (float)m2, (float)(i00 / det));
    statB[p] = make_float4((float)(i01 / det), (float)(i02 / det), (float)(i11 / det), (float)(i12 / det));
    statC[p] = (float)(i22 / det);
}

// One-time re-layout of the cost volume (the input format float[D][H][W], README.md:85-91, is fixed only at the API):
// dst[((((y/4) * Wb + x/4) * D + d) * 4 + y%4) * 4 + x%4] = src[d][y][x].  All disparities of a 4x4 pixel block are
// contiguous (64 B per disparity), so the two samples (d0, d0+1) of a pixel, of its neighbours in x AND of the next
// rows of the streaming gather share 128-byte lines / DRAM pages instead of being scattered over ndisp slices
// H*W*4 bytes apart.   grid = (ceil(W/32), ceil(H/4), ceil(D/8)), block = 256
// Volume preparation fused into the same pass (main.cpp:146-199, 353-370): `transform` selects which source column the element
// (d, y, x) is read from --
//   0 plain; 1 fillOutOfView(vol, 0): x' = max(x, d); 2 fillOutOfView(vol, 1): x' = min(x, W - 1 - d);
//   3 the RIGHT view derived from the (unfilled) LEFT volume: fillOutOfView(convertVolumeL2R(fillOutOfView(volL, 0)), 1), i.e.
//     volR[d][y][x] = volL[d][y][min(x + d, W - 1)]  (margin = 0, main.cpp:363).
// `src` holds the disparities [d_lo, d_lo + nd) of the caller's volume (a slab of the host upload, or the whole volume).
__global__ void lexp_relayout_volume(const float* __restrict__ src, float* __restrict__ dst, int D, int H, int W, int Wb, int d_lo, int nd,
                                     int transform) {
    __shared__ float tile[8][4][33];  // [d][row][x]
    const int x0 = blockIdx.x * 32, y0 = blockIdx.y * 4, d0 = blockIdx.z * 8;   // d0: relative to the slab
    for (int i = threadIdx.x; i < 8 * 4 * 32; i += 256) {
        const int xx = i & 31, rr = (i >> 5) & 3, dd = i >> 7;
        const int x = x0 + xx, y = y0 + rr, ds = d0 + dd, d = d_lo + ds;
        float v = 0.0f;
        if (ds < nd && y < H && x < W) {
            int xs = x;
            if (transform == 1) xs = max(x, min(d, W - 1));
            else if (transform == 2) xs = min(x, max(W - 1 - d, 0));
            else if (transform == 3) xs = min(x + d, W - 1);
            v = src[((size_t)ds * H + y) * W + xs];
        }
        tile[dd][rr][xx] = v;
    }
    __syncthreads();
    // consecutive threads write consecutive floats of the destination: [xb 8][d 8][row 4][px 4]
    for (int i = threadIdx.x; i < 8 * 8 * 16; i += 256) {
        const int q = i & 3, rr = (i >> 2) & 3, dd = (i >> 4) & 7, xb = i >> 7;
        const int d = d_lo + d0 + dd;
        if (d0 + dd < nd && (x0 >> 2) + xb < Wb)
            dst[((((size_t)blockIdx.y * Wb + (x0 >> 2) + xb) * D + d) * 4 + rr) * 4 + q] = tile[dd][rr][xb * 4 + q];
    }
}

// NaiveStereoEnergy constructor (StereoEnergy.h:647-662): ExI = merge(I * (1 - alpha), alpha * Sobel_x(gray)), with
// cvtColor(BGR2GRAY) = (B*0.114f + G*0.587f) + R*0.299f and Sobel(dx=1, ksize=1, scale=0.5, BORDER_REPLICATE) in float.
__global__ void lexp_build_exi(const uchar4* __restrict__ guide, float4* __restrict__ exi, int H, int W, float s_col, float alpha) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    auto gray = [&](int xx) {
        const uchar4 g = guide[(size_t)y * W + min(max(xx, 0), W - 1)];
        return __fadd_rn(__fadd_rn(__fmul_rn((float)g.x, 0.114f), __fmul_rn((float)g.y, 0.587f)), __fmul_rn((float)g.z, 0.299f));
    };
    const uchar4 g = guide[(size_t)y * W + x];
    const float gx = __fmul_rn(__fsub_rn(gray(x + 1), gray(x - 1)), 0.5f);
    exi[(size_t)y * W + x] = make_float4(__fmul_rn((float)g.x, s_col), __fmul_rn((float)g.y, s_col), __fmul_rn((float)g.z, s_col),
                                         __fmul_rn(gx, alpha));
}

// upload-time scan: does the cost volume hold any NaN / Inf?  (the fast sampler multiplies by 0 weights)
__global__ void lexp_scan_nonfinite(const float* __restrict__ vol, size_t n, int* __restrict__ flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    bool bad = false;
    for (; i < n; i += stride) bad |= !isfinite(vol[i]);
#ifndef LEXP_EMU
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
#else
    if (bad) atomicOr(flag, 1);  // emulated threads do not run in warp lock-step
#endif
}

__global__ void lexp_add_i32(int* p, int delta) { *p += delta; }

__global__ void lexp_fill_f32(float* __restrict__ dst, size_t n, float v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) dst[i] = v;
}

// planar float[9][H][W] view of the statistics (lexp_get_stats)
__global__ void lexp_stats_unpack(const float4* __restrict__ statA, const float4* __restrict__ statB, const float* __restrict__ statC,
                                  float* __restrict__ out9, size_t HW) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const float4 a = statA[p], b = statB[p];
    out9[p] = a.x; out9[HW + p] = a.y; out9[2 * HW + p] = a.z; out9[3 * HW + p] = a.w;
    out9[4 * HW + p] = b.x; out9[5 * HW + p] = b.y; out9[6 * HW + p] = b.z; out9[7 * HW + p] = b.w;
    out9[8 * HW + p] = statC[p];
}

}  // namespace lexp
