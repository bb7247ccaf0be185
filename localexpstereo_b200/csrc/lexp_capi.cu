// lexp_capi.cu -- host side of the C-ABI declared in include/lexp_cuda.h.
// Owns device memory (guide, statistics, volumes, plans), tiles calls into CTA work items and
// launches the sm_100a kernels of lexp_kernels.cuh.  No CPU compute fallback exists here.
#include "../../include/lexp_cuda.h"
#include "lexp_kernels.cuh"
#include "lexp_gc.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <array>
#include <atomic>
#include <chrono>
#include <thread>
#include <climits>
#include <linux/futex.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <condition_variable>
#include <map>
#include <memory>
#include <set>
#include <mutex>
#include <string>
#include <vector>

using namespace lexp;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

// kernel launch: CUDA's <<<>>> for nvcc; the same call goes to the fiber scheduler of tests/emu/ when the file is compiled
// with g++ -DLEXP_EMU into the CPU test emulator (test infrastructure only, never part of liblexp_cuda.so)
#ifndef LEXP_EMU
#define LEXP_LAUNCH(kern, grid, block, smem, stream, ...) kern<<<grid, block, smem, stream>>>(__VA_ARGS__)
#else
#define LEXP_LAUNCH(kern, grid, block, smem, stream, ...) emu::launch(kern, dim3(grid), dim3(block), (size_t)(smem), __VA_ARGS__)
#endif

#define LEXP_CUDA(expr)                                                                                  \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            std::string m__ = std::string(#expr) + ": " + cudaGetErrorString(e__);                      \
            cudaGetLastError(); /* reset: a launch check after this failure must not report it again */  \
            return fail(LEXP_ERR_CUDA, m__);                                                             \
        }                                                                                                \
    } while (0)

// futex on a 32-bit word: block while *addr == expected / wake every waiter (the combiner's followers sleep in the kernel instead of
// spinning: with 128 OpenMP threads on 128 hardware threads, polling starves the one thread that stages and launches the batch)
void futex_wait(std::atomic<int>* addr, int expected) { syscall(SYS_futex, reinterpret_cast<int*>(addr), FUTEX_WAIT_PRIVATE, expected, nullptr, nullptr, 0); }
void futex_wake_all(std::atomic<int>* addr) { syscall(SYS_futex, reinterpret_cast<int*>(addr), FUTEX_WAKE_PRIVATE, INT_MAX, nullptr, nullptr, 0); }
inline void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
}

int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return (s && *s) ? atoi(s) : dflt;
}

}  // namespace

struct lexp_plan {
    lexp_ctx* ctx = nullptr;
    int ncalls = 0, nitems = 0, max_vw = 0;
    size_t smem = 0;  // dynamic shared memory of the largest item
    std::vector<lexp_rect> filt, targ;
    std::vector<int> compact_off;  // per call
    int64_t sum_f = 0, sum_s = 0, alg_bytes = 0;
    Item* d_items = nullptr;
    std::vector<Item> h_items;    // host copy (the combiner of concurrent lexp_eval_cell calls concatenates them)
    Plane4* d_planes = nullptr;   // staging for host planes
    float* d_compact = nullptr;   // lazily allocated compact output (host path)
    float* h_compact = nullptr;   // pinned
    // PatchMatch phase (lexp_plan_set_units / lexp_plan_pm_step)
    CallInfo* d_calls = nullptr;  // [ncalls] unitRegion, signals per step, cell id
    long long sync_off = -1;           // byte offset in the context's synchronisation arena of CellSync[ncalls + 1]: per-call completion
                                       // counters / proposal hand-over, then the completion counter of the group's last launch
    std::vector<int> items_per_call;
    // graph-cut move (lexp_plan_gc_step): region + scratch offset of every call
    GcCell* d_gc_cells = nullptr;
    long long gc_nodes = 0;       // sum of the calls' targetRect areas
    int gc_max_nodes = 0;         // largest cell: above the context's gc_big_nodes the move runs as phase kernels over all SMs
    GcBlock* d_gc_blocks = nullptr;   // block map of the phase kernels (lexp_gc.cuh)
    int gc_nblocks = 0;
    char* d_gc_ctl = nullptr;     // int done[ncalls], active[ncalls], g_flags[2] (padded to 8 bytes), double konst_part[nblocks], sink_part[nblocks]
};

struct lexp_ctx {
    lexp_params p{};
    int R = 0;
    cudaStream_t stream = nullptr;
    uchar4* d_guide[2] = {nullptr, nullptr};
    float4* d_statA[2] = {nullptr, nullptr};
    float4* d_statB[2] = {nullptr, nullptr};
    float* d_statC[2] = {nullptr, nullptr};
    char* d_gs[2] = {nullptr, nullptr};   // backing allocation of guide + statistics
    float4* d_exi[2] = {nullptr, nullptr}; // NaiveStereoEnergy: ExI planes
    size_t gs_bytes = 0;
    size_t persist_bytes = 0;             // L2 set-aside for persisting accesses (0: unsupported)
    int persist_mode = -1;                // view whose window is currently installed on the stream
    float* d_vol[2] = {nullptr, nullptr};   // blocked copy float[Hb][Wb][D][4][4] (owned)
    float* d_cur_cost[2] = {nullptr, nullptr};     // PatchMatch phase: currentCost_[mode]   float [H][W]
    float4* d_cur_label[2] = {nullptr, nullptr};   //                   currentLabeling_[mode] Plane[H][W]
    char* d_sync_arena = nullptr;                  // CellSync records of all plans (zeroed by lexp_pm_reset_sync once per iteration)
    size_t sync_cap = 0, sync_used = 0;
    int* d_flags[2] = {nullptr, nullptr};          // epoch flags int[kMaxPeers] of the multi-GPU cell shard (peers store into them);
                                                   // d_flags[m][kMaxPeers] is this rank's epoch base (lexp_pm_advance_epoch)
    struct Peers {                                 // copies of the state the epilogue writes: entry 0 = this context's own
        int world = 1, rank = 0;
        float* cost[kMaxPeers] = {};
        float4* label[kMaxPeers] = {};
        int* flags[kMaxPeers] = {};
        void* ipc_opened[3 * kMaxPeers] = {};      // cudaIpcOpenMemHandle mappings to close
        int n_opened = 0;
    } peers[2];
    // pairwise terms / graph-cut move (lexp_gc.cuh; SURVEY.md section 8 f-2, f-3)
    float sm_lambda = 1.0f, sm_omega = 10.0f, sm_th = 1.0f, sm_eps = 0.01f;   // Parameters of main.cpp:73 (paramsGF) / StereoEnergy.h:26-36
    float4* d_coef[2] = {nullptr, nullptr};        // forward smoothness coefficients {GE, EG, LG, GG} per pixel (smoothnessCoeff[mode])
    bool coef_valid[2] = {false, false};
    float* d_prop_cost[2] = {nullptr, nullptr};    // proposalCost image of the graph-cut steps (FastGCStereo.h:25)
    float* d_gc_scratch = nullptr;                 // kGcWords planes of gc_scratch_nodes words: the residual network of a group's moves
    long long gc_scratch_nodes = 0;
    int gc_threads = 1024, gc_relabel_every = 24, gc_max_rounds = 1 << 22;
    int gc_big_nodes = 32768;                      // cells with more nodes run as phase kernels over all SMs (LEXP_GC_BIG_NODES)
    int* h_gc_flags = nullptr;                     // pinned: the two decision flags of the phase path
    int64_t launches = 0;
    std::mutex mu;
    int tile_oh = 128;    // max output rows per work item
    bool tile_oh_fixed = false;  // LEXP_TILE_OH given: no per-plan search
    int num_sms = 148;
    int ctas_per_sm = kMinCtas;  // CTA slots per SM the planner fills (LEXP_CTAS_PER_SM)
    bool pdl = false;            // launch with programmatic stream serialization (builds with -DLEXP_PDL=1; LEXP_PDL_OFF=1 disables)
    bool overlap = false;        // lexp_set_overlap: launches with device-resident planes may overlap their predecessors
    bool chain_ok = false;       // the last operation this context put on its stream was a launch of lexp_fused_kernel: only then may the
                                 // next launch carry the programmatic-serialization attribute.  After a memcpy / memset (plane upload, counter
                                 // reset, state upload) the next launch is an ordinary one: a kernel launched with the attribute right after a
                                 // copy was observed reading the copy's destination before the copy had landed
    size_t smem_cap = 0;         // upper bound on a work item's dynamic shared memory, 0: none (LEXP_SMEM_CAP)
    size_t smem_limit = 0;
    size_t window_max = 0;
    bool smem_configured[2] = {false, false};
    bool own_stream = true;
    bool vol_finite[2] = {false, false};
    // single-cell plans of lexp_eval_cell, keyed by (filterRect, targetRect): the unchanged reference loop calls the
    // virtual again and again with the same rects (LayerManager.h:14-24), so the tiling / device upload is done once
    std::mutex cache_mu;
    std::map<std::array<int, 8>, lexp_plan*> cell_plans;
    // every live plan of this context (user plans and cached cell plans): lexp_destroy releases their device memory and
    // orphans them (ctx = nullptr), so that a plan handle that outlives its context stays safe to destroy
    std::mutex plans_mu;
    std::set<lexp_plan*> live_plans;
    // Combining of CONCURRENT lexp_eval_cell calls.  The unchanged reference loop issues one blocking call per cell from an OpenMP
    // `parallel for` over the cells of a disjoint group (FastGCStereo.h:30-49).  Every call queues a request; the first thread to find
    // no leader becomes one: it gives the other threads of the group a few microseconds to arrive (they all return from the previous
    // proposal at about the same time), then evaluates the whole queue with ONE batched launch (the cached work items of the cells
    // concatenated -- same items, bit-identical results) whose compact tiles land in a mapped pinned buffer; every caller then copies
    // its own tile into its cost image, in parallel.  Waiting threads poll their own request (no condition variable: with 128 OpenMP
    // threads one notify_all per batch cost more than the kernel); leadership is handed to a queued request when a batch is done.
    struct CellReq {
        int mode, with_check;
        lexp_plan* pl;
        lexp_plane plane;
        float* base;
        ptrdiff_t step_bytes;
        int status = LEXP_OK;
        std::string err;
        const float* tile = nullptr;           // where the leader's batch put this call's compact tile (pinned host memory)
        std::atomic<int>* copies_left = nullptr;   // the batch's count of tiles not yet copied out: the buffer is reused after it hits 0
        std::atomic<int> state{0};             // 0 queued, 1 done (tile ready / error), 2 lead the next batch
    };
    std::mutex comb_mu;
    std::vector<CellReq*> comb_q;
    std::atomic<int> comb_n{0};    // = comb_q.size(), readable without the mutex (the leader's collection window polls it)
    std::atomic<int> comb_gen{0};  // bumped (and futex-woken) whenever requests change state: what waiting callers sleep on
    bool comb_leader = false;      // a leader is collecting / running a batch
    bool combine = true;           // LEXP_COMBINE=0: every call on its own (the round-1 behaviour)
    int comb_window_us = 30;       // LEXP_COMBINE_WINDOW_US: how long a leader waits for the queue to stop growing
    std::atomic<size_t> comb_seen{1};   // largest batch so far: a leader stops collecting as soon as that many calls are queued
    struct CombBuf {               // staging of one batch: pinned (mapped) host memory, plus device copies of items / planes
        Item* h_items = nullptr; Plane4* h_planes = nullptr; float* h_out = nullptr;
        Item* d_items = nullptr; Plane4* d_planes = nullptr; float* d_out = nullptr;   // d_out: device address of h_out (zero-copy)
        size_t items_cap = 0, planes_cap = 0, out_cap = 0;
        std::atomic<int> copies_left{0};
    } cb[2];
    int cb_next = 0;
    int64_t combined_batches = 0, combined_calls = 0;
#if LEXP_TRACE
    long long* d_trace = nullptr;
    size_t trace_cap = 0;
#endif
};

namespace {

#if LEXP_TRACE
// diagnosis build: per-team averages of {total cycles, waiting for input, waiting for an output buffer} of one launch
void report_trace(lexp_ctx* c, int nitems) {
    constexpr int NW = kThreads / 32;
    std::vector<long long> h((size_t)nitems * NW * 4);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return;
    if (cudaMemcpy(h.data(), c->d_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return;
    const char* names[5] = {"A", "H1", "H2", "C", "E"};
    const int first[6] = {0, kWarpsA, kWarpsA + 1, kWarpsA + kWarpsH, kWarpsA + kWarpsH + kWarpsC, NW};
    const char* path = getenv("LEXP_TRACE_FILE");
    FILE* f = path ? fopen(path, "a") : stderr;
    if (!f) return;
    double chunks = 0;
    for (int i = 0; i < nitems; i++) chunks += (double)(h[(size_t)i * NW * 4 + 3] & 0xffffffffLL);
    fprintf(f, "launch items=%d chunks/item=%.1f", nitems, chunks / nitems);
    for (int t = 0; t < 5; t++) {
        double tot = 0, win = 0, wout = 0, wld = 0;
        long long n = 0;
        for (int i = 0; i < nitems; i++)
            for (int w = first[t]; w < first[t + 1]; w++) {
                const long long* o = &h[((size_t)i * NW + w) * 4];
                tot += (double)o[0]; win += (double)o[1]; wout += (double)o[2]; wld += (double)((unsigned long long)o[3] >> 32); n++;
            }
        fprintf(f, " | %s total %.0f wait_in %.0f wait_out %.0f busy %.0f wait_ld %.0f", names[t], tot / n, win / n, wout / n,
                (tot - win - wout) / n, wld / n);
    }
    fprintf(f, "\n");
    if (path) fclose(f);
}
#endif

template <int R_T, bool NAIVE, bool PM>
int launch_fused_t(lexp_ctx* c, const KParams& kp_in, int nitems, size_t smem, bool allow_pdl) {
    KParams kp = kp_in;
#if LEXP_TRACE
    {
        const size_t need = (size_t)nitems * (kThreads / 32) * 4;
        if (need > c->trace_cap) {
            cudaStreamSynchronize(c->stream);
            cudaFree(c->d_trace); c->d_trace = nullptr; c->trace_cap = 0;
            LEXP_CUDA(cudaMalloc(&c->d_trace, 2 * need * sizeof(long long)));
            c->trace_cap = 2 * need;
        }
        kp.trace = c->d_trace;
    }
#endif
    auto kern = lexp_fused_kernel<R_T, NAIVE, PM>;
    if (!c->smem_configured[PM]) {  // one R instantiation per context (and one more for the PatchMatch phase)
        LEXP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_limit));
        c->smem_configured[PM] = true;
    }
#if LEXP_PDL && !defined(LEXP_EMU)
    if (c->pdl && allow_pdl && c->chain_ok) {  // programmatic dependent launch: see LEXP_PDL in lexp_kernels.cuh
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)nitems); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = c->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        LEXP_CUDA(cudaLaunchKernelEx(&cfg, kern, kp));
    } else
#endif
    LEXP_LAUNCH(kern, nitems, kThreads, smem, c->stream, kp);
    LEXP_CUDA(cudaGetLastError());
    c->launches++;
    c->chain_ok = true;
#if LEXP_TRACE
    report_trace(c, nitems);
#endif
    return LEXP_OK;
}

int launch_fused(lexp_ctx* c, const KParams& kp, int nitems, size_t smem, bool allow_pdl = true) {
    if (smem > c->smem_limit) return fail(LEXP_ERR_INVALID, "tile needs more shared memory than the device offers");
    if (c->p.energy_kind == 1) {
        switch (c->R) {
            case 10: return launch_fused_t<10, true, false>(c, kp, nitems, smem, allow_pdl);
            default: return launch_fused_t<0, true, false>(c, kp, nitems, smem, allow_pdl);
        }
    }
    if (kp.pm_mode) {   // PatchMatch phase: proposal prologue + fused update epilogue compiled in
        switch (c->R) {
            case 10: return launch_fused_t<10, false, true>(c, kp, nitems, smem, allow_pdl);
            case 16: return launch_fused_t<16, false, true>(c, kp, nitems, smem, allow_pdl);
            default: return launch_fused_t<0, false, true>(c, kp, nitems, smem, allow_pdl);
        }
    }
    switch (c->R) {
        case 10: return launch_fused_t<10, false, false>(c, kp, nitems, smem, allow_pdl);
        case 16: return launch_fused_t<16, false, false>(c, kp, nitems, smem, allow_pdl);
        default: return launch_fused_t<0, false, false>(c, kp, nitems, smem, allow_pdl);
    }
}

void release_plan_memory(lexp_plan* pl) {
    cudaFree(pl->d_items); pl->d_items = nullptr;
    cudaFree(pl->d_planes); pl->d_planes = nullptr;
    cudaFree(pl->d_compact); pl->d_compact = nullptr;
    if (pl->h_compact) { cudaFreeHost(pl->h_compact); pl->h_compact = nullptr; }
    cudaFree(pl->d_calls); pl->d_calls = nullptr;
    cudaFree(pl->d_gc_cells); pl->d_gc_cells = nullptr;
    cudaFree(pl->d_gc_blocks); pl->d_gc_blocks = nullptr;
    cudaFree(pl->d_gc_ctl); pl->d_gc_ctl = nullptr;
}

// compact device buffer + pinned host mirror of the staged host paths: both or neither
int ensure_compact(lexp_plan* pl, size_t nout) {
    if (pl->d_compact && pl->h_compact) return LEXP_OK;
    cudaFree(pl->d_compact); pl->d_compact = nullptr;
    if (pl->h_compact) { cudaFreeHost(pl->h_compact); pl->h_compact = nullptr; }
    cudaError_t e = cudaMalloc(&pl->d_compact, nout * sizeof(float));
    if (e == cudaSuccess) e = cudaHostAlloc(&pl->h_compact, nout * sizeof(float), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaFree(pl->d_compact); pl->d_compact = nullptr; pl->h_compact = nullptr;
        cudaGetLastError();
        return fail(LEXP_ERR_NOMEM, std::string("staging buffers of the host path: ") + cudaGetErrorString(e));
    }
    return LEXP_OK;
}

// Zero-copy output is taken only for host memory that CUDA itself knows as page-locked (cudaHostRegister / cudaHostAlloc) over the WHOLE
// range [p, p + bytes): first and last byte must both be registered host memory with a device alias at the same offset.  A bare
// cudaHostGetDevicePointer is not enough: it also succeeds for a buffer that merely starts inside somebody else's registration (the
// kernel then writes past the end of the mapping: an illegal address), and on systems where the GPU can address pageable memory
// (HMM / ATS) for memory nobody registered at all.  Returns the device alias of p, or nullptr (= take the staged path).
void* mapped_alias(void* p, size_t bytes) {
#ifdef LEXP_EMU
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, p, 0) != cudaSuccess || !d) return nullptr;
    void* e = nullptr;
    if (bytes > 1 && (cudaHostGetDevicePointer(&e, static_cast<char*>(p) + bytes - 1, 0) != cudaSuccess || !e)) return nullptr;
    return d;
#else
    cudaPointerAttributes a0{}, a1{};
    if (cudaPointerGetAttributes(&a0, p) != cudaSuccess || a0.type != cudaMemoryTypeHost || !a0.devicePointer) { cudaGetLastError(); return nullptr; }
    if (bytes > 1) {
        char* last = static_cast<char*>(p) + bytes - 1;
        if (cudaPointerGetAttributes(&a1, last) != cudaSuccess || a1.type != cudaMemoryTypeHost || !a1.devicePointer ||
            static_cast<char*>(a1.devicePointer) - static_cast<char*>(a0.devicePointer) != (ptrdiff_t)(bytes - 1)) { cudaGetLastError(); return nullptr; }
    }
    return a0.devicePointer;
#endif
}

// p lies in page-locked host memory that CUDA knows of (cudaHostRegister / cudaHostAlloc)
bool registered_host(const void* p) {
#ifdef LEXP_EMU
    void* d = nullptr;
    return cudaHostGetDevicePointer(&d, const_cast<void*>(p), 0) == cudaSuccess && d;
#else
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
#endif
}

int check_rects(const lexp_ctx* c, const lexp_rect& f, const lexp_rect& t) {
    const int H = c->p.height, W = c->p.width;
    if (f.width <= 0 || f.height <= 0 || t.width <= 0 || t.height <= 0) return fail(LEXP_ERR_INVALID, "empty rect");
    if (f.x < 0 || f.y < 0 || f.x + f.width > W || f.y + f.height > H) return fail(LEXP_ERR_INVALID, "filterRect outside image");
    if (t.x < f.x || t.y < f.y || t.x + t.width > f.x + f.width || t.y + t.height > f.y + f.height)
        return fail(LEXP_ERR_INVALID, "targetRect not inside filterRect");
    return LEXP_OK;
}

struct PmArgs {   // PatchMatch phase (lexp_plan_pm_step); nullptr = plain unary evaluation
    int pm_mode, prop_kind, prop_m, step_index;
    unsigned long long seed;
    Plane4* planes_out;
    int publish_epoch;
    int wait_epochs[kMaxPeers];
    unsigned wait_mask;
};

// overlap_ok: the launch may start while the previous launches of the stream are still running (programmatic dependent launch).
// Only when nothing this launch reads at its start was produced by the work right before it in the stream: never after a
// host-to-device copy of its planes (measured: such a launch can read the plane array before the copy has landed), and for
// device-resident planes only if the caller opted in (lexp_set_overlap).
int run_plan(lexp_ctx* c, lexp_plan* pl, int mode, const Plane4* d_planes, float* d_out, long long pitch, int compact,
             int with_check, const PmArgs* pm = nullptr, bool overlap_ok = false) {
    if (mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "mode must be 0 or 1");
    if (c->p.energy_kind == 1) {
        if (!c->d_exi[0] || !c->d_exi[1]) return fail(LEXP_ERR_STATE, "NaiveStereoEnergy needs the images of both views");
    } else if (!c->d_guide[mode] || !c->d_vol[mode]) return fail(LEXP_ERR_STATE, "image / volume of this view not set");
    if (c->persist_bytes && c->persist_mode != mode) {
        // keep the plane-independent inputs (statistics, guide) resident in L2 across the K steps of a group;
        // (the cost-volume gathers are plain read-only loads; see profiles/r1_experiments.md)
        cudaStreamAttrValue av{};
        av.accessPolicyWindow.base_ptr = c->d_gs[mode];
        // default: pin a prefix [statA | statC | guide | ..] of exactly the set-aside size with hit ratio 1 (measured 1 %
        // better than LEXP_L2_PERSIST=2: the whole allocation with a fractional hit ratio)
        const bool prefix = env_int("LEXP_L2_PERSIST", 1) != 2;
        av.accessPolicyWindow.num_bytes = prefix ? std::min(c->gs_bytes, c->persist_bytes) : std::min(c->gs_bytes, c->window_max);
        av.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)c->persist_bytes / (double)av.accessPolicyWindow.num_bytes);
        av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        av.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
        if (cudaStreamSetAttribute(c->stream, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess) c->persist_mode = mode;
        else { cudaGetLastError(); c->persist_bytes = 0; }
    }
    KParams kp{};
    kp.vol = c->d_vol[mode];
    kp.Wb = (c->p.width + 3) / 4;
    kp.guide = c->d_guide[mode];
    kp.statA = c->d_statA[mode];
    kp.statB = c->d_statB[mode];
    kp.statC = c->d_statC[mode];
    kp.items = pl->d_items;
    kp.planes = d_planes;
    kp.out = d_out;
    kp.out_pitch = pitch;
    kp.out_compact = compact;
    kp.H = c->p.height; kp.W = c->p.width; kp.D = c->p.ndisp;
    kp.th_col = c->p.th_col; kp.min_disp = c->p.min_disp; kp.max_disp = c->p.max_disp;
    kp.with_check = with_check;
    kp.R = c->R;
    kp.exi_own = c->d_exi[mode];
    kp.exi_other = c->d_exi[1 - mode];
    kp.thresh_color = c->p.th_col * (1.0f - c->p.alpha);    // StereoEnergy.h:663
    kp.thresh_gradient = c->p.th_grad * c->p.alpha;          // StereoEnergy.h:664
    kp.mode = mode;
    kp.fast_ok = (c->vol_finite[mode] && c->p.min_disp == 0.0f && c->p.max_disp == (float)(c->p.ndisp - 1) && c->p.th_col >= 0.0f) ? 1 : 0;
    kp.smem_plane_off = (int)pl->smem - 16;
    if (pm) {
        kp.pm_mode = pm->pm_mode; kp.prop_kind = pm->prop_kind; kp.prop_m = pm->prop_m; kp.step_index = pm->step_index;
        kp.seed = pm->seed; kp.planes_out = pm->planes_out;
        kp.cur_cost = c->d_cur_cost[mode]; kp.cur_label = c->d_cur_label[mode];
        kp.calls = pl->d_calls;
        kp.cell_sync = reinterpret_cast<CellSync*>(c->d_sync_arena + pl->sync_off);
        const lexp_ctx::Peers& pr = c->peers[mode];
        kp.n_copies = pr.world; kp.my_rank = pr.rank;
        kp.copy_cost[0] = c->d_cur_cost[mode]; kp.copy_label[0] = c->d_cur_label[mode]; kp.copy_flags[0] = c->d_flags[mode];
        for (int i = 1; i < pr.world; i++) { kp.copy_cost[i] = pr.cost[i]; kp.copy_label[i] = pr.label[i]; kp.copy_flags[i] = pr.flags[i]; }
        kp.publish_epoch = pm->publish_epoch; kp.wait_mask = pm->wait_mask;
        for (int i = 0; i < kMaxPeers; i++) kp.wait_epochs[i] = pm->wait_epochs[i];
        kp.epoch_base = c->d_flags[mode] + kMaxPeers;
        kp.err_flag = c->d_flags[mode] + kMaxPeers + 1;
        kp.launch_done = reinterpret_cast<int*>(kp.cell_sync + pl->ncalls);
    }
    // PatchMatch phase with device-side proposers: every launch may start early; the steps of a cell are ordered by its counters, the
    // groups by epoch flags (lexp_plan_pm_step_ex)
    return launch_fused(c, kp, pl->nitems, pl->smem, overlap_ok);
}

// Scan a slab (disparities [d_lo, d_lo + nd) of the caller's volume, on the device) for NaN/Inf and re-lay it out into the context's
// blocked copy, applying the volume-preparation transform of lexp_relayout_volume on the way.  Asynchronous; d_flag accumulates.
int ingest_slab(lexp_ctx* c, int mode, const float* d_src, int d_lo, int nd, int transform, int* d_flag) {
    const int D = c->p.ndisp, H = c->p.height, W = c->p.width, Wb = (W + 3) / 4, Hb = (H + 3) / 4;
    LEXP_LAUNCH(lexp_scan_nonfinite, 148 * 8, 256, 0, c->stream, d_src, (size_t)nd * H * W, d_flag);
    dim3 grd((W + 31) / 32, Hb, (nd + 7) / 8);
    LEXP_LAUNCH(lexp_relayout_volume, grd, 256, 0, c->stream, d_src, c->d_vol[mode], D, H, W, Wb, d_lo, nd, transform);
    c->launches += 2;
    LEXP_CUDA(cudaGetLastError());
    return LEXP_OK;
}

int check_transform(int mode, int transform) {
    if (transform < LEXP_VOL_PLAIN || transform > LEXP_VOL_RIGHT_FROM_LEFT) return fail(LEXP_ERR_INVALID, "bad volume transform");
    if (transform == LEXP_VOL_RIGHT_FROM_LEFT && mode != 1) return fail(LEXP_ERR_INVALID, "LEXP_VOL_RIGHT_FROM_LEFT prepares view 1");
    return LEXP_OK;
}
// relayout selector: fillOutOfView depends on the view (main.cpp:153-175)
int kernel_transform(int mode, int transform) {
    return transform == LEXP_VOL_PLAIN ? 0 : transform == LEXP_VOL_RIGHT_FROM_LEFT ? 3 : (mode == 0 ? 1 : 2);
}

int alloc_volume(lexp_ctx* c, int mode, int** d_flag) {
    const int D = c->p.ndisp, H = c->p.height, W = c->p.width, Wb = (W + 3) / 4, Hb = (H + 3) / 4;
    if (!c->d_vol[mode]) LEXP_CUDA(cudaMalloc(&c->d_vol[mode], (size_t)Hb * Wb * D * 16 * sizeof(float)));
    LEXP_CUDA(cudaMalloc(d_flag, sizeof(int)));
    LEXP_CUDA(cudaMemsetAsync(*d_flag, 0, sizeof(int), c->stream));
    return LEXP_OK;
}

int finish_volume(lexp_ctx* c, int mode, int* d_flag) {
    int h = 1;
    cudaError_t e = cudaMemcpyAsync(&h, d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_flag);
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("volume ingest: ") + cudaGetErrorString(e));
    c->vol_finite[mode] = (h == 0);
    return LEXP_OK;
}

}  // namespace

extern "C" {

const char* lexp_last_error(void) { return g_err.c_str(); }
int lexp_version(void) { return 100; }

int lexp_create(const lexp_params* params, lexp_ctx** out_ctx) {
    if (!params || !out_ctx) return fail(LEXP_ERR_INVALID, "null argument");
    if (params->height <= 0 || params->width <= 0 || (params->ndisp < 2 && params->energy_kind == 0)) return fail(LEXP_ERR_INVALID, "bad H/W/D");
    if ((size_t)params->height * params->width >= (1ull << 30)) return fail(LEXP_ERR_INVALID, "image too large (H*W must be < 2^30)");
    if (params->windR < 2 || params->windR / 2 > 24) return fail(LEXP_ERR_INVALID, "windR/2 must be in [1, 24]");
    if (params->energy_kind != 0 && params->energy_kind != 1) return fail(LEXP_ERR_INVALID, "energy_kind must be 0 or 1");
    int ndev = 0;
    LEXP_CUDA(cudaGetDeviceCount(&ndev));
    if (params->device < 0 || params->device >= ndev) return fail(LEXP_ERR_INVALID, "bad device ordinal");
    LEXP_CUDA(cudaSetDevice(params->device));
    cudaDeviceProp prop;
    LEXP_CUDA(cudaGetDeviceProperties(&prop, params->device));
    if (prop.major < 10) return fail(LEXP_ERR_INVALID, "this library is built for sm_100a (B200) only");
    lexp_ctx* c = new lexp_ctx();
    c->p = *params;
    c->R = params->windR / 2;  // CostVolumeEnergy.h:30
    c->smem_limit = prop.sharedMemPerBlockOptin;
    c->tile_oh = std::max(8, env_int("LEXP_TILE_OH", 128));
    c->tile_oh_fixed = getenv("LEXP_TILE_OH") != nullptr;
    c->num_sms = prop.multiProcessorCount;
    // kMinCtas CTAs must fit next to each other: 1 KB of every CTA's shared memory is reserved by the system.  With the
    // default build (2 CTAs) no cap is needed: the widest tile needs ~93 KB.
    c->ctas_per_sm = env_int("LEXP_CTAS_PER_SM", kMinCtas);
    c->pdl = LEXP_PDL && !env_int("LEXP_PDL_OFF", 0);
    c->combine = env_int("LEXP_COMBINE", 1) != 0;
    c->comb_window_us = std::max(0, env_int("LEXP_COMBINE_WINDOW_US", 30));
    c->smem_cap = (size_t)env_int("LEXP_SMEM_CAP", 0);
    c->gc_threads = std::min(1024, std::max(32, env_int("LEXP_GC_THREADS", 1024) / 32 * 32));
    c->gc_relabel_every = std::max(1, env_int("LEXP_GC_RELABEL_EVERY", 24));
    c->gc_big_nodes = std::max(0, env_int("LEXP_GC_BIG_NODES", 32768));
    if (env_int("LEXP_L2_PERSIST", 1) && prop.persistingL2CacheMaxSize > 0) {
        const size_t want = (size_t)prop.persistingL2CacheMaxSize;
        if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
            c->persist_bytes = want;
            c->window_max = (size_t)prop.accessPolicyMaxWindowSize;
        } else cudaGetLastError();
        if (env_int("LEXP_DEBUG", 0))
            fprintf(stderr, "[lexp] L2 %d B, persisting max %d B, window max %d B, set-aside %zu B\n", prop.l2CacheSize,
                    prop.persistingL2CacheMaxSize, prop.accessPolicyMaxWindowSize, c->persist_bytes);
    }
    if (max_tile_ow(c->R) < 8) { delete c; return fail(LEXP_ERR_INVALID, "windR too large for the tile width"); }
    LEXP_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    *out_ctx = c;
    return LEXP_OK;
}

int lexp_destroy(lexp_ctx* c) {
    if (!c) return LEXP_OK;
    cudaSetDevice(c->p.device);
    cudaStreamSynchronize(c->stream);
    for (auto& kv : c->cell_plans) lexp_plan_destroy(kv.second);
    c->cell_plans.clear();
    for (lexp_plan* pl : c->live_plans) {  // user plans that outlive the context: orphaned, lexp_plan_destroy then only deletes
        release_plan_memory(pl);
        pl->ctx = nullptr;
    }
    c->live_plans.clear();
    for (auto& b : c->cb) {
        cudaFree(b.d_items); cudaFree(b.d_planes);
        if (b.h_items) cudaFreeHost(b.h_items);
        if (b.h_planes) cudaFreeHost(b.h_planes);
        if (b.h_out) cudaFreeHost(b.h_out);
    }
    for (int m = 0; m < 2; m++) {
        cudaFree(c->d_gs[m]);
        cudaFree(c->d_exi[m]);
        cudaFree(c->d_vol[m]);
#ifndef LEXP_EMU
        for (int i = 0; i < c->peers[m].n_opened; i++) cudaIpcCloseMemHandle(c->peers[m].ipc_opened[i]);
#endif
        cudaFree(c->d_cur_cost[m]);
        cudaFree(c->d_cur_label[m]);
        cudaFree(c->d_flags[m]);
        cudaFree(c->d_coef[m]);
        cudaFree(c->d_prop_cost[m]);
    }
    cudaFree(c->d_gc_scratch);
    if (c->h_gc_flags) cudaFreeHost(c->h_gc_flags);
    cudaFree(c->d_sync_arena);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return LEXP_OK;
}

int lexp_set_image(lexp_ctx* c, int mode, const uint8_t* bgr, ptrdiff_t step) {
    if (!c || !bgr || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const int H = c->p.height, W = c->p.width;
    const size_t HW = (size_t)H * W;
    c->coef_valid[mode] = false;
    std::vector<uchar4> tmp(HW);
    for (int y = 0; y < H; y++) {
        const uint8_t* row = bgr + (ptrdiff_t)y * step;
        for (int x = 0; x < W; x++) tmp[(size_t)y * W + x] = make_uchar4(row[3 * x], row[3 * x + 1], row[3 * x + 2], 0);
    }
    if (!c->d_gs[mode]) {
        // one allocation [statA | statC | guide | statB] so that a single L2 access-policy window can pin a prefix
        const size_t HWp = (HW + 63) / 64 * 64;
        LEXP_CUDA(cudaMalloc(&c->d_gs[mode], HWp * (16 + 4 + 4 + 16)));
        char* b = c->d_gs[mode];
        c->d_statA[mode] = reinterpret_cast<float4*>(b);
        c->d_statC[mode] = reinterpret_cast<float*>(b + HWp * 16);
        c->d_guide[mode] = reinterpret_cast<uchar4*>(b + HWp * 20);
        c->d_statB[mode] = reinterpret_cast<float4*>(b + HWp * 24);
        c->gs_bytes = HWp * 40;
    }
    LEXP_CUDA(cudaMemcpyAsync(c->d_guide[mode], tmp.data(), HW * sizeof(uchar4), cudaMemcpyHostToDevice, c->stream));
    int* d_rs = nullptr;
    LEXP_CUDA(cudaMalloc(&d_rs, 9 * HW * sizeof(int)));
    dim3 blk(128), grd((W + 127) / 128, H);
    LEXP_LAUNCH(lexp_stats_rowsum, grd, blk, 0, c->stream, c->d_guide[mode], d_rs, H, W, c->R);
    LEXP_LAUNCH(lexp_stats_finish, grd, blk, 0, c->stream, d_rs, c->d_statA[mode], c->d_statB[mode], c->d_statC[mode], H, W, c->R, (double)c->p.eps);
    c->launches += 2;
    if (c->p.energy_kind == 1) {
        if (!c->d_exi[mode] && cudaMalloc(&c->d_exi[mode], HW * sizeof(float4)) != cudaSuccess) { cudaFree(d_rs); return fail(LEXP_ERR_NOMEM, "ExI allocation failed"); }
        const float s_col = (float)(1.0 - (double)c->p.alpha);  // `I[m] * (1.0 - params.alpha)`, StereoEnergy.h:659
        LEXP_LAUNCH(lexp_build_exi, grd, blk, 0, c->stream, c->d_guide[mode], c->d_exi[mode], H, W, s_col, c->p.alpha);
        c->launches++;
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_rs);
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("statistics kernels: ") + cudaGetErrorString(e));
    return LEXP_OK;
}

// Host volume float[D][H][W]: uploaded in slabs of disparities through one device staging buffer, never as a second full-size device
// copy (17 GB per view at 4K).  Every copy is issued ON THE CONTEXT'S STREAM: the stream is non-blocking, so a plain cudaMemcpy (legacy
// default stream) is not ordered against its kernels -- and a synchronous copy from pageable memory returns once the data is staged,
// possibly before the DMA has landed: the re-layout kernel was observed reading a slab that had not arrived yet (flaky 1e-2 cost errors
// on the GPU).  Stream order also protects the staging buffer: the copy of slab k+1 follows the re-layout of slab k.
int lexp_set_volume_host_ex(lexp_ctx* c, int mode, const float* vol, int transform) {
    if (!c || !vol || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    { int rc = check_transform(mode, transform); if (rc) return rc; }
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const int D = c->p.ndisp, H = c->p.height, W = c->p.width;
    const size_t plane = (size_t)H * W;
    int slab = (int)std::max<size_t>(8, std::min<size_t>((size_t)D, ((size_t)env_int("LEXP_UPLOAD_SLAB_MB", 512) << 20) / (plane * sizeof(float))));
    slab = std::min(D, (slab + 7) / 8 * 8);
    int* d_flag = nullptr;
    { int rc = alloc_volume(c, mode, &d_flag); if (rc) return rc; }
    float* stage = nullptr;
    int rc = LEXP_OK;
    cudaError_t e = cudaMalloc(&stage, (size_t)slab * plane * sizeof(float));
    const int tk = kernel_transform(mode, transform);
    for (int d_lo = 0; d_lo < D && e == cudaSuccess && rc == LEXP_OK; d_lo += slab) {
        const int nd = std::min(slab, D - d_lo);
        e = cudaMemcpyAsync(stage, vol + (size_t)d_lo * plane, (size_t)nd * plane * sizeof(float), cudaMemcpyHostToDevice, c->stream);
        if (e != cudaSuccess) break;
        rc = ingest_slab(c, mode, stage, d_lo, nd, tk, d_flag);
    }
    if (e != cudaSuccess && rc == LEXP_OK) rc = fail(LEXP_ERR_CUDA, std::string("volume upload: ") + cudaGetErrorString(e));
    const int rc2 = finish_volume(c, mode, d_flag);   // synchronises the stream
    cudaFree(stage);
    return rc ? rc : rc2;
}

// The cost-volume file of the reference: raw float[D][H][W] without a header (`loadMatBinary(inputDir + "im0.acrt", volL, false)`,
// main.cpp:353-358,364; Utilities.hpp:173-201).  Streamed: slabs of disparities are read into two page-locked buffers in turn and uploaded
// on the context's stream while the next one is being read -- the 17 GB volume of the 4K configuration never has to exist in host memory.
int lexp_set_volume_file(lexp_ctx* c, int mode, const char* path, int transform) {
    if (!c || !path || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    { int rc = check_transform(mode, transform); if (rc) return rc; }
    const int D = c->p.ndisp, H = c->p.height, W = c->p.width;
    const size_t plane = (size_t)H * W;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(LEXP_ERR_INVALID, std::string("cost volume file not found: ") + path);
    if (fseek(f, 0, SEEK_END) != 0 || (unsigned long long)ftell(f) != (unsigned long long)D * plane * sizeof(float)) {
        fclose(f);
        return fail(LEXP_ERR_INVALID, std::string("cost volume file is not float[D][H][W] of this context's size: ") + path);
    }
    rewind(f);
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    if (cudaSetDevice(c->p.device) != cudaSuccess) { fclose(f); return fail(LEXP_ERR_CUDA, "cudaSetDevice"); }
    int slab = (int)std::max<size_t>(8, std::min<size_t>((size_t)D, ((size_t)env_int("LEXP_UPLOAD_SLAB_MB", 512) << 20) / (plane * sizeof(float))));
    slab = std::min(D, (slab + 7) / 8 * 8);
    int* d_flag = nullptr;
    { int rc = alloc_volume(c, mode, &d_flag); if (rc) { fclose(f); return rc; } }
    float* stage = nullptr;
    float* host[2] = {nullptr, nullptr};
    cudaEvent_t copied[2] = {nullptr, nullptr};
    int rc = LEXP_OK;
    cudaError_t e = cudaMalloc(&stage, (size_t)slab * plane * sizeof(float));
    for (int i = 0; i < 2 && e == cudaSuccess; i++) {
        e = cudaHostAlloc(&host[i], (size_t)slab * plane * sizeof(float), cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming);
    }
    const int tk = kernel_transform(mode, transform);
    for (int d_lo = 0, i = 0; d_lo < D && e == cudaSuccess && rc == LEXP_OK; d_lo += slab, i ^= 1) {
        const int nd = std::min(slab, D - d_lo);
        e = cudaEventSynchronize(copied[i]);   // the upload that last read this host buffer has finished (no-op the first time)
        if (e != cudaSuccess) break;
        if (fread(host[i], sizeof(float), (size_t)nd * plane, f) != (size_t)nd * plane) { rc = fail(LEXP_ERR_INVALID, std::string("short read: ") + path); break; }
        e = cudaMemcpyAsync(stage, host[i], (size_t)nd * plane * sizeof(float), cudaMemcpyHostToDevice, c->stream);   // behind the previous slab's re-layout
        if (e == cudaSuccess) e = cudaEventRecord(copied[i], c->stream);
        if (e != cudaSuccess) break;
        rc = ingest_slab(c, mode, stage, d_lo, nd, tk, d_flag);
    }
    fclose(f);
    if (e != cudaSuccess && rc == LEXP_OK) rc = fail(LEXP_ERR_CUDA, std::string("volume file upload: ") + cudaGetErrorString(e));
    const int rc2 = finish_volume(c, mode, d_flag);   // synchronises the stream
    cudaFree(stage);
    for (int i = 0; i < 2; i++) { if (host[i]) cudaFreeHost(host[i]); if (copied[i]) cudaEventDestroy(copied[i]); }
    return rc ? rc : rc2;
}

int lexp_set_volume_device_ex(lexp_ctx* c, int mode, const float* vol, int transform) {
    if (!c || !vol || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    { int rc = check_transform(mode, transform); if (rc) return rc; }
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    cudaPointerAttributes at;
    LEXP_CUDA(cudaPointerGetAttributes(&at, vol));
    if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)
        return fail(LEXP_ERR_INVALID, "lexp_set_volume_device needs a device pointer");
    LEXP_CUDA(cudaSetDevice(c->p.device));
    // the caller's volume was produced on a stream this library does not know (e.g. torch's): the context's own stream is
    // non-blocking, so nothing orders its re-layout kernel behind that producer -- wait for the device once (one-time set-up call)
    LEXP_CUDA(cudaDeviceSynchronize());
    int* d_flag = nullptr;
    { int rc = alloc_volume(c, mode, &d_flag); if (rc) return rc; }
    const int rc = ingest_slab(c, mode, vol, 0, c->p.ndisp, kernel_transform(mode, transform), d_flag);
    const int rc2 = finish_volume(c, mode, d_flag);
    return rc ? rc : rc2;
}

int lexp_set_volume_host(lexp_ctx* c, int mode, const float* vol) { return lexp_set_volume_host_ex(c, mode, vol, LEXP_VOL_PLAIN); }
int lexp_set_volume_device(lexp_ctx* c, int mode, const float* vol) { return lexp_set_volume_device_ex(c, mode, vol, LEXP_VOL_PLAIN); }

int lexp_get_stats(lexp_ctx* c, int mode, float* out9) {
    if (!c || !out9 || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_statA[mode]) return fail(LEXP_ERR_STATE, "image not set");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const size_t HW = (size_t)c->p.height * c->p.width;
    float* d9 = nullptr;
    LEXP_CUDA(cudaMalloc(&d9, 9 * HW * sizeof(float)));
    LEXP_LAUNCH(lexp_stats_unpack, (unsigned)((HW + 255) / 256), 256, 0, c->stream, c->d_statA[mode], c->d_statB[mode], c->d_statC[mode], d9, HW);
    c->launches++;
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = cudaMemcpy(out9, d9, 9 * HW * sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(d9);
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("get_stats: ") + cudaGetErrorString(e));
    return LEXP_OK;
}

int lexp_plan_create(lexp_ctx* c, int n, const lexp_rect* filt, const lexp_rect* targ, lexp_plan** out_plan) {
    if (!c || !filt || !targ || !out_plan || n <= 0) return fail(LEXP_ERR_INVALID, "bad argument");
    for (int i = 0; i < n; i++) {
        int rc = check_rects(c, filt[i], targ[i]);
        if (rc) return rc;
    }
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const int R = c->R;
    int ow_max = max_tile_ow(R);
    if (c->smem_cap)  // narrower tiles so that every work item fits the per-CTA shared-memory budget of the build
        while (ow_max > 8 && fused_smem_bytes(ow_max + 4 * R, 128, R) > c->smem_cap) ow_max -= 4;
    // Row segmentation: every segment re-streams 4R warm-up rows, but more items fill the 2 x #SM CTA slots better.
    // Pick the segment height that minimises  waves x (rows streamed per item)  for this plan.
    int oh_max = c->tile_oh;
    if (!c->tile_oh_fixed) {
        const int64_t slots = (int64_t)c->ctas_per_sm * c->num_sms;
        double best = 1e300;
        for (int cand = 24; cand <= 128; cand += 4) {
            int64_t items = 0;
            int max_rows = 0;
            for (int i = 0; i < n; i++) {
                const int ncol = (targ[i].width + ow_max - 1) / ow_max, nrow = (targ[i].height + cand - 1) / cand;
                items += (int64_t)ncol * nrow;
                max_rows = std::max(max_rows, (targ[i].height + nrow - 1) / nrow);
            }
            const double waves = (double)((items + slots - 1) / slots);
            const double cost = waves * (max_rows + 4 * R + 12);
            if (cost < best - 1e-9) { best = cost; oh_max = cand; }
        }
    }
    lexp_plan* pl = new lexp_plan();
    pl->ctx = c;
    pl->ncalls = n;
    pl->filt.assign(filt, filt + n);
    pl->targ.assign(targ, targ + n);
    pl->compact_off.resize(n);
    pl->items_per_call.assign(n, 0);
    std::vector<Item> items;
    int64_t coff = 0;
    for (int i = 0; i < n; i++) {
        const lexp_rect &f = filt[i], &t = targ[i];
        pl->compact_off[i] = (int)coff;
        const int ncol = (t.width + ow_max - 1) / ow_max, nrow = (t.height + oh_max - 1) / oh_max;
        for (int rj = 0; rj < nrow; rj++) {
            const int y0 = t.y + (int)((int64_t)t.height * rj / nrow), y1 = t.y + (int)((int64_t)t.height * (rj + 1) / nrow);
            for (int cj = 0; cj < ncol; cj++) {
                const int x0 = t.x + (int)((int64_t)t.width * cj / ncol), x1 = t.x + (int)((int64_t)t.width * (cj + 1) / ncol);
                Item it{};
                it.fx = f.x; it.fy = f.y; it.fw = f.width; it.fh = f.height;
                it.ox0 = x0; it.oy0 = y0; it.ow = x1 - x0; it.oh = y1 - y0;
                it.call = i;
                it.compact_off = (int)(coff + (int64_t)(y0 - t.y) * t.width + (x0 - t.x));
                it.compact_stride = t.width;
                it.flags = (t.width == 1 && t.height == 1) ? 1 : 0;
                items.push_back(it);
                pl->items_per_call[i]++;
                pl->max_vw = std::max(pl->max_vw, it.ow + 4 * R);
                pl->smem = std::max(pl->smem, fused_smem_bytes(it.ow + 4 * R, it.oh, R));
            }
        }
        coff += (int64_t)t.width * t.height;
        // work accounting (SURVEY.md section 8d): F = filterRect px, S = targetRect px,
        // A = targetRect dilated by R, clipped to filterRect
        const int64_t F = (int64_t)f.width * f.height, S = (int64_t)t.width * t.height;
        const int ax0 = std::max(t.x - R, f.x), ax1 = std::min(t.x + t.width + R, f.x + f.width);
        const int ay0 = std::max(t.y - R, f.y), ay1 = std::min(t.y + t.height + R, f.y + f.height);
        const int64_t A = (int64_t)(ax1 - ax0) * (ay1 - ay0);
        pl->sum_f += F; pl->sum_s += S;
        pl->alg_bytes += 20 * F + 36 * A + 4 * S;
    }
    if (coff > 0x7fffffffLL) { delete pl; return fail(LEXP_ERR_INVALID, "plan output too large"); }
    // big items first: the hardware scheduler then back-fills with small ones
    std::stable_sort(items.begin(), items.end(), [R](const Item& a, const Item& b) {
        return (int64_t)(a.ow + 4 * R) * (a.oh + 4 * R) > (int64_t)(b.ow + 4 * R) * (b.oh + 4 * R);
    });
    pl->nitems = (int)items.size();
    pl->h_items = items;
    cudaError_t e = cudaMalloc(&pl->d_items, items.size() * sizeof(Item));
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_planes, (size_t)n * sizeof(Plane4));
    // on the context's (non-blocking) stream, then synchronised: a legacy-stream cudaMemcpy is not ordered against the launches that read the items
    if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_items, items.data(), items.size() * sizeof(Item), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        cudaFree(pl->d_items); cudaFree(pl->d_planes);
        delete pl;
        return fail(LEXP_ERR_CUDA, std::string("plan upload: ") + cudaGetErrorString(e));
    }
    {
        std::lock_guard<std::mutex> lk2(c->plans_mu);
        c->live_plans.insert(pl);
    }
    *out_plan = pl;
    return LEXP_OK;
}

int lexp_plan_destroy(lexp_plan* pl) {
    if (!pl) return LEXP_OK;
    if (lexp_ctx* c = pl->ctx) {  // nullptr: the context was destroyed first and has already released the plan's memory
        cudaSetDevice(c->p.device);
        cudaStreamSynchronize(c->stream);
        release_plan_memory(pl);
        std::lock_guard<std::mutex> lk(c->plans_mu);
        c->live_plans.erase(pl);
    }
    delete pl;
    return LEXP_OK;
}

int lexp_plan_num_calls(const lexp_plan* pl) { return pl ? pl->ncalls : 0; }
int lexp_plan_num_items(const lexp_plan* pl) { return pl ? pl->nitems : 0; }

int lexp_plan_work(const lexp_plan* pl, int64_t* sf, int64_t* ss, int64_t* ab) {
    if (!pl) return fail(LEXP_ERR_INVALID, "null plan");
    if (sf) *sf = pl->sum_f;
    if (ss) *ss = pl->sum_s;
    if (ab) *ab = pl->alg_bytes;
    return LEXP_OK;
}

int lexp_plan_eval_device(lexp_ctx* c, lexp_plan* pl, int mode, const lexp_plane* planes, int planes_on_device,
                          float* d_cost_image, ptrdiff_t step_bytes, int with_check) {
    if (!c || !pl || !planes || !d_cost_image || pl->ctx != c) return fail(LEXP_ERR_INVALID, "bad argument");
    if (step_bytes % 4 != 0 || step_bytes < (ptrdiff_t)c->p.width * 4) return fail(LEXP_ERR_INVALID, "bad row pitch");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const Plane4* dp = reinterpret_cast<const Plane4*>(planes);
    if (!planes_on_device) {
        LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
        dp = pl->d_planes;
        c->chain_ok = false;
    }
    return run_plan(c, pl, mode, dp, d_cost_image, step_bytes / 4, 0, with_check, nullptr, planes_on_device && c->overlap);
}

int lexp_plan_eval_device_tiles(lexp_ctx* c, lexp_plan* pl, int mode, const lexp_plane* planes, int planes_on_device,
                                float* d_tiles, int with_check) {
    if (!c || !pl || !planes || !d_tiles || pl->ctx != c) return fail(LEXP_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const Plane4* dp = reinterpret_cast<const Plane4*>(planes);
    if (!planes_on_device) {
        LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
        dp = pl->d_planes;
        c->chain_ok = false;
    }
    return run_plan(c, pl, mode, dp, d_tiles, 0, 1, with_check, nullptr, planes_on_device && c->overlap);
}

// Host planes in, per-call contiguous tiles out into HOST memory; blocking.  For the step-wise restructured loop
// (INTEGRATION.md section 3): the fusion of cell i reads its proposal costs from a cv::Mat header over tile i
// (cv::Mat(h, w, CV_32F, tiles + offset_i)), so nothing has to be scattered into an H x W image, and consecutive rows of a
// tile are contiguous in memory (full-line PCIe writes on the zero-copy path).
int lexp_plan_eval_host_tiles(lexp_ctx* c, lexp_plan* pl, int mode, const lexp_plane* planes, float* tiles, int with_check) {
    if (!c || !pl || !planes || !tiles || pl->ctx != c) return fail(LEXP_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
    void* dptr = mapped_alias(tiles, (size_t)pl->sum_s * sizeof(float));
    if (dptr) {  // registered (mapped) buffer: the kernel writes it directly
        int rc = run_plan(c, pl, mode, pl->d_planes, reinterpret_cast<float*>(dptr), 0, 1, with_check);
        if (rc) return rc;
        LEXP_CUDA(cudaStreamSynchronize(c->stream));
        return LEXP_OK;
    }
    // not a mapped buffer: compact device buffer, then one contiguous copy
    const size_t nout = (size_t)pl->sum_s;
    { int rc0 = ensure_compact(pl, nout); if (rc0) return rc0; }
    int rc = run_plan(c, pl, mode, pl->d_planes, pl->d_compact, 0, 1, with_check);
    if (rc) return rc;
    if (registered_host(tiles)) {  // starts inside a registration that does not cover it: one copy cannot span both kinds of memory
        LEXP_CUDA(cudaMemcpyAsync(pl->h_compact, pl->d_compact, nout * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        LEXP_CUDA(cudaStreamSynchronize(c->stream));
        memcpy(tiles, pl->h_compact, nout * sizeof(float));
        return LEXP_OK;
    }
    LEXP_CUDA(cudaMemcpyAsync(tiles, pl->d_compact, nout * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    LEXP_CUDA(cudaStreamSynchronize(c->stream));
    return LEXP_OK;
}

int lexp_plan_eval_host(lexp_ctx* c, lexp_plan* pl, int mode, const lexp_plane* planes, float* cost_image,
                        ptrdiff_t step_bytes, int with_check) {
    if (!c || !pl || !planes || !cost_image || pl->ctx != c) return fail(LEXP_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    {   // zero-copy path: the caller's image is page-locked + mapped (lexp_host_register)
        // the calls write rows t.y .. t.y + t.height - 1 of the image: the range that must be mapped spans them all
        int y_lo = INT_MAX, y_hi = -1, x_hi = 0;
        for (const lexp_rect& t : pl->targ) { y_lo = std::min(y_lo, t.y); y_hi = std::max(y_hi, t.y + t.height - 1); x_hi = std::max(x_hi, t.x + t.width); }
        char* lo = reinterpret_cast<char*>(cost_image) + (ptrdiff_t)y_lo * step_bytes;
        const size_t span = step_bytes > 0 && y_hi >= y_lo ? (size_t)(y_hi - y_lo) * (size_t)step_bytes + (size_t)x_hi * sizeof(float) : 0;
        void* dlo = span ? mapped_alias(lo, span) : nullptr;
        void* dptr = dlo ? static_cast<char*>(dlo) - (ptrdiff_t)y_lo * step_bytes : nullptr;
        if (dptr) {
            if (step_bytes % 4 != 0) return fail(LEXP_ERR_INVALID, "bad row pitch");
            LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
            int rc = run_plan(c, pl, mode, pl->d_planes, reinterpret_cast<float*>(dptr), step_bytes / 4, 0, with_check);
            if (rc) return rc;
            LEXP_CUDA(cudaStreamSynchronize(c->stream));
            return LEXP_OK;
        }
    }   // not a mapped buffer: staged path below
    const size_t nout = (size_t)pl->sum_s;
    { int rc0 = ensure_compact(pl, nout); if (rc0) return rc0; }
    LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
    int rc = run_plan(c, pl, mode, pl->d_planes, pl->d_compact, 0, 1, with_check);
    if (rc) return rc;
    LEXP_CUDA(cudaMemcpyAsync(pl->h_compact, pl->d_compact, nout * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    LEXP_CUDA(cudaStreamSynchronize(c->stream));
    // scatter the per-call tiles into the caller's image: costs(targetRect) only (CostVolumeEnergy.h:169-171)
    for (int i = 0; i < pl->ncalls; i++) {
        const lexp_rect& t = pl->targ[i];
        const float* src = pl->h_compact + pl->compact_off[i];
        for (int y = 0; y < t.height; y++) {
            float* dst = reinterpret_cast<float*>(reinterpret_cast<char*>(cost_image) + (ptrdiff_t)(t.y + y) * step_bytes) + t.x;
            memcpy(dst, src + (size_t)y * t.width, (size_t)t.width * sizeof(float));
        }
    }
    return LEXP_OK;
}

int lexp_eval_batch(lexp_ctx* c, int mode, int n, const lexp_rect* filt, const lexp_rect* targ, const lexp_plane* planes,
                    float* cost_image, ptrdiff_t step_bytes, int with_check) {
    lexp_plan* pl = nullptr;
    int rc = lexp_plan_create(c, n, filt, targ, &pl);
    if (rc) return rc;
    rc = lexp_plan_eval_host(c, pl, mode, planes, cost_image, step_bytes, with_check);
    std::string keep = g_err;
    lexp_plan_destroy(pl);
    g_err = keep;
    return rc;
}

namespace {

// One batched launch for the queued single-cell requests of one (mode, with_check): the work items of the cached per-cell plans are
// concatenated in pinned staging memory (call index = position in the batch, compact outputs back to back), the kernel writes the
// compact tiles straight into mapped pinned host memory, and every request learns where its tile is (the callers copy them out).
int run_combined(lexp_ctx* c, const std::vector<lexp_ctx::CellReq*>& reqs) {
    size_t nitems = 0, nout = 0, smem = 0;
    for (auto* r : reqs) { nitems += r->pl->h_items.size(); nout += (size_t)r->pl->sum_s; smem = std::max(smem, r->pl->smem); }
    if (nout > 0x7fffffffULL) return fail(LEXP_ERR_INVALID, "combined output too large");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    lexp_ctx::CombBuf& b = c->cb[c->cb_next];
    c->cb_next ^= 1;
    // the callers of the batch that used this buffer two batches ago must have copied their tiles out
    for (int spin = 0; b.copies_left.load(std::memory_order_acquire) > 0; spin++) {
        if (spin > 2000) std::this_thread::sleep_for(std::chrono::microseconds(5)); else cpu_relax();
    }
    if (nitems > b.items_cap || reqs.size() > b.planes_cap || nout > b.out_cap) {
        LEXP_CUDA(cudaStreamSynchronize(c->stream));
        if (nitems > b.items_cap) {
            cudaFree(b.d_items); b.d_items = nullptr; if (b.h_items) cudaFreeHost(b.h_items); b.h_items = nullptr; b.items_cap = 0;
            LEXP_CUDA(cudaMalloc(&b.d_items, 2 * nitems * sizeof(Item)));
            LEXP_CUDA(cudaHostAlloc(&b.h_items, 2 * nitems * sizeof(Item), cudaHostAllocDefault));
            b.items_cap = 2 * nitems;
        }
        if (reqs.size() > b.planes_cap) {
            cudaFree(b.d_planes); b.d_planes = nullptr; if (b.h_planes) cudaFreeHost(b.h_planes); b.h_planes = nullptr; b.planes_cap = 0;
            LEXP_CUDA(cudaMalloc(&b.d_planes, 2 * reqs.size() * sizeof(Plane4)));
            LEXP_CUDA(cudaHostAlloc(&b.h_planes, 2 * reqs.size() * sizeof(Plane4), cudaHostAllocDefault));
            b.planes_cap = 2 * reqs.size();
        }
        if (nout > b.out_cap) {
            if (b.h_out) cudaFreeHost(b.h_out);
            b.h_out = nullptr; b.d_out = nullptr; b.out_cap = 0;
            LEXP_CUDA(cudaHostAlloc(&b.h_out, 2 * nout * sizeof(float), cudaHostAllocMapped));
            LEXP_CUDA(cudaHostGetDevicePointer(&b.d_out, b.h_out, 0));
            b.out_cap = 2 * nout;
        }
    }
    size_t at = 0, off = 0;
    for (size_t i = 0; i < reqs.size(); i++) {
        const lexp_plan* pl = reqs[i]->pl;
        for (Item it : pl->h_items) {
            it.call = (int)i;
            it.compact_off += (int)off;  // the plan's own call starts at offset 0
            b.h_items[at++] = it;
        }
        reqs[i]->tile = b.h_out + off;
        reqs[i]->copies_left = &b.copies_left;
        off += (size_t)pl->sum_s;
        const lexp_plane& p = reqs[i]->plane;
        b.h_planes[i] = Plane4{p.a, p.b, p.c, p.v};
    }
    LEXP_CUDA(cudaMemcpyAsync(b.d_items, b.h_items, nitems * sizeof(Item), cudaMemcpyHostToDevice, c->stream));
    LEXP_CUDA(cudaMemcpyAsync(b.d_planes, b.h_planes, reqs.size() * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
    lexp_plan batch;  // a view: nothing in it is owned
    batch.ctx = c;
    batch.ncalls = (int)reqs.size();
    batch.nitems = (int)nitems;
    batch.smem = smem;
    batch.d_items = b.d_items;
    int rc = run_plan(c, &batch, reqs[0]->mode, b.d_planes, b.d_out, 0, 1, reqs[0]->with_check);
    batch.d_items = nullptr;
    if (rc) return rc;
    LEXP_CUDA(cudaStreamSynchronize(c->stream));
    b.copies_left.store((int)reqs.size(), std::memory_order_release);
    c->combined_batches++;
    c->combined_calls += (int64_t)reqs.size();
    return LEXP_OK;
}

// a caller's own part of a combined batch: costs(targetRect) only (CostVolumeEnergy.h:169-171)
void copy_out_tile(lexp_ctx::CellReq& r) {
    const lexp_rect& t = r.pl->targ[0];
    for (int y = 0; y < t.height; y++) {
        float* dst = reinterpret_cast<float*>(reinterpret_cast<char*>(r.base) + (ptrdiff_t)(t.y + y) * r.step_bytes) + t.x;
        memcpy(dst, r.tile + (size_t)y * t.width, (size_t)t.width * sizeof(float));
    }
    r.copies_left->fetch_sub(1, std::memory_order_acq_rel);
}

}  // namespace

int lexp_eval_cell(lexp_ctx* c, int mode, const lexp_rect* filt, const lexp_rect* targ, const lexp_plane* plane, float* costs,
                   ptrdiff_t step_bytes, int with_check) {
    if (!c || !filt || !targ || !plane || !costs) return fail(LEXP_ERR_INVALID, "null argument");
    // `costs` addresses element (filterRect.y, filterRect.x); rebase to image element (0,0)
    float* base = reinterpret_cast<float*>(reinterpret_cast<char*>(costs) - (ptrdiff_t)filt->y * step_bytes) - filt->x;
    const std::array<int, 8> key = {filt->x, filt->y, filt->width, filt->height, targ->x, targ->y, targ->width, targ->height};
    lexp_plan* pl = nullptr;
    {
        std::lock_guard<std::mutex> lk(c->cache_mu);
        auto itp = c->cell_plans.find(key);
        if (itp != c->cell_plans.end()) pl = itp->second;
    }
    if (!pl) {
        int rc = lexp_plan_create(c, 1, filt, targ, &pl);
        if (rc) return rc;
        std::lock_guard<std::mutex> lk(c->cache_mu);
        auto ins = c->cell_plans.emplace(key, pl);
        if (!ins.second) {  // another thread created it meanwhile
            lexp_plan_destroy(pl);
            pl = ins.first->second;
        } else if (c->cell_plans.size() > 200000) {  // unbounded callers (initCurrentFast with a labeling: one rect per pixel)
            c->cell_plans.erase(ins.first);
            int rc2 = lexp_plan_eval_host(c, pl, mode, plane, base, step_bytes, with_check);
            std::string keep = g_err;
            lexp_plan_destroy(pl);
            g_err = keep;
            return rc2;
        }
    }
    if (!c->combine || mode < 0 || mode > 1) return lexp_plan_eval_host(c, pl, mode, plane, base, step_bytes, with_check);

    lexp_ctx::CellReq req;
    req.mode = mode; req.with_check = with_check; req.pl = pl; req.plane = *plane; req.base = base; req.step_bytes = step_bytes;
    bool lead = false;
    {
        std::lock_guard<std::mutex> lk(c->comb_mu);
        c->comb_q.push_back(&req);
        c->comb_n.store((int)c->comb_q.size(), std::memory_order_release);
        if (!c->comb_leader) { c->comb_leader = true; lead = true; }
    }
    for (;;) {
        if (!lead) {   // sleep until the own request is done, or is asked to lead the next batch
            int st;
            for (int spin = 0;; spin++) {
                const int g = c->comb_gen.load(std::memory_order_acquire);
                if ((st = req.state.load(std::memory_order_acquire)) != 0) break;
                if (spin < 200) cpu_relax(); else futex_wait(&c->comb_gen, g);
            }
            if (st == 1) break;
            req.state.store(0, std::memory_order_relaxed);   // st == 2: lead
        }
        // ---- leader: give the group's other threads a moment to arrive, then serve everything that is queued
        using clk = std::chrono::steady_clock;
        const auto t0 = clk::now();
        int seen = 0;
        auto last_growth = t0;
        for (;;) {
            const int n = c->comb_n.load(std::memory_order_acquire);
            const auto now = clk::now();
            if (n != seen) { seen = n; last_growth = now; }
            if ((size_t)n >= c->comb_seen.load(std::memory_order_relaxed) || now - t0 > std::chrono::microseconds(c->comb_window_us) ||
                now - last_growth > std::chrono::microseconds(c->comb_window_us / 4 + 1)) break;
            for (int i = 0; i < 64; i++) cpu_relax();
        }
        std::vector<lexp_ctx::CellReq*> all;
        {
            std::lock_guard<std::mutex> lk(c->comb_mu);
            all.swap(c->comb_q);
            c->comb_n.store(0, std::memory_order_release);
        }
        if (all.size() > c->comb_seen.load()) c->comb_seen.store(all.size());
        // one launch per (mode, with_check) present in the queue (the reference's loop uses a single combination at a time)
        while (!all.empty()) {
            std::vector<lexp_ctx::CellReq*> grp, rest;
            for (auto* r : all) (r->mode == all[0]->mode && r->with_check == all[0]->with_check ? grp : rest).push_back(r);
            const int rc = grp.size() == 1 && grp[0] == &req && rest.empty()
                               ? lexp_plan_eval_host(c, pl, mode, plane, base, step_bytes, with_check)   // alone: the plain single-cell path
                               : run_combined(c, grp);
            for (auto* r : grp) {
                r->status = rc;
                if (rc) { r->err = g_err; r->tile = nullptr; }
                if (r != &req) r->state.store(1, std::memory_order_release);
            }
            all.swap(rest);
        }
        {   // hand the leadership to a request that arrived meanwhile, or retire
            std::lock_guard<std::mutex> lk(c->comb_mu);
            if (c->comb_q.empty()) c->comb_leader = false;
            else c->comb_q.front()->state.store(2, std::memory_order_release);
        }
        c->comb_gen.fetch_add(1, std::memory_order_acq_rel);   // one wake-up for everybody whose state changed
        futex_wake_all(&c->comb_gen);
        break;   // the leader's own request was part of its batch
    }
    if (req.status) { g_err = req.err; return req.status; }
    if (req.tile) copy_out_tile(req);
    return LEXP_OK;
}

int lexp_combine_stats(const lexp_ctx* c, int64_t* batches, int64_t* calls) {
    if (!c) return fail(LEXP_ERR_INVALID, "null ctx");
    if (batches) *batches = c->combined_batches;
    if (calls) *calls = c->combined_calls;
    return LEXP_OK;
}

int lexp_host_register(void* ptr, size_t bytes) {
    if (!ptr || !bytes) return fail(LEXP_ERR_INVALID, "bad argument");
    LEXP_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable));
    return LEXP_OK;
}

int lexp_host_unregister(void* ptr) {
    if (!ptr) return fail(LEXP_ERR_INVALID, "bad argument");
    LEXP_CUDA(cudaHostUnregister(ptr));
    return LEXP_OK;
}

int lexp_sync(lexp_ctx* c) {
    if (!c) return fail(LEXP_ERR_INVALID, "null ctx");
    LEXP_CUDA(cudaSetDevice(c->p.device));
    LEXP_CUDA(cudaStreamSynchronize(c->stream));
    return LEXP_OK;
}

void* lexp_stream(lexp_ctx* c) { return c ? (void*)c->stream : nullptr; }

int lexp_set_stream(lexp_ctx* c, void* s) {
    if (!c) return fail(LEXP_ERR_INVALID, "null ctx");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    // no synchronisation here (the call must be legal while the caller captures a CUDA graph): ordering between the
    // old and the new stream is the caller's business
    if (c->own_stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); c->own_stream = false; }
    c->stream = (cudaStream_t)s;
    c->persist_mode = -1;
    return LEXP_OK;
}
int64_t lexp_launch_count(const lexp_ctx* c) { return c ? c->launches : 0; }

int lexp_set_overlap(lexp_ctx* c, int on) {
    if (!c) return fail(LEXP_ERR_INVALID, "null ctx");
    std::lock_guard<std::mutex> lk(c->mu);
    c->overlap = on != 0;
    return LEXP_OK;
}

// ---- PatchMatch phase on the device (FastGCStereo.h:94-157 with doGC == false) ---------------------------------------------
int lexp_pm_begin(lexp_ctx* c, int mode, const float* cost, const lexp_plane* labeling) {
    if (!c || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const size_t HW = (size_t)c->p.height * c->p.width;
    if (!c->d_cur_cost[mode]) LEXP_CUDA(cudaMalloc(&c->d_cur_cost[mode], HW * sizeof(float)));
    if (!c->d_cur_label[mode]) LEXP_CUDA(cudaMalloc(&c->d_cur_label[mode], HW * sizeof(float4)));
    if (!c->d_flags[mode]) {
        LEXP_CUDA(cudaMalloc(&c->d_flags[mode], (kMaxPeers + 2) * sizeof(int)));   // + epoch base + error flag
        LEXP_CUDA(cudaMemsetAsync(c->d_flags[mode], 0, (kMaxPeers + 2) * sizeof(int), c->stream));   // epochs only grow: never reset while peers run
    }
    if (cost) LEXP_CUDA(cudaMemcpyAsync(c->d_cur_cost[mode], cost, HW * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    else {
        LEXP_LAUNCH(lexp_fill_f32, 148 * 4, 256, 0, c->stream, c->d_cur_cost[mode], HW, __builtin_inff());   // currentCost_ = INFINITY (:137)
        LEXP_CUDA(cudaGetLastError());
        c->launches++;
    }
    if (labeling) LEXP_CUDA(cudaMemcpyAsync(c->d_cur_label[mode], labeling, HW * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    else LEXP_CUDA(cudaMemsetAsync(c->d_cur_label[mode], 0, HW * sizeof(float4), c->stream));
    if (cost || labeling) LEXP_CUDA(cudaStreamSynchronize(c->stream));  // the host buffers may be pageable
    return LEXP_OK;
}

int lexp_pm_get(lexp_ctx* c, int mode, float* cost, lexp_plane* labeling) {
    if (!c || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const size_t HW = (size_t)c->p.height * c->p.width;
    if (cost) LEXP_CUDA(cudaMemcpyAsync(cost, c->d_cur_cost[mode], HW * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (labeling) LEXP_CUDA(cudaMemcpyAsync(labeling, c->d_cur_label[mode], HW * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    int err = 0;
    LEXP_CUDA(cudaMemcpyAsync(&err, c->d_flags[mode] + kMaxPeers + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LEXP_CUDA(cudaStreamSynchronize(c->stream));
    if (err == 2) return fail(LEXP_ERR_STATE, "a graph-cut move stopped at its round limit: the state is not the result of minimum cuts");
    if (err) return fail(LEXP_ERR_STATE, "a wait for a peer rank's group epoch timed out (multi-GPU cell shard): the state is incomplete");
    return LEXP_OK;
}

int lexp_pm_device_state(lexp_ctx* c, int mode, float** d_cost, lexp_plane** d_labeling) {
    if (!c || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    if (d_cost) *d_cost = c->d_cur_cost[mode];
    if (d_labeling) *d_labeling = reinterpret_cast<lexp_plane*>(c->d_cur_label[mode]);
    return LEXP_OK;
}

int lexp_plan_set_units(lexp_plan* pl, const lexp_rect* units, const int* cell_ids) {
    if (!pl || !units) return fail(LEXP_ERR_INVALID, "bad argument");
    lexp_ctx* c = pl->ctx;
    if (!c) return fail(LEXP_ERR_STATE, "the plan's context has been destroyed");
    const int H = c->p.height, W = c->p.width;
    std::vector<CallInfo> h(pl->ncalls);
    for (int i = 0; i < pl->ncalls; i++) {
        const lexp_rect& u = units[i];
        if (u.width <= 0 || u.height <= 0 || u.x < 0 || u.y < 0 || u.x + u.width > W || u.y + u.height > H)
            return fail(LEXP_ERR_INVALID, "unitRegion outside the image");
        h[i] = CallInfo{u.x, u.y, u.width, u.height, pl->items_per_call[i] * kWarpsE, cell_ids ? cell_ids[i] : i, pl->items_per_call[i], 0};
    }
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    if (!pl->d_calls) LEXP_CUDA(cudaMalloc(&pl->d_calls, (size_t)pl->ncalls * sizeof(CallInfo)));
    LEXP_CUDA(cudaMemcpyAsync(pl->d_calls, h.data(), h.size() * sizeof(CallInfo), cudaMemcpyHostToDevice, c->stream));   // stream-ordered (see lexp_plan_create)
    LEXP_CUDA(cudaStreamSynchronize(c->stream));
    if (pl->sync_off < 0) {   // a slice of the context's synchronisation arena (offsets survive a re-allocation of the arena)
        const size_t need = ((size_t)pl->ncalls + 1) * sizeof(CellSync);
        if (c->sync_used + need > c->sync_cap) {
            const size_t cap = std::max<size_t>(2 * c->sync_cap, std::max<size_t>(1 << 20, c->sync_used + need));
            char* na = nullptr;
            LEXP_CUDA(cudaMalloc(&na, cap));
            LEXP_CUDA(cudaMemsetAsync(na, 0, cap, c->stream));
            LEXP_CUDA(cudaStreamSynchronize(c->stream));
            cudaFree(c->d_sync_arena);   // the stream is idle (synchronised above); the records are zeroed before every iteration anyway
            c->d_sync_arena = na; c->sync_cap = cap;
        }
        pl->sync_off = (long long)c->sync_used;
        c->sync_used += need;
    }
    return LEXP_OK;
}

// Zero the completion counters of ALL plans of the context (asynchronous): once before the steps of an initialisation / iteration
// are issued -- not between groups, so that all launches of an iteration form one programmatic-dependent-launch chain.
int lexp_pm_reset_sync(lexp_ctx* c) {
    if (!c) return fail(LEXP_ERR_INVALID, "null ctx");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    if (c->sync_used) LEXP_CUDA(cudaMemsetAsync(c->d_sync_arena, 0, c->sync_used, c->stream));
    return LEXP_OK;
}

int lexp_plan_pm_step_ex(lexp_ctx* c, lexp_plan* pl, int mode, int step_index, int kind, int m, uint64_t seed, const lexp_plane* planes,
                         int planes_on_device, lexp_plane* d_planes_out, int flags, int publish_epoch, const int* wait_epochs, unsigned wait_mask) {
    if (!c || !pl || pl->ctx != c || mode < 0 || mode > 1 || step_index < 0) return fail(LEXP_ERR_INVALID, "bad argument");
    if (kind < LEXP_PROP_LIST || kind > LEXP_PROP_RANDOM || m < 0 || m > 120) return fail(LEXP_ERR_INVALID, "bad proposer kind / m");
    if (kind == LEXP_PROP_LIST && !planes) return fail(LEXP_ERR_INVALID, "LEXP_PROP_LIST needs planes");
    if (!pl->d_calls || pl->sync_off < 0) return fail(LEXP_ERR_STATE, "lexp_plan_set_units has not been called for this plan");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    if (c->p.energy_kind != 0) return fail(LEXP_ERR_INVALID, "the device PatchMatch phase is implemented for the cost-volume energy");
    if (publish_epoch < 0 || (wait_mask >> kMaxPeers) || (wait_mask && !wait_epochs)) return fail(LEXP_ERR_INVALID, "bad epoch / mask");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const Plane4* dp = nullptr;
    if (kind == LEXP_PROP_LIST) {
        dp = reinterpret_cast<const Plane4*>(planes);
        if (!planes_on_device) {
            LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
            dp = pl->d_planes;
            c->chain_ok = false;
        }
    }
    PmArgs pm{(flags & LEXP_PM_INIT) ? 2 : 1, kind, m, step_index, (unsigned long long)seed, reinterpret_cast<Plane4*>(d_planes_out),
              publish_epoch, {0, 0, 0, 0, 0, 0, 0, 0}, wait_mask};
    if (wait_epochs)
        for (int i = 0; i < kMaxPeers; i++) pm.wait_epochs[i] = wait_epochs[i];
    return run_plan(c, pl, mode, dp, nullptr, 0, 0, 1, &pm, kind != LEXP_PROP_LIST || (planes_on_device && c->overlap));
}

int lexp_plan_pm_step(lexp_ctx* c, lexp_plan* pl, int mode, int step_index, int kind, int m, uint64_t seed, const lexp_plane* planes,
                      int planes_on_device, lexp_plane* d_planes_out, int flags) {
    return lexp_plan_pm_step_ex(c, pl, mode, step_index, kind, m, seed, planes, planes_on_device, d_planes_out, flags, 0, nullptr, 0u);
}

int lexp_pm_advance_epoch(lexp_ctx* c, int mode, int delta) {
    if (!c || mode < 0 || mode > 1 || delta < 0) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_flags[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    LEXP_LAUNCH(lexp_add_i32, 1, 1, 0, c->stream, c->d_flags[mode] + kMaxPeers, delta);
    LEXP_CUDA(cudaGetLastError());
    c->launches++;
    return LEXP_OK;
}

// ---- pairwise terms and the graph-cut move (lexp_gc.cuh) ------------------------------------------------------------------------------
namespace {
// smoothnessCoeff[mode] on the device (StereoEnergy.h:131-163), rebuilt after lexp_set_image / lexp_set_smoothness.  Caller holds c->mu.
int ensure_coef(lexp_ctx* c, int mode) {
    if (c->coef_valid[mode]) return LEXP_OK;
    if (!c->d_guide[mode]) return fail(LEXP_ERR_STATE, "image of this view not set");
    const int H = c->p.height, W = c->p.width;
    if (!c->d_coef[mode]) LEXP_CUDA(cudaMalloc(&c->d_coef[mode], (size_t)H * W * sizeof(float4)));
    dim3 blk(128), grd((W + 127) / 128, H);
    LEXP_LAUNCH(lexp_smooth_coeff_kernel, grd, blk, 0, c->stream, c->d_guide[mode], c->d_coef[mode], H, W, c->sm_omega, c->sm_eps);
    LEXP_CUDA(cudaGetLastError());
    c->launches++;
    c->coef_valid[mode] = true;
    return LEXP_OK;
}
int upload_gc_cells(lexp_ctx* c, int n, const lexp_rect* regions, GcCell** d_cells, long long* nodes) {
    std::vector<GcCell> h((size_t)n);
    long long at = 0;
    for (int i = 0; i < n; i++) {
        h[i] = GcCell{regions[i].x, regions[i].y, regions[i].width, regions[i].height, at};
        at += (long long)regions[i].width * regions[i].height;
    }
    LEXP_CUDA(cudaMalloc(d_cells, (size_t)n * sizeof(GcCell)));
    LEXP_CUDA(cudaMemcpyAsync(*d_cells, h.data(), (size_t)n * sizeof(GcCell), cudaMemcpyHostToDevice, c->stream));
    LEXP_CUDA(cudaStreamSynchronize(c->stream));   // h is pageable and local
    *nodes = at;
    return LEXP_OK;
}
}  // namespace

namespace {
void gc_phase(int phase, lexp_ctx* c, lexp_plan* pl, const GcParams& gp, const GcPhaseCtl& ctl, int cur) {   // (no template: C linkage block)
#define LEXP_GC_PHASE_CASE(PH) case PH: LEXP_LAUNCH((lexp_gc_phase_kernel<PH>), pl->gc_nblocks, kGcPhaseThreads, 0, c->stream, gp, ctl, cur); break;
    switch (phase) {
        LEXP_GC_PHASE_CASE(GC_PH_BUILD) LEXP_GC_PHASE_CASE(GC_PH_GATHER) LEXP_GC_PHASE_CASE(GC_PH_CLEAR) LEXP_GC_PHASE_CASE(GC_PH_RELAX)
        LEXP_GC_PHASE_CASE(GC_PH_ACTIVE) LEXP_GC_PHASE_CASE(GC_PH_PUSH) LEXP_GC_PHASE_CASE(GC_PH_RELABEL) LEXP_GC_PHASE_CASE(GC_PH_APPLY)
    }
#undef LEXP_GC_PHASE_CASE
    c->launches++;
}
// block map + control block of the phase kernels (once per plan)
int ensure_gc_phase_plan(lexp_ctx* c, lexp_plan* pl) {
    if (pl->d_gc_blocks) return LEXP_OK;
    std::vector<GcBlock> blocks;
    for (int i = 0; i < pl->ncalls; i++) {
        const int n = pl->targ[i].width * pl->targ[i].height;
        for (int first = 0; first < n; first += kGcPhaseThreads) blocks.push_back(GcBlock{i, first});
    }
    pl->gc_nblocks = (int)blocks.size();
    const size_t ints = ((size_t)2 * pl->ncalls + 2 + 1) / 2 * 2;   // done, active, g_flags; doubles follow 8-byte aligned
    if (!c->h_gc_flags) LEXP_CUDA(cudaHostAlloc(&c->h_gc_flags, 2 * sizeof(int), cudaHostAllocDefault));
    GcBlock* d_blocks = nullptr;
    char* d_ctl = nullptr;
    cudaError_t e = cudaMalloc(&d_blocks, blocks.size() * sizeof(GcBlock));
    if (e == cudaSuccess) e = cudaMalloc(&d_ctl, ints * sizeof(int) + 2 * blocks.size() * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_blocks, blocks.data(), blocks.size() * sizeof(GcBlock), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);   // `blocks` is local
    if (e != cudaSuccess) {   // both buffers or neither
        cudaFree(d_blocks); cudaFree(d_ctl); pl->gc_nblocks = 0;
        cudaGetLastError();
        return fail(LEXP_ERR_CUDA, std::string("graph-cut phase plan: ") + cudaGetErrorString(e));
    }
    pl->d_gc_blocks = d_blocks; pl->d_gc_ctl = d_ctl;
    return LEXP_OK;
}
// The expansion moves of a plan with large cells: the phases of lexp_gc_move_kernel as kernels over all SMs, all cells in lockstep, two
// flags read back per decision (lexp_gc.cuh).  Blocking.
int run_gc_phases(lexp_ctx* c, lexp_plan* pl, const GcParams& gp, double* d_flows_out) {
    { int rc = ensure_gc_phase_plan(c, pl); if (rc) return rc; }
    const size_t ints = ((size_t)2 * pl->ncalls + 2 + 1) / 2 * 2;
    int* ibase = reinterpret_cast<int*>(pl->d_gc_ctl);
    GcPhaseCtl ctl{};
    ctl.blocks = pl->d_gc_blocks; ctl.done = ibase; ctl.active = ibase + pl->ncalls; ctl.g_flags = ibase + 2 * pl->ncalls;
    ctl.konst_part = reinterpret_cast<double*>(pl->d_gc_ctl + ints * sizeof(int)); ctl.sink_part = ctl.konst_part + pl->gc_nblocks;
    ctl.ncells = pl->ncalls;
    LEXP_CUDA(cudaMemsetAsync(ibase, 0, ints * sizeof(int), c->stream));
    gc_phase(GC_PH_BUILD, c, pl, gp, ctl, 0);
    auto flag = [&](int which, int* out) -> cudaError_t {   // read a decision flag back (and leave it cleared for the next use)
        cudaError_t e = cudaMemcpyAsync(c->h_gc_flags + which, ctl.g_flags + which, sizeof(int), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(ctl.g_flags + which, 0, sizeof(int), c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        *out = c->h_gc_flags[which];
        return e;
    };
    int cur = 0, rounds = 0;
    for (;;) {
        gc_phase(GC_PH_GATHER, c, pl, gp, ctl, cur);    // global relabelling: pending pushes, then exact distances by relaxation passes
        gc_phase(GC_PH_CLEAR, c, pl, gp, ctl, cur);
        for (int changed = 1; changed;) {
            for (int pass = 0; pass < 8; pass++) gc_phase(GC_PH_RELAX, c, pl, gp, ctl, cur);
            LEXP_CUDA(flag(0, &changed));
        }
        gc_phase(GC_PH_ACTIVE, c, pl, gp, ctl, cur);
        LEXP_LAUNCH(lexp_gc_phase_decide, (pl->ncalls + 127) / 128, 128, 0, c->stream, ctl);
        c->launches++;
        int any_active = 0;
        LEXP_CUDA(flag(1, &any_active));
        if (!any_active) break;
        if (rounds >= c->gc_max_rounds) {   // bounded like every loop of the device path; reported by lexp_pm_get
            const int two = 2;
            LEXP_CUDA(cudaMemcpyAsync(gp.err_flag, &two, sizeof(int), cudaMemcpyHostToDevice, c->stream));
            LEXP_CUDA(cudaStreamSynchronize(c->stream));
            break;
        }
        for (int r = 0; r < c->gc_relabel_every; r++, rounds++) {
            gc_phase(GC_PH_PUSH, c, pl, gp, ctl, cur);
            gc_phase(GC_PH_RELABEL, c, pl, gp, ctl, cur);
            cur ^= 1;
        }
    }
    gc_phase(GC_PH_APPLY, c, pl, gp, ctl, cur);
    if (d_flows_out) {
        LEXP_LAUNCH(lexp_gc_phase_flows, (pl->ncalls + 127) / 128, 128, 0, c->stream, ctl, pl->gc_nblocks, d_flows_out);
        c->launches++;
    }
    LEXP_CUDA(cudaGetLastError());
    return LEXP_OK;
}
}  // namespace

int lexp_set_smoothness(lexp_ctx* c, float lambda, float omega, float th_smooth, float epsilon) {
    if (!c) return fail(LEXP_ERR_INVALID, "null ctx");
    if (!(omega > 0.0f) || !(lambda >= 0.0f) || !(th_smooth >= 0.0f) || !(epsilon >= 0.0f)) return fail(LEXP_ERR_INVALID, "bad smoothness parameters");
    std::lock_guard<std::mutex> lk(c->mu);
    c->sm_lambda = lambda; c->sm_omega = omega; c->sm_th = th_smooth; c->sm_eps = epsilon;
    c->coef_valid[0] = c->coef_valid[1] = false;
    return LEXP_OK;
}

int lexp_get_smooth_coeff(lexp_ctx* c, int mode, float* out8) {
    if (!c || !out8 || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    { int rc = ensure_coef(c, mode); if (rc) return rc; }
    const int H = c->p.height, W = c->p.width;
    const size_t HW = (size_t)H * W;
    float* d8 = nullptr;
    LEXP_CUDA(cudaMalloc(&d8, 8 * HW * sizeof(float)));
    dim3 blk(128), grd((W + 127) / 128, H);
    LEXP_LAUNCH(lexp_smooth_coeff_unpack, grd, blk, 0, c->stream, c->d_coef[mode], d8, H, W);
    c->launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out8, d8, 8 * HW * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d8);
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("get_smooth_coeff: ") + cudaGetErrorString(e));
    return LEXP_OK;
}

int lexp_pairwise_terms(lexp_ctx* c, int mode, int n, const lexp_rect* regions, const lexp_plane* planes, float* out_host) {
    if (!c || !regions || !planes || !out_host || n <= 0 || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_label[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    const int H = c->p.height, W = c->p.width;
    for (int i = 0; i < n; i++)
        if (regions[i].width <= 0 || regions[i].height <= 0 || regions[i].x < 0 || regions[i].y < 0 || regions[i].x + regions[i].width > W ||
            regions[i].y + regions[i].height > H) return fail(LEXP_ERR_INVALID, "region outside the image");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    { int rc = ensure_coef(c, mode); if (rc) return rc; }
    GcCell* d_cells = nullptr;
    Plane4* d_planes = nullptr;
    float* d_out = nullptr;
    long long nodes = 0;
    int rc = upload_gc_cells(c, n, regions, &d_cells, &nodes);
    cudaError_t e = cudaSuccess;
    if (rc == LEXP_OK) {
        e = cudaMalloc(&d_planes, (size_t)n * sizeof(Plane4));
        if (e == cudaSuccess) e = cudaMalloc(&d_out, (size_t)nodes * 12 * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_planes, planes, (size_t)n * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) {
            LEXP_LAUNCH(lexp_pairwise_kernel, n, 256, 0, c->stream, d_cells, d_planes, c->d_cur_label[mode], c->d_coef[mode], d_out, H, W, c->sm_lambda, c->sm_th);
            c->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(out_host, d_out, (size_t)nodes * 12 * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    cudaFree(d_cells); cudaFree(d_planes); cudaFree(d_out);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("pairwise_terms: ") + cudaGetErrorString(e));
    return LEXP_OK;
}

int lexp_plan_init_step(lexp_ctx* c, lexp_plan* pl, int mode, const lexp_plane* planes, int planes_on_device) {
    if (!c || !pl || pl->ctx != c || !planes || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    c->chain_ok = false;   // copies / other kernels around the fused launch: it is an ordinary one
    const int H = c->p.height, W = c->p.width;
    if (!c->d_prop_cost[mode]) LEXP_CUDA(cudaMalloc(&c->d_prop_cost[mode], (size_t)H * W * sizeof(float)));
    if (!pl->d_gc_cells) {
        int rc = upload_gc_cells(c, pl->ncalls, pl->targ.data(), &pl->d_gc_cells, &pl->gc_nodes);
        if (rc) return rc;
        for (const lexp_rect& t : pl->targ) pl->gc_max_nodes = std::max(pl->gc_max_nodes, t.width * t.height);
    }
    const Plane4* dp = reinterpret_cast<const Plane4*>(planes);
    if (!planes_on_device) {
        LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
        dp = pl->d_planes;
    }
    { int rc = run_plan(c, pl, mode, dp, c->d_prop_cost[mode], W, 0, 1); if (rc) return rc; }   // ComputeUnaryPotential (:111)
    c->chain_ok = false;
    LEXP_LAUNCH(lexp_gc_assign_kernel, pl->ncalls, 256, 0, c->stream, pl->d_gc_cells, dp, c->d_prop_cost[mode], c->d_cur_cost[mode], c->d_cur_label[mode], W);
    LEXP_CUDA(cudaGetLastError());
    c->launches++;
    return LEXP_OK;
}

int lexp_get_disparities(lexp_ctx* c, int mode, float* out_host) {
    if (!c || !out_host || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_label[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    const int H = c->p.height, W = c->p.width;
    float* d = nullptr;
    LEXP_CUDA(cudaMalloc(&d, (size_t)H * W * sizeof(float)));
    dim3 blk(128), grd((W + 127) / 128, H);
    LEXP_LAUNCH(lexp_disparity_kernel, grd, blk, 0, c->stream, c->d_cur_label[mode], d, H, W);
    c->launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_host, d, (size_t)H * W * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("lexp_get_disparities: ") + cudaGetErrorString(e));
    return LEXP_OK;
}

// cvutils::io::save_pfm_file (Utilities.hpp:84-137) for a 1-channel float image: "Pf\n<w> <h>\n<-1/255 as %lf>\n", rows bottom-up, native
// (little-endian) floats -- the file main.cpp:319,410 writes as disp0.pfm.
int lexp_save_pfm(const char* path, const float* image, int width, int height, ptrdiff_t step_bytes) {
    if (!path || !image || width <= 0 || height <= 0 || step_bytes < (ptrdiff_t)width * 4) return fail(LEXP_ERR_INVALID, "bad argument");
    FILE* f = fopen(path, "wb");
    if (!f) return fail(LEXP_ERR_INVALID, std::string("cannot open for writing: ") + path);
    fprintf(f, "Pf\n%d %d\n%lf\n", width, height, -1.0 / 255.0);
    bool ok = true;
    for (int y = height - 1; y >= 0 && ok; y--)   // pfm stores rows in inverse order
        ok = fwrite(reinterpret_cast<const char*>(image) + (ptrdiff_t)y * step_bytes, sizeof(float), (size_t)width, f) == (size_t)width;
    ok = (fclose(f) == 0) && ok;
    return ok ? LEXP_OK : fail(LEXP_ERR_INVALID, std::string("write failed: ") + path);
}

int lexp_energy(lexp_ctx* c, int mode, double* data_term, double* smoothness_term) {
    if (!c || mode < 0 || mode > 1 || (!data_term && !smoothness_term)) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    std::lock_guard<std::mutex> lk(c->mu);
    c->chain_ok = false;   // copies / other kernels follow on the stream: the next fused launch is an ordinary one
    LEXP_CUDA(cudaSetDevice(c->p.device));
    { int rc = ensure_coef(c, mode); if (rc) return rc; }
    const int H = c->p.height, W = c->p.width;
    const int nblocks = (int)(((size_t)H * W + 255) / 256);
    double* d_part = nullptr;
    LEXP_CUDA(cudaMalloc(&d_part, (2 * (size_t)nblocks + 2) * sizeof(double)));
    LEXP_LAUNCH(lexp_energy_kernel, nblocks, 256, 0, c->stream, c->d_cur_cost[mode], c->d_cur_label[mode], c->d_coef[mode], d_part, H, W, c->sm_lambda, c->sm_th);
    LEXP_LAUNCH(lexp_energy_finish, 1, 1, 0, c->stream, d_part, nblocks, d_part + 2 * (size_t)nblocks);
    c->launches += 2;
    double h[2] = {0.0, 0.0};
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, d_part + 2 * (size_t)nblocks, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_part);
    if (e != cudaSuccess) return fail(LEXP_ERR_CUDA, std::string("lexp_energy: ") + cudaGetErrorString(e));
    if (data_term) *data_term = h[0];
    if (smoothness_term) *smoothness_term = h[1];
    return LEXP_OK;
}

int lexp_plan_gc_step(lexp_ctx* c, lexp_plan* pl, int mode, int kind, int m, uint64_t seed, const lexp_plane* planes, int planes_on_device,
                      lexp_plane* d_planes_out, double* d_flows_out) {
    if (!c || !pl || pl->ctx != c || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (kind < LEXP_PROP_LIST || kind > LEXP_PROP_RANDOM || m < 0 || m > 120) return fail(LEXP_ERR_INVALID, "bad proposer kind / m");
    if (kind == LEXP_PROP_LIST && !planes) return fail(LEXP_ERR_INVALID, "LEXP_PROP_LIST needs planes");
    if (!pl->d_calls) return fail(LEXP_ERR_STATE, "lexp_plan_set_units has not been called for this plan");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    c->chain_ok = false;   // copies / other kernels around the fused launch: it is an ordinary one
    { int rc = ensure_coef(c, mode); if (rc) return rc; }
    const int H = c->p.height, W = c->p.width;
    if (!c->d_prop_cost[mode]) LEXP_CUDA(cudaMalloc(&c->d_prop_cost[mode], (size_t)H * W * sizeof(float)));
    if (!pl->d_gc_cells) {
        int rc = upload_gc_cells(c, pl->ncalls, pl->targ.data(), &pl->d_gc_cells, &pl->gc_nodes);
        if (rc) return rc;
        for (const lexp_rect& t : pl->targ) pl->gc_max_nodes = std::max(pl->gc_max_nodes, t.width * t.height);
    }
    if (pl->gc_nodes > c->gc_scratch_nodes) {   // the residual network of the largest group so far
        LEXP_CUDA(cudaStreamSynchronize(c->stream));
        cudaFree(c->d_gc_scratch); c->d_gc_scratch = nullptr; c->gc_scratch_nodes = 0;
        LEXP_CUDA(cudaMalloc(&c->d_gc_scratch, (size_t)pl->gc_nodes * kGcWords * sizeof(float)));
        c->gc_scratch_nodes = pl->gc_nodes;
    }
    // (1) the proposals (FastGCStereo.h:47): the PatchMatch phase's device proposers, or the caller's list
    Plane4* dp = pl->d_planes;
    if (kind == LEXP_PROP_LIST) {
        if (planes_on_device) dp = const_cast<Plane4*>(reinterpret_cast<const Plane4*>(planes));
        else LEXP_CUDA(cudaMemcpyAsync(pl->d_planes, planes, (size_t)pl->ncalls * sizeof(Plane4), cudaMemcpyHostToDevice, c->stream));
    }
    if (kind != LEXP_PROP_LIST || d_planes_out) {
        LEXP_LAUNCH(lexp_gc_propose_kernel, (pl->ncalls + 127) / 128, 128, 0, c->stream, pl->d_calls, pl->ncalls, dp, reinterpret_cast<Plane4*>(d_planes_out),
                    (unsigned long long)seed, c->d_cur_label[mode], W, kind, m, c->p.min_disp, c->p.max_disp);
        LEXP_CUDA(cudaGetLastError());
        c->launches++;
    }
    // (2) ComputeUnaryPotential(filterRegion, sharedRegion, proposalCost(filterRegion), label) (:49)
    { int rc = run_plan(c, pl, mode, dp, c->d_prop_cost[mode], W, 0, 1); if (rc) return rc; }
    c->chain_ok = false;
    // (3) expansionMoveBK + copyTo / setTo (:53-59)
    GcParams gp{};
    gp.cells = pl->d_gc_cells; gp.planes = dp; gp.prop_cost = c->d_prop_cost[mode];
    gp.cur_cost = c->d_cur_cost[mode]; gp.cur_label = c->d_cur_label[mode]; gp.coef = c->d_coef[mode];
    gp.scratch = c->d_gc_scratch; gp.scratch_nodes = c->gc_scratch_nodes;
    gp.flows_out = d_flows_out; gp.iters_out = nullptr; gp.err_flag = c->d_flags[mode] + kMaxPeers + 1;
    gp.H = H; gp.W = W; gp.lambda = c->sm_lambda; gp.th_smooth = c->sm_th;
    gp.relabel_every = c->gc_relabel_every; gp.max_rounds = c->gc_max_rounds;
    if (pl->gc_max_nodes > c->gc_big_nodes) return run_gc_phases(c, pl, gp, d_flows_out);   // large cells: phase kernels over all SMs (blocking)
    LEXP_LAUNCH(lexp_gc_move_kernel, pl->ncalls, c->gc_threads, 0, c->stream, gp);
    LEXP_CUDA(cudaGetLastError());
    c->launches++;
    return LEXP_OK;
}

int lexp_pm_ipc_export(lexp_ctx* c, int mode, void* out) {
    if (!c || !out || mode < 0 || mode > 1) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
#ifdef LEXP_EMU
    return fail(LEXP_ERR_INVALID, "no inter-process memory on the emulator");
#else
    static_assert(sizeof(cudaIpcMemHandle_t) == 64 && LEXP_PM_IPC_BYTES == 3 * 64, "handle layout");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    cudaIpcMemHandle_t* h = reinterpret_cast<cudaIpcMemHandle_t*>(out);
    LEXP_CUDA(cudaIpcGetMemHandle(&h[0], c->d_cur_cost[mode]));
    LEXP_CUDA(cudaIpcGetMemHandle(&h[1], c->d_cur_label[mode]));
    LEXP_CUDA(cudaIpcGetMemHandle(&h[2], c->d_flags[mode]));
    return LEXP_OK;
#endif
}

int lexp_pm_ipc_connect(lexp_ctx* c, int mode, int rank, int world, const void* all) {
    if (!c || !all || mode < 0 || mode > 1 || world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return fail(LEXP_ERR_INVALID, "bad argument");
    if (!c->d_cur_cost[mode]) return fail(LEXP_ERR_STATE, "lexp_pm_begin has not been called for this view");
#ifdef LEXP_EMU
    return fail(LEXP_ERR_INVALID, "no inter-process memory on the emulator");
#else
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    lexp_ctx::Peers& pr = c->peers[mode];
    for (int i = 0; i < pr.n_opened; i++) cudaIpcCloseMemHandle(pr.ipc_opened[i]);
    pr = lexp_ctx::Peers();
    const cudaIpcMemHandle_t* h = reinterpret_cast<const cudaIpcMemHandle_t*>(all);
    int slot = 1;   // entry 0 is this rank's own copy
    for (int r = 0; r < world; r++) {
        if (r == rank) continue;
        void* p[3];
        for (int k = 0; k < 3; k++) {
            LEXP_CUDA(cudaIpcOpenMemHandle(&p[k], h[3 * r + k], cudaIpcMemLazyEnablePeerAccess));
            pr.ipc_opened[pr.n_opened++] = p[k];
        }
        pr.cost[slot] = (float*)p[0]; pr.label[slot] = (float4*)p[1]; pr.flags[slot] = (int*)p[2];
        slot++;
    }
    pr.world = world; pr.rank = rank;
    return LEXP_OK;
#endif
}

int lexp_pm_connect_local(lexp_ctx* c, int mode, int rank, int world, lexp_ctx* const* peer_ctx) {
    if (!c || !peer_ctx || mode < 0 || mode > 1 || world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return fail(LEXP_ERR_INVALID, "bad argument");
    if (peer_ctx[rank] != c) return fail(LEXP_ERR_INVALID, "peer_contexts[rank] must be this context");
    std::lock_guard<std::mutex> lk(c->mu);
    LEXP_CUDA(cudaSetDevice(c->p.device));
    lexp_ctx::Peers pr;
    int slot = 1;
    for (int r = 0; r < world; r++) {
        if (r == rank) continue;
        lexp_ctx* o = peer_ctx[r];
        if (!o || !o->d_cur_cost[mode] || o->p.height != c->p.height || o->p.width != c->p.width)
            return fail(LEXP_ERR_STATE, "peer context without a PatchMatch-phase state of the same size");
#ifndef LEXP_EMU
        if (o->p.device != c->p.device) {
            cudaError_t e = cudaDeviceEnablePeerAccess(o->p.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(LEXP_ERR_CUDA, std::string("peer access: ") + cudaGetErrorString(e));
            cudaGetLastError();
        }
#endif
        pr.cost[slot] = o->d_cur_cost[mode]; pr.label[slot] = o->d_cur_label[mode]; pr.flags[slot] = o->d_flags[mode];
        slot++;
    }
    pr.world = world; pr.rank = rank;
    c->peers[mode] = pr;
    return LEXP_OK;
}

// ---- the PatchMatch phase as one object (host-side schedule of FastGCStereo.h:143-157 around lexp_plan_pm_step_ex) -----------
struct lexp_pm_sweep {
    lexp_ctx* ctx = nullptr;
    int mode = 0, rank = 0, world = 1;
    struct Group { lexp_plan* plan; int layer, group; std::vector<int> owners; };
    std::vector<Group> sched;                                  // every (layer, group) in order, the same on all ranks
    std::vector<std::vector<std::pair<int, int>>> proposers;   // per layer: (kind, K)
    lexp_plan* init_plan = nullptr;
    std::vector<int> init_owners, init_index;                  // ranks that initialise units; this rank's units of layer 0
    int n_init = 0;
    int rel = 0;                                               // groups issued since the epoch base was last advanced
    int last_rel[kMaxPeers];
    bool has[kMaxPeers];
};

namespace {
// random stream of one launch (= localexpstereo_b200.sweep.pm_seed)
uint64_t pm_launch_seed(uint64_t base, int mode, int iteration, int layer, int group, int step) {
    uint64_t z = base * 0x9E3779B97F4A7C15ull + (uint64_t)(mode + 1) * 0xD1B54A32D192ED03ull + (uint64_t)(iteration + 1) * 0x8CB92BA72F3D8DD7ull +
                 (uint64_t)(layer + 1) * 0xABC98388FB8FAC03ull + (uint64_t)(group + 1) * 0x2545F4914F6CDD1Dull + (uint64_t)(step + 1) * 0xDA942042E4DD58B5ull;
    z = (z ^ (z >> 33)) * 0xFF51AFD7ED558CCDull;
    return z ^ (z >> 29);
}
int sweep_step(lexp_pm_sweep* s, lexp_plan* plan, int step_index, int kind, int m, uint64_t seed, const lexp_plane* planes, int flags, bool first, bool last) {
    int we[kMaxPeers];
    unsigned mask = 0;
    for (int r = 0; r < kMaxPeers; r++) { we[r] = s->has[r] ? s->last_rel[r] : 0; if (first && s->has[r]) mask |= 1u << r; }
    return lexp_plan_pm_step_ex(s->ctx, plan, s->mode, step_index, kind, m, seed, planes, 0, nullptr, flags, last ? s->rel + 1 : 0, we, mask);
}
void sweep_group_done(lexp_pm_sweep* s, const std::vector<int>& owners) {
    s->rel++;
    for (int r : owners) { s->last_rel[r] = s->rel; s->has[r] = true; }
}
int sweep_advance(lexp_pm_sweep* s) {
    const int delta = s->rel;
    for (int r = 0; r < kMaxPeers; r++) s->last_rel[r] -= delta;
    s->rel = 0;
    return lexp_pm_advance_epoch(s->ctx, s->mode, delta);
}
}  // namespace

int lexp_pm_sweep_create(lexp_ctx* c, int mode, int n_layers, const int* unit_sizes, const int* n_prop, const int* prop_kind, const int* prop_K,
                         int rank, int world, lexp_pm_sweep** out) {
    if (!c || !unit_sizes || !n_prop || !prop_kind || !prop_K || !out || n_layers < 1 || mode < 0 || mode > 1 || world < 1 || world > kMaxPeers ||
        rank < 0 || rank >= world)
        return fail(LEXP_ERR_INVALID, "bad argument");
    auto s = std::unique_ptr<lexp_pm_sweep>(new lexp_pm_sweep());
    s->ctx = c; s->mode = mode; s->rank = rank; s->world = world;
    for (int r = 0; r < kMaxPeers; r++) { s->last_rel[r] = 0; s->has[r] = false; }
    const int W = c->p.width, H = c->p.height, windR = c->p.windR;
    int cell_base = 0, pk = 0;
    auto cleanup = [&]() { for (auto& g : s->sched) lexp_plan_destroy(g.plan); lexp_plan_destroy(s->init_plan); };
    for (int li = 0; li < n_layers; li++) {
        s->proposers.emplace_back();
        for (int j = 0; j < n_prop[li]; j++, pk++) {
            if ((prop_kind[pk] != LEXP_PROP_EXPANSION && prop_kind[pk] != LEXP_PROP_RANDOM) || prop_K[pk] < 0) { cleanup(); return fail(LEXP_ERR_INVALID, "proposer kinds: LEXP_PROP_EXPANSION / LEXP_PROP_RANDOM"); }
            s->proposers.back().push_back({prop_kind[pk], prop_K[pk]});
        }
        int hb = 0, wb = 0;
        int rc = lexp_layer_geometry(W, H, windR, unit_sizes[li], &hb, &wb, nullptr, nullptr, nullptr, nullptr);
        if (rc) { cleanup(); return rc; }
        const int n = hb * wb;
        std::vector<lexp_rect> unit(n), shared(n), filt(n);
        std::vector<int> group_of(n);
        rc = lexp_layer_geometry(W, H, windR, unit_sizes[li], &hb, &wb, unit.data(), shared.data(), filt.data(), group_of.data());
        if (rc) { cleanup(); return rc; }
        for (int g = 0; g < 16; g++) {   // disjointRegionSets in group order, empty ones erased (LayerManager.h:168-182)
            std::vector<int> cells;
            for (int r = 0; r < n; r++) if (group_of[r] == g) cells.push_back(r);
            if (cells.empty()) continue;
            lexp_pm_sweep::Group G{nullptr, li, (int)std::count_if(s->sched.begin(), s->sched.end(), [li](const lexp_pm_sweep::Group& x) { return x.layer == li; }), {}};
            for (int r = 0; r < world; r++) if ((int)cells.size() > r) G.owners.push_back(r);   // round-robin deal: rank r owns cells[r::world]
            std::vector<lexp_rect> f, t, u;
            std::vector<int> ids;
            for (size_t k = (size_t)rank; k < cells.size(); k += (size_t)world) { f.push_back(filt[cells[k]]); t.push_back(shared[cells[k]]); u.push_back(unit[cells[k]]); ids.push_back(cell_base + cells[k]); }
            if (!f.empty()) {
                rc = lexp_plan_create(c, (int)f.size(), f.data(), t.data(), &G.plan);
                if (!rc) rc = lexp_plan_set_units(G.plan, u.data(), ids.data());
                if (rc) { lexp_plan_destroy(G.plan); cleanup(); return rc; }
            }
            s->sched.push_back(G);
        }
        if (li == 0) {   // initCurrentFast: filterRegion = unit +- windR (FastGCStereo.h:109-110)
            s->n_init = n;
            std::vector<lexp_rect> f, u;
            for (int r = rank; r < n; r += world) {
                const lexp_rect& q = unit[r];
                const int x0 = std::max(q.x - windR, 0), y0 = std::max(q.y - windR, 0), x1 = std::min(q.x + q.width + windR, W), y1 = std::min(q.y + q.height + windR, H);
                f.push_back(lexp_rect{x0, y0, x1 - x0, y1 - y0}); u.push_back(q); s->init_index.push_back(r);
            }
            for (int r = 0; r < world; r++) if (n > r) s->init_owners.push_back(r);
            if (!f.empty()) {
                rc = lexp_plan_create(c, (int)f.size(), f.data(), u.data(), &s->init_plan);
                if (!rc) rc = lexp_plan_set_units(s->init_plan, u.data(), s->init_index.data());
                if (rc) { cleanup(); return rc; }
            }
        }
        cell_base += n;
    }
    *out = s.release();
    return LEXP_OK;
}

int lexp_pm_sweep_destroy(lexp_pm_sweep* s) {
    if (!s) return LEXP_OK;
    for (auto& g : s->sched) lexp_plan_destroy(g.plan);
    lexp_plan_destroy(s->init_plan);
    delete s;
    return LEXP_OK;
}

int lexp_pm_sweep_num_init_labels(const lexp_pm_sweep* s) { return s ? s->n_init : 0; }

int lexp_pm_sweep_init(lexp_pm_sweep* s, const lexp_plane* labels) {
    if (!s || !labels) return fail(LEXP_ERR_INVALID, "bad argument");
    int rc = lexp_pm_reset_sync(s->ctx);
    if (rc) return rc;
    if (s->init_plan) {
        std::vector<lexp_plane> mine;
        for (int r : s->init_index) mine.push_back(labels[r]);
        if (s->ctx->p.energy_kind != 0) {   // the image-based energy has no PatchMatch-phase kernel: unary launch + assignment (single GPU)
            if (s->world != 1) return fail(LEXP_ERR_INVALID, "the image-based energy runs on one GPU");
            rc = lexp_plan_init_step(s->ctx, s->init_plan, s->mode, mine.data(), 0);
            if (rc == LEXP_OK) rc = lexp_sync(s->ctx);   // `mine` is local and pageable
            return rc;
        }
        rc = sweep_step(s, s->init_plan, 0, LEXP_PROP_LIST, 0, 0, mine.data(), LEXP_PM_INIT, true, true);
        if (rc) return rc;
    }
    sweep_group_done(s, s->init_owners);
    return sweep_advance(s);
}

int lexp_pm_sweep_iteration(lexp_pm_sweep* s, int iteration, uint64_t seed, int* n_launches) {
    if (!s || iteration < 0) return fail(LEXP_ERR_INVALID, "bad argument");
    int rc = lexp_pm_reset_sync(s->ctx);
    if (rc) return rc;
    const float range = s->ctx->p.max_disp - s->ctx->p.min_disp;
    int launches = 0;
    for (auto& g : s->sched) {
        std::vector<std::pair<int, int>> steps;   // (kind, m) as the `while (prop->isContinued())` loops produce them (FastGCStereo.h:41-46)
        for (auto& pr : s->proposers[g.layer])
            for (int it = 0; it < pr.second; it++) {
                if (pr.first == LEXP_PROP_RANDOM && (double)(range * exp2f(-(float)(iteration + it + 1))) < 0.1) break;   // Proposer.h:149-152
                steps.push_back({pr.first, pr.first == LEXP_PROP_RANDOM ? iteration + it : 0});
            }
        if (steps.empty()) { sweep_group_done(s, {}); continue; }   // every proposer stopped early: no rank launches or publishes anything
        if (g.plan) {
            for (size_t k = 0; k < steps.size(); k++) {
                rc = sweep_step(s, g.plan, (int)k, steps[k].first, steps[k].second, pm_launch_seed(seed, s->mode, iteration, g.layer, g.group, (int)k), nullptr, 0,
                                k == 0, k + 1 == steps.size());
                if (rc) return rc;
                launches++;
            }
        }
        sweep_group_done(s, g.owners);
    }
    if (n_launches) *n_launches = launches;
    return sweep_advance(s);
}

// One iteration of the main loop of FastGCStereo::run (FastGCStereo.h:171-184, doGC == true) over the sweep's schedule: every proposal
// step is lexp_plan_gc_step (proposals -> unary costs -> expansionMoveBK -> copyTo / setTo), ordered by the stream.  Single GPU.
int lexp_pm_sweep_gc_iteration(lexp_pm_sweep* s, int iteration, uint64_t seed, int* n_steps) {
    if (!s || iteration < 0) return fail(LEXP_ERR_INVALID, "bad argument");
    if (s->world != 1) return fail(LEXP_ERR_INVALID, "the graph-cut iterations run on one GPU (the cell shard covers the PatchMatch phase)");
    const float range = s->ctx->p.max_disp - s->ctx->p.min_disp;
    int steps_done = 0;
    for (auto& g : s->sched) {
        if (!g.plan) continue;
        int k = 0;
        for (auto& pr : s->proposers[g.layer])
            for (int it = 0; it < pr.second; it++, k++) {
                if (pr.first == LEXP_PROP_RANDOM && (double)(range * exp2f(-(float)(iteration + it + 1))) < 0.1) break;   // Proposer.h:149-152
                const int rc = lexp_plan_gc_step(s->ctx, g.plan, s->mode, pr.first, pr.first == LEXP_PROP_RANDOM ? iteration + it : 0,
                                                 pm_launch_seed(seed, s->mode, iteration, g.layer, g.group, k), nullptr, 0, nullptr, nullptr);
                if (rc) return rc;
                steps_done++;
            }
    }
    if (n_steps) *n_steps = steps_done;
    return LEXP_OK;
}

// LayerManager::addLayer, LayerManager.h:88-185 (the #else branch that merges small edge cells).
int lexp_layer_geometry(int width, int height, int windR, int u, int* hb_out, int* wb_out, lexp_rect* unit, lexp_rect* shared,
                        lexp_rect* filt, int* group_of) {
    if (width <= 0 || height <= 0 || u <= 0 || windR < 0) return fail(LEXP_ERR_INVALID, "bad layer arguments");
    const int minsize = std::max(2, u / 2);
    const int frac_h = height % u, frac_w = width % u;
    const int split_h = frac_h >= minsize ? 1 : 0, split_w = frac_w >= minsize ? 1 : 0;
    const int hb = height / u + split_h, wb = width / u + split_w;
    if (hb_out) *hb_out = hb;
    if (wb_out) *wb_out = wb;
    if (!unit || !shared || !filt) return LEXP_OK;
    auto clip = [&](int x, int y, int w, int h) {
        const int x0 = std::max(x, 0), y0 = std::max(y, 0), x1 = std::min(x + w, width), y1 = std::min(y + h, height);
        lexp_rect r{0, 0, 0, 0};
        if (x1 > x0 && y1 > y0) { r.x = x0; r.y = y0; r.width = x1 - x0; r.height = y1 - y0; }
        return r;
    };
    for (int i = 0; i < hb; i++)
        for (int j = 0; j < wb; j++) {
            const int r = i * wb + j;
            unit[r] = clip(j * u, i * u, u, u);
            shared[r] = clip((j - 1) * u, (i - 1) * u, 3 * u, 3 * u);
            filt[r] = clip((j - 1) * u - windR, (i - 1) * u - windR, 3 * u + 2 * windR, 3 * u + 2 * windR);
            if (group_of) group_of[r] = (i % 4) * 4 + (j % 4);
        }
    if (!split_w) {
        for (int i = 0; i < hb; i++) unit[i * wb + wb - 1].width += frac_w;
        if (wb >= 2)
            for (int i = 0; i < hb; i++) {
                const int r = i * wb + wb - 2;
                shared[r].width += frac_w;
                filt[r] = clip(filt[r].x, filt[r].y, filt[r].width + frac_w, filt[r].height);
            }
    }
    if (!split_h) {
        for (int j = 0; j < wb; j++) unit[(hb - 1) * wb + j].height += frac_h;
        if (hb >= 2)
            for (int j = 0; j < wb; j++) {
                const int r = (hb - 2) * wb + j;
                shared[r].height += frac_h;
                filt[r] = clip(filt[r].x, filt[r].y, filt[r].width, filt[r].height + frac_h);
            }
    }
    return LEXP_OK;
}

}  // extern "C"
