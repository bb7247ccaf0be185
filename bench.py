#!/usr/bin/env python
"""bench.py -- plane-hypothesis cost evals/sec of the unary-cost hot path (BASELINE.json metric).

A *step* is one local-expansion sweep over one view: 3 layers x <=16 disjoint groups x K proposal
steps = 240 batched evaluations (FastGCStereo.h:22-72), on synthetic inputs of the shape
BASELINE.json names.  `value` = filterRect-pixel evals of the whole job / device time, inputs
resident in HBM.  `e2e` = same sweep through the host-buffer API (planes H2D, costs D2H).
`--impl reference` times the reference's CPU implementation on the host cores: oracle/_ref (the reference's own
CostVolumeEnergy / NaiveStereoEnergy classes compiled from its headers by oracle/build_ref.py, kind "reference",
driven by the OpenMP loop of FastGCStereo.h:30-49); the plain-C restatement oracle/lexp_oracle.c (kind "port") stands in
when oracle/_ref is absent, and its rate is reported next to the reference's in the `sample` note.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (W, H, D, windR)   -- BASELINE.json configs[2] / [1] / [4]
    "synthetic_2048x1536x256_r20": (2048, 1536, 256, 20),
    "adirondack_shape_1436x992x290_r20": (1436, 992, 290, 20),
    "synthetic_4k_3840x2160x512_r32": (3840, 2160, 512, 32),
    "tiny_450x375x64_r20": (450, 375, 64, 20),
    "middv2_cones_shape_450x375x64_naive": (450, 375, 64, 20),   # configs[0]: NaiveStereoEnergy, layers 5/15/25 (main.cpp:304-306)
    "probe_2048x1536x16_r20": (2048, 1536, 16, 20),   # TLB / DRAM-locality probe (not a BASELINE config)
}
TH_COL, EPS = 0.5, 1e-4  # main.cpp:26,351 / main.cpp:73
METRIC = "plane-hypothesis cost evals/sec"
UNIT = "evals/s"


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def pick_threads(run_once):
    """The CPU arm gets its best thread count: all hardware threads or one per core pair, whichever is faster here
    (torchrun exports OMP_NUM_THREADS=1, so the count is always passed explicitly)."""
    n = host_threads()
    best, best_t = n, None
    for cand in sorted({n, max(1, n // 2)}, reverse=True):
        run_once(cand)  # warm
        dt = None
        for _ in range(3):  # best of 3: single trials are noisy on a shared host
            t0 = time.perf_counter()
            run_once(cand)
            d = time.perf_counter() - t0
            dt = d if dt is None else min(dt, d)
        if best_t is None or dt < best_t:
            best, best_t = cand, dt
    return best


def make_inputs(W, H, D, need_right=False):
    from localexpstereo_b200 import synth
    imL = synth.synthetic_image(H, W, 42)
    rng = np.random.default_rng(1234)
    vol = rng.random((D, H, W), dtype=np.float32)
    return imL, vol


DUMP_LIMIT_BYTES = 60 << 20   # data of all dumped arrays; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes what the timed path computed as out_dir/<name>.npy (float32), so that two builds can be compared output for output.
    Arrays whose first axes are the image's H x W: when all of them together exceed DUMP_LIMIT_BYTES, the same seeded sample of
    pixels (np.random.default_rng(0), ascending raster order) is taken from every one of them."""
    os.makedirs(out_dir, exist_ok=True)
    H, W = next(iter(arrays.values())).shape[:2]
    total = sum(a.size * 4 for a in arrays.values())
    idx = None
    if total > DUMP_LIMIT_BYTES:
        n = int(H * W * DUMP_LIMIT_BYTES // total)
        idx = np.sort(np.random.default_rng(0).choice(H * W, n, replace=False))
    for name, a in arrays.items():
        a = np.asarray(a, np.float32)
        if idx is not None:
            a = a.reshape((H * W,) + a.shape[2:])[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def all_planes(sweep, D):
    from localexpstereo_b200 import synth
    per_layer = [synth.synthetic_planes(sweep.layer(li).unitRegions, sweep.steps[li], D, 7 + li) for li in range(len(sweep.steps))]
    return [np.ascontiguousarray(per_layer[g.layer][:, g.cells, :]) for g in sweep.groups]  # [K][n][4] per group plan


# ---------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's CPU implementation of the path, for timing only (never on the product path).

    kind "reference": oracle/_ref/liblexp_ref.so -- the reference's own classes compiled from its headers over the cv:: layer
    of oracle/cvshim (its box filter is that layer's, not OpenCV's hand-vectorised one), cells of a group in an OpenMP
    parallel for with one Reusable per cell across its K proposals, exactly the loop of FastGCStereo.h:30-49 minus fusion.
    kind "port": oracle/lexp_oracle.c, the plain-C restatement (running-sum box filter, per-thread scratch).
    Both are calibrated on one group (rates in the `sample` note); the compiled reference is the one timed whenever it is
    available, at its better thread count; the port stands in when oracle/_ref is absent."""

    def __init__(self, W, H, D, windR, imL, vol, naive=False, imR=None):
        self.W, self.H, self.naive = W, H, naive
        self.out = np.zeros((H, W), np.float32)
        self.arms = {}
        try:
            from oracle import ref_binding
            if ref_binding.available() or ref_binding.build_ref.reference_present():
                if naive:
                    self.arms["reference"] = ref_binding.RefEnergy(imL, imR if imR is not None else imL, windR=windR, eps=EPS, th_col=10.0, th_grad=2.0,
                                                                   alpha=0.9, max_disp=D - 1, min_disp=0.0, kind=1)
                else:
                    self.arms["reference"] = ref_binding.RefEnergy(imL, imL, vol, vol, windR=windR, eps=EPS, th_col=TH_COL, max_disp=D - 1, min_disp=0.0, kind=0)
        except Exception as e:  # the prebuilt library is optional on the GPU box
            print(f"[bench] oracle/_ref unavailable ({e}); CPU arm = port", file=sys.stderr)
        if not naive:
            from oracle.c_oracle import COracle
            orc = COracle(H, W, D, windR, EPS, TH_COL, D - 1)
            orc.set_image(0, imL)
            orc.set_volume(0, vol)
            self.arms["port"] = orc
        if not self.arms:
            raise RuntimeError("no CPU implementation available for this workload")
        self.kind, self.nthr, self.calib = None, None, {}

    def run_group(self, kind, fr, tr, planes_kn4, nthr):
        """planes_kn4: [K][n][4] -- all K proposal steps of one disjoint group."""
        if kind == "reference":
            self.arms[kind].unary_group(fr, tr, np.ascontiguousarray(np.transpose(planes_kn4, (1, 0, 2))), 0, True, self.out, nthr)
        else:
            for k in range(planes_kn4.shape[0]):
                self.arms[kind].unary_batch(0, fr, tr, planes_kn4[k], self.out, True, nthr)

    def calibrate(self, fr, tr, planes_kn4):
        evals = sum(f[2] * f[3] for f in fr) * planes_kn4.shape[0]
        best = None
        for kind in self.arms:
            nthr = pick_threads(lambda n: self.run_group(kind, fr, tr, planes_kn4, n))
            t0 = time.perf_counter()
            self.run_group(kind, fr, tr, planes_kn4, nthr)
            rate = evals / (time.perf_counter() - t0)
            self.calib[kind] = {"evals_per_s": rate, "threads": nthr}
            if best is None or rate > best[0]:
                best = (rate, kind, nthr)
        # the reference's own code is the baseline whenever it is available (its calibration rate and the port's are both
        # reported in the `sample` note); the port only stands in when oracle/_ref is absent
        if "reference" in self.calib:
            self.kind, self.nthr = "reference", self.calib["reference"]["threads"]
        else:
            _, self.kind, self.nthr = best
        return self.kind, self.nthr

    def run(self, fr, tr, planes_kn4):
        self.run_group(self.kind, fr, tr, planes_kn4, self.nthr)

    def time_sample(self, sample):
        """sample: [(filter rects, target rects, planes [K][n][4])].  Returns (evals, seconds) of one pass."""
        evals = sum(sum(f[2] * f[3] for f in fr) * pls.shape[0] for fr, _, pls in sample)
        t0 = time.perf_counter()
        for fr, tr, pls in sample:
            self.run(fr, tr, pls)
        return evals, time.perf_counter() - t0

    def calib_note(self):
        return "; ".join(f"{k}: {v['evals_per_s']:.3g} evals/s @ {v['threads']} thr" for k, v in self.calib.items())

    def close(self):
        for a in self.arms.values():
            a.close()


def cpu_baseline_beside(W, H, D, windR, imL, vol_h, naive, imR_h, groups, layer_of, planes_h):
    """`cpu_baseline` of our arm: group 0 of every layer, all its proposal steps, on the host cores.  `groups[i]` has .layer,
    .group, .cells, .n_steps; `layer_of(l)` gives the rectangles; `planes_h[i]` is [K][n][4]."""
    arm = CpuArm(W, H, D, windR, imL, vol_h, naive=naive, imR=imR_h)
    sample, used = [], []
    for gi, g in enumerate(groups):
        if g.group != 0:
            continue
        lay = layer_of(g.layer)
        sample.append(([lay.filterRegions[r] for r in g.cells], [lay.sharedRegions[r] for r in g.cells], np.ascontiguousarray(planes_h[gi])))
        used.append(f"L{g.layer}g0x{g.n_steps}")
    arm.calibrate(*sample[0])  # also warms
    tot_e, tot_t = arm.time_sample(sample)
    cpu = {"value": tot_e / tot_t, "unit": UNIT, "cores": arm.nthr, "kind": arm.kind,
           "sample": f"group 0 of each layer, all steps ({'+'.join(used)}; {tot_e} evals in {tot_t:.2f} s); calibration: {arm.calib_note()}"}
    arm.close()
    return cpu


def run_reference(args, W, H, D, windR, rank, world):
    """CPU arm with all host threads, on a bounded sample of the sweep (group 0 of every layer, all proposal steps)."""
    if rank != 0:
        return
    # nothing of the product is loaded in this process (VERDICT r1 weak #7): the cell rectangles come from the reference's own
    # LayerManager (oracle/_ref) or, without it, from the oracle's restatement; inputs from the package's pure-numpy generators
    from localexpstereo_b200 import synth   # numpy only; importing the package does not load liblexp_cuda.so
    from oracle import lexp_oracle as O
    naive = args.workload.endswith("_naive")
    imL, vol = make_inputs(W, H, D)
    imR = synth.synthetic_image(H, W, 43) if naive else None
    arm = CpuArm(W, H, D, windR, imL, None if naive else vol, naive=naive, imR=imR)
    try:
        from oracle import ref_binding
        make_layer = ref_binding.layer if (ref_binding.available() or ref_binding.build_ref.reference_present()) else O.make_layer
    except Exception:
        make_layer = O.make_layer
    units = [5, 15, 25] if naive else [int(W * 0.01), int(W * 0.03), int(W * 0.09)]   # main.cpp:304-306 / 395-397
    steps = [9, 3, 3]                                                                     # Exp(1)+Ransac(1)+Random(7) | Exp(2)+Ransac(1) x 2
    sample = []  # (filter rects, target rects, planes [K][n][4]) of group 0 of every layer: 15 of the 240 batched evaluations
    for li, u in enumerate(units):
        lay = make_layer(W, H, windR, u)
        cells = lay["groups"][0]
        pls = np.ascontiguousarray(synth.synthetic_planes(lay["unit"], steps[li], D, 7 + li)[:, cells, :])
        sample.append(([lay["filter"][r] for r in cells], [lay["shared"][r] for r in cells], pls))
    kind, nthr = arm.calibrate(*sample[0])
    for _ in range(args.warmup):
        arm.time_sample(sample)
    evals, dt = 0, 0.0
    for _ in range(args.steps):
        e, t = arm.time_sample(sample)
        evals, dt = e, dt + t
    dt /= args.steps
    val = evals / dt
    nb = sum(p.shape[0] for _, _, p in sample)
    desc = (f"group 0 of each of the 3 layers, all K=9/3/3 steps ({nb} of 240 batched evaluations, {evals} evals per step); "
            f"calibration on layer 0: {arm.calib_note()}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64 guided filter / f32 sampling", "data": "synthetic",
        "config": {"workload": args.workload, "W": W, "H": H, "ndisp": D, "windR": windR, "sample": desc},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": nthr, "kind": kind, "sample": desc},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))
    arm.close()


# ---------------------------------------------------------------------------------------------
def run_ours(args, W, H, D, windR, rank, world, local_rank):
    """Our arm.  `value`: the sweep (3 layers x 16 groups x K = 9/3/3 batched evaluations = 240 launches of lexp_fused_kernel) as the
    device-resident PatchMatch phase -- proposals drawn on the device, unary costs, fused `cur > prop` update of currentCost_ /
    currentLabeling_ in HBM; at N > 1 the cells of every group are sharded over the ranks and every accepted update is stored by
    the kernel into all ranks' copies of the state over NVLink (no collective on the data path; NCCL only broadcasts the inputs once).
    The image-based NaiveStereoEnergy workload (configs[0]) times the plain unary sweep instead (no device PatchMatch phase for it)."""
    import torch
    import localexpstereo_b200 as L
    from localexpstereo_b200 import synth
    from localexpstereo_b200.sweep import PMSweep, UnarySweep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    naive = args.workload.endswith("_naive")
    shard = world > 1 and not args.replicas
    shard_rank, shard_world = (rank, world) if shard else (0, 1)

    # ---- inputs: generated once (rank 0) and broadcast over NCCL to the ranks of a cell shard; one image pair per rank for --replicas
    if shard:
        img_t = torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
        vol_d = torch.empty((D, H, W), dtype=torch.float32, device=dev)
        if rank == 0:
            imL, vol_h = make_inputs(W, H, D)
            img_t.copy_(torch.from_numpy(imL)); vol_d.copy_(torch.from_numpy(vol_h))
        dist.broadcast(img_t, 0)
        dist.broadcast(vol_d, 0)
        imL = img_t.cpu().numpy()
        vol_h = None if rank else vol_h
        del img_t
    else:
        imL, vol_h = make_inputs(W, H, D)
        vol_d = torch.from_numpy(vol_h).to(dev)
    if naive:  # -mode MiddV2: image-based energy, th_col 10 / th_grad 2 / alpha 0.9 (StereoEnergy.h:26-37), layers 5/15/25
        prm = L.Parameters(windR=windR, filterName="GF", filter_param1=EPS)
        imR_h = synth.synthetic_image(H, W, 43)
        E = L.NaiveStereoEnergy(imL, imR_h, prm, D - 1, device=local_rank)
    else:
        prm = L.Parameters(windR=windR, filterName="GF", filter_param1=EPS, th_col=TH_COL)
        E = L.CostVolumeEnergy(imL, None, vol_d, None, prm, D - 1, device=local_rank)
    del vol_d  # the context keeps its own blocked copy
    torch.cuda.empty_cache()
    stream = torch.cuda.current_stream(dev)
    E.set_stream(stream.cuda_stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, n):
        """n calls of fn on the current stream between two events, bracketed by barriers; ms per call, max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def capture(fn):
        """fn's launches as one CUDA graph (no per-launch CPU work in the timed region); eager launches if capture fails."""
        if args.no_graph:
            return fn, False
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                E.set_stream(torch.cuda.current_stream(dev).cuda_stream)
                fn()
            E.set_stream(stream.cuda_stream)
            torch.cuda.synchronize(dev)
            return g.replay, True
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); using eager launches\n")
            E.set_stream(stream.cuda_stream)
            return fn, False

    # ---- the unary-only sweep (round 1's `value`; still the headline for the NaiveStereoEnergy workload)
    unary = UnarySweep(E, unit_sizes=[5, 15, 25] if naive else None, rank=shard_rank, world=shard_world)
    planes_h = all_planes(unary, D)
    evals_per_step = unary.total_filter_px * (world if args.replicas else 1)  # whole job, all ranks
    unary_info = None
    cost_d = torch.zeros((H, W), dtype=torch.float32, device=dev)
    if naive or world == 1:
        planes_d = [torch.from_numpy(p).to(dev) for p in planes_h]

        def sweep_unary():
            for gi, g in enumerate(unary.groups):
                base, n = planes_d[gi].data_ptr(), g.plan.num_calls
                for k in range(g.n_steps):
                    g.plan.eval_device(base + k * n * 16, cost_d.data_ptr(), W * 4, True, 0, planes_on_device=True)

        E.set_overlap(True)   # all plane arrays of the sweep are on the device before its first launch: consecutive launches may overlap
        for _ in range(args.warmup):
            sweep_unary()
        run_u, graph_u = capture(sweep_unary)
        run_u(); run_u()
        ms_u = timed(run_u, args.steps)
        unary_info = {"ms_per_step": ms_u, "value": evals_per_step / (ms_u * 1e-3), "unit": UNIT, "cuda_graph": graph_u,
                      "note": "the same 240 batched evaluations with host-supplied planes, unary maps written to an H x W image in HBM (no proposals, no update)"}

    # ---- the PatchMatch-phase sweep: `value`
    pms = None
    clocks = ClockSampler(local_rank)
    if not naive:
        pms = PMSweep(E, rank=shard_rank, world=shard_world)
        pms.begin()
        if shard:
            handles = [None] * world
            dist.all_gather_object(handles, pms.energy.pm_ipc_export(0))
            pms.connect(handles)
            barrier()
        init_labels = synth.synthetic_planes([pms.lm.layers[0].unitRegions[i] for i in range(len(pms.lm.layers[0].unitRegions))], 1, D, 99)[0]
        pms.init(init_labels[pms.init_index])
        launches_per_step = 0
        for it in range(args.warmup):
            launches_per_step = pms.iteration(it, 4321)
        barrier()
        IT = args.warmup  # the replayed iteration: fixed index (same proposal distribution every step; the state keeps evolving)
        run_pm, graph_pm = capture(lambda: pms.iteration(IT, 4321))
        run_pm(); run_pm()
        if rank == 0:
            clocks.start()
        ms_per_step = timed(run_pm, args.steps)
        clk = clocks.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:   # the state after the last timed step: currentCost_ / currentLabeling_
            st_c, st_l = pms.get()
            dump_outputs(args.dump_outputs, {"current_cost": st_c, "current_labeling": st_l})
        launches = launches_per_step * args.steps
        graph_used = graph_pm
        local_alg = unary.local_alg_bytes   # same cells, same K = 9/3/3 evaluations per cell visit as the unary sweep
    else:
        if rank == 0:
            clocks.start()
        ms_per_step = timed(run_u, args.steps)
        clk = clocks.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:   # the unary maps of the last timed step, as written into the H x W cost image
            dump_outputs(args.dump_outputs, {"cost_image": cost_d.cpu().numpy()})
        launches = unary.launches_per_sweep * args.steps
        graph_used = graph_u
        local_alg = unary.local_alg_bytes
    value = evals_per_step / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel (lexp_fused_kernel).  It is the ONLY kernel of the timed region, and with programmatic
    # dependent launch consecutive launches overlap (the next one fills the last, partly empty wave), so a per-launch duration is
    # not defined: achieved = algorithmic bytes this rank's launches of a sweep move / the timed region's own duration
    # (kernel_ms_per_step == ms_per_step; at N > 1 the stores into the peers' copies are part of the kernel).
    # `ms_by_layer`: one eager sweep bracketed per layer (3 event pairs; includes that layer's launch gaps).
    peak, peak_src = measured_peak_gbs()
    achieved = local_alg / (ms_per_step * 1e-3) / 1e9
    by_layer = {}
    if world == 1:
        evs = []
        if pms is not None:
            gen, cur = pms.iteration_by_group(IT, 4321), None
            for (li, gi, g, owners) in list(pms.schedule):
                if li != cur:
                    e = torch.cuda.Event(enable_timing=True); e.record(stream); evs.append((li, e)); cur = li
                next(gen)
            for _ in gen:
                pass
        else:
            cur = None
            for gi, g in enumerate(unary.groups):
                if g.layer != cur:
                    e = torch.cuda.Event(enable_timing=True); e.record(stream); evs.append((g.layer, e)); cur = g.layer
                base, n = planes_d[gi].data_ptr(), g.plan.num_calls
                for k in range(g.n_steps):
                    g.plan.eval_device(base + k * n * 16, cost_d.data_ptr(), W * 4, True, 0, planes_on_device=True)
        e = torch.cuda.Event(enable_timing=True); e.record(stream); evs.append((None, e))
        torch.cuda.synchronize(dev)
        by_layer = {str(evs[i][0]): round(evs[i][1].elapsed_time(evs[i + 1][1]), 4) for i in range(len(evs) - 1)}

    # ---- end to end: the same sweep through the C-ABI with HOST buffers, copies inside the timed region
    n_e2e = args.steps
    e2e_unary = None
    if naive or world == 1:
        cost_h = np.zeros((H, W), np.float32)
        L.host_register(cost_h)  # page-locked + mapped: unary tiles land in the host image without a bounce buffer
        for ph in planes_h:
            L.host_register(ph)  # the per-step inputs (plane hypotheses) are copied H2D from pinned memory

        def sweep_host():
            for gi, g in enumerate(unary.groups):
                for k in range(g.n_steps):
                    g.plan.eval_host(planes_h[gi][k], cost_h, True, 0)

        sweep_host()  # warm-up (allocates the pinned staging buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            sweep_host()
        torch.cuda.synchronize(dev)
        dt = (time.perf_counter() - t0) / n_e2e
        L.host_unregister(cost_h)
        for ph in planes_h:
            L.host_unregister(ph)
        e2e_unary = {"value": evals_per_step / dt, "unit": UNIT, "h2d_bytes_per_step": sum(g.plan.num_calls * 16 * g.n_steps for g in unary.groups),
                     "d2h_bytes_per_step": unary.local_target_px * 4,
                     "path": "unary maps: the 240 batched evaluations one by one through lexp_plan_eval_host, plane hypotheses H2D, every unary "
                             "map D2H into the host cost image (what the graph-cut iterations need on the host, FastGCStereo.h:49-53)"}
    if pms is not None:
        # PatchMatch-phase iteration (FastGCStereo.h:143-157, doGC == false) through lexp_pm_begin / lexp_plan_pm_step / lexp_pm_get:
        # currentCost_ + currentLabeling_ go H2D from page-locked host memory on every rank, the sweep runs on the device(s), and
        # rank 0 -- whose copy of the state every rank's kernels have written -- brings the state back D2H.
        st_cost = np.zeros((H, W), np.float32)
        st_lab = np.zeros((H, W, 4), np.float32)
        L.host_register(st_cost); L.host_register(st_lab)
        pms.get(out_cost=st_cost, out_labeling=st_lab)
        before = float(st_cost.mean())

        def pm_iteration(it):
            pms.begin(st_cost, st_lab)                                             # H2D: 20 B per pixel
            if dist is not None:
                dist.barrier()                                                     # no peer may write into a copy that is still being uploaded
            pms.iteration(it, 4321)                                                # 240 launches, device-resident
            if rank == 0 or not shard:
                pms.get(out_cost=st_cost, out_labeling=st_lab)                     # D2H: 20 B per pixel (blocking)
            else:
                E.sync()
            if dist is not None:
                dist.barrier()

        pm_iteration(IT)  # warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            pm_iteration(IT)   # the same iteration index as the timed device sweep: the same 240 evaluations (no RandomProposer early stop)
        dtp = torch.tensor([(time.perf_counter() - t0) / n_e2e], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(dtp, op=dist.ReduceOp.MAX)
        dt_pm = float(dtp.item())
        if rank == 0:
            assert np.isfinite(st_cost).all() and float(st_cost.mean()) <= before   # the sweeps really lowered the energy
        L.host_unregister(st_cost); L.host_unregister(st_lab)
        e2e = {"value": evals_per_step / dt_pm, "unit": UNIT, "h2d_bytes_per_step": H * W * 20 * world,
               "d2h_bytes_per_step": H * W * 20 * (world if args.replicas else 1), "ms_per_step": dt_pm * 1e3,
               "path": "PatchMatch-phase iteration (FastGCStereo.h:143-157, doGC == false) through lexp_pm_begin / lexp_plan_pm_step / "
                       "lexp_pm_get: currentCost_ + currentLabeling_ H2D from page-locked host memory (every rank), the 240 batched "
                       "evaluations with device-side proposals and the fused cur > prop update, state D2H (rank 0's copy holds everything)"}
        if e2e_unary is not None:
            e2e["unary_maps"] = e2e_unary
    else:
        e2e = e2e_unary

    # ---- CPU baseline beside it (rank 0, N = 1): the reference's CPU implementation on a bounded sample
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_beside(W, H, D, windR, imL, None if naive else vol_h, naive, imR_h if naive else None, unary.groups, unary.layer, planes_h)

    if rank == 0:
        if naive:
            par = "unary sweep"
        elif args.replicas:
            par = f"replicas x{world} (one image pair per GPU), PatchMatch-phase sweep"
        else:
            par = f"cell-shard x{world}, PatchMatch-phase sweep" + (": accepted updates stored into all ranks' copies of the state by the kernel "
                                                                   "(peer memory over NVLink), epoch flags at group boundaries; inputs broadcast once over NCCL" if world > 1 else "")
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if args.replicas else "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "W": W, "H": H, "ndisp": D, "windR": windR, "th_col": TH_COL, "eps": EPS,
                       "layers_unit": unary.unit_sizes, "steps_per_layer": unary.steps,
                       "evals_per_step": evals_per_step, "target_px_per_step": unary.total_target_px,
                       "batched_evaluations_per_step": launches // args.steps,
                       "parallelism": par, "cuda_graph": graph_used,
                       "l2": "inputs larger than L2 (cost volume %.2f GB; proposals follow the evolving state)" % (4.0 * D * H * W / 1e9)},
            "clocks": clk,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         # DRAM read+write of ONE layer-0 launch (500 cells, algorithmic 2.34e8 B) from the ncu --set full capture
                         # summarised in profiles/r2_fused_ncu_L0.md; only known for the default workload at N = 1
                         "traffic": (229575680 + 9689856) if (args.workload == "synthetic_2048x1536x256_r20" and world == 1) else None,
                         "traffic_note": "per layer-0 launch of 500 cells (algorithmic 2.34e8 B); profiles/r2_fused_ncu_L0.md",
                         "kernel": "lexp_fused_kernel", "peak_source": peak_src,
                         "algorithmic_bytes_per_step": local_alg, "kernel_ms_per_step": ms_per_step, "ms_by_layer": by_layer},
        }
        if unary_info is not None and not naive:
            out["unary_sweep"] = unary_info
        if cpu is not None:
            out["cpu_baseline"] = cpu
        print(json.dumps(out), flush=True)
    if dist is not None:
        # captured graphs and peer mappings: synchronise, then leave without running destructors
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    if pms is not None:
        pms.close()
    unary.close()
    E.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="synthetic_2048x1536x256_r20", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the sweep eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path computed in its last step to DIR/<name>.npy (float32, at most "
                         "64 MB in all: a seeded sample of pixels beyond that); the inputs depend only on the arguments")
    ap.add_argument("--replicas", action="store_true",
                    help="BASELINE.json configs[3] style: every rank sweeps its OWN image pair (weak scaling, no data-path collective) "
                         "instead of sharding the cells of one pair (default, strong scaling)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    W, H, D, windR = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, W, H, D, windR, rank, world)
    else:
        run_ours(args, W, H, D, windR, rank, world, local_rank)


if __name__ == "__main__":
    main()
