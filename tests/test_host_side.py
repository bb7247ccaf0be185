"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, the LayerManager
geometry served through it equals the oracle's, and the cell-shard logic is consistent across 2 gloo ranks.
No compute entry point is called here (that needs a GPU)."""
import os
import re
import socket

import numpy as np
import pytest

from oracle import lexp_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from localexpstereo_b200 import _capi, build
    build.build()
    hdr = open(os.path.join(ROOT, "include", "lexp_cuda.h")).read()
    declared = set(re.findall(r"LEXP_API\s+[\w\s\*]+?\b(lexp_\w+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_capi.SO_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/lexp_cuda.h but not exported"
    assert declared == set(_capi.SYMBOLS), declared ^ set(_capi.SYMBOLS)
    assert _capi.lib().lexp_version() >= 100


def test_no_cpu_fallback_when_library_is_missing(monkeypatch):
    from localexpstereo_b200 import _capi
    monkeypatch.setattr(_capi, "_lib", None)
    monkeypatch.setattr(_capi, "SO_PATH", "/nonexistent/liblexp_cuda.so")
    with pytest.raises(_capi.LexpError):
        _capi.lib()


@pytest.mark.parametrize("W,H,u,windR", [(450, 375, 5, 20), (450, 375, 15, 20), (450, 375, 25, 20), (2048, 1536, 20, 20), (2048, 1536, 61, 20),
                                         (2048, 1536, 184, 20), (1436, 992, 14, 20), (1436, 992, 129, 20), (3840, 2160, 38, 32),
                                         (3840, 2160, 345, 32), (37, 29, 5, 4), (10, 10, 7, 3), (64, 64, 64, 8), (33, 70, 16, 6)])
def test_layer_manager_geometry_matches_oracle(W, H, u, windR):
    """LayerManager::addLayer (LayerManager.h:88-185) through lexp_layer_geometry vs the numpy restatement."""
    import localexpstereo_b200 as L
    lay = L.LayerManager(W, H, windR).addLayer(u)
    ref = O.make_layer(W, H, windR, u)
    assert lay.heightBlocks == ref["heightBlocks"] and lay.widthBlocks == ref["widthBlocks"]
    assert lay.unitRegions == ref["unit"] and lay.sharedRegions == ref["shared"] and lay.filterRegions == ref["filter"]
    assert lay.disjointRegionSets == ref["groups"]
    # invariants the kernels rely on
    for un, sh, fi in zip(lay.unitRegions, lay.sharedRegions, lay.filterRegions):
        assert fi[0] <= sh[0] and fi[1] <= sh[1] and fi[0] + fi[2] >= sh[0] + sh[2] and fi[1] + fi[3] >= sh[1] + sh[3]
        assert fi[0] == max(sh[0] - windR, 0) or fi[0] == 0
    for g in lay.disjointRegionSets:  # cells of a group never overlap (FastGCStereo.h:30 runs them concurrently)
        occ = np.zeros((H, W), np.int32)
        for r in g:
            x, y, w, h = lay.sharedRegions[r]
            occ[y:y + h, x:x + w] += 1
        assert occ.max() <= 1


def test_survey_cell_counts():
    import localexpstereo_b200 as L
    from localexpstereo_b200.sweep import v3_layer_units
    assert v3_layer_units(2048) == [20, 61, 184]
    lm = L.LayerManager(2048, 1536, 20)
    counts = [len(lm.addLayer(u).unitRegions) for u in v3_layer_units(2048)]
    assert counts == [7854, 850, 88]  # SURVEY.md section 8 table


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _shard_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import localexpstereo_b200 as L
    from localexpstereo_b200.sweep import shard_cells, tile_offsets
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    lay = L.LayerManager(210, 150, 20).addLayer(10)
    ok = True
    for g in lay.disjointRegionSets:
        mine = shard_cells(g, rank, world)
        rects = [lay.sharedRegions[r] for r in mine]
        offs, total = tile_offsets(rects)
        # every rank publishes its padded tile buffer filled with (cell id + pixel index); emulates the all-gather of unary tiles
        sizes = [None] * world
        dist.all_gather_object(sizes, total)
        mx = max(sizes)
        buf = torch.full((mx,), -1.0)
        for r, o, rc in zip(mine, offs, rects):
            buf[o:o + rc[2] * rc[3]] = float(r) + torch.arange(rc[2] * rc[3]) * 1e-6
        gathered = [torch.empty(mx) for _ in range(world)]
        dist.all_gather(gathered, buf)
        # reassemble on every rank and check against the unsharded layout
        seen = []
        for rk in range(world):
            cells_rk = shard_cells(g, rk, world)
            rects_rk = [lay.sharedRegions[r] for r in cells_rk]
            offs_rk, _ = tile_offsets(rects_rk)
            for r, o, rc in zip(cells_rk, offs_rk, rects_rk):
                tile = gathered[rk][o:o + rc[2] * rc[3]]
                ok &= bool(abs(float(tile[0]) - float(r)) < 1e-3 and abs(float(tile[-1]) - (r + (rc[2] * rc[3] - 1) * 1e-6)) < 1e-2)
                seen.append(int(r))
        ok &= sorted(seen) == sorted(g)
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, ok))


def test_cell_shard_all_gather_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _pm_shard_worker(rank, world, port, q):
    """Host-side logic of the multi-GPU PatchMatch-phase cell shard across real processes: every rank derives the same
    (layer, group) schedule and cell ownership, and the epoch every rank waits for is exactly the one its peer publishes."""
    import torch.distributed as dist
    import localexpstereo_b200 as L
    from localexpstereo_b200.sweep import EpochClock, pm_schedule
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    lm = L.LayerManager(210, 150, 20)
    sched = pm_schedule(lm, [10, 31, 70], world)
    ok = True
    for (li, gi, by_rank, owners) in sched:   # a partition of every group's cells
        cells = sorted(int(c) for r in range(world) for c in by_rank[r])
        ok &= cells == sorted(lm.layers[li].disjointRegionSets[gi]) and owners == [r for r in range(world) if len(by_rank[r])]
    clock = EpochClock(rank, world)
    published, waited = [], []   # absolute epochs
    n0 = len(lm.layers[0].unitRegions)
    rounds = [[(None, None, None, [r for r in range(world) if len(range(r, n0, world))])]] + [sched, sched]   # init, two iterations
    for groups in rounds:
        for (_, _, by_rank, owners) in groups:
            mine = by_rank is None or len(by_rank[rank]) > 0
            if mine and rank in owners:
                a = clock.sync_args(True, True)
                published.append(clock.base + a["publish_epoch"])
                waited.append({r: clock.base + a["wait_epochs"][r] for r in range(world) if (a["wait_mask"] >> r) & 1 and r != rank})
            clock.group_done(owners)
        clock.advance()
    allp, allw = [None] * world, [None] * world
    dist.all_gather_object(allp, published)
    dist.all_gather_object(allw, waited)
    for a in range(world):            # every awaited epoch is one the peer really publishes, and it is published earlier
        for j, w in enumerate(allw[a]):
            for r, e in w.items():
                ok &= e in allp[r] and e < allp[a][j]
    ok &= all(p == sorted(set(p)) for p in allp) and len(allw[rank]) > 40
    # graph replay: from the second iteration on the relative numbers repeat exactly
    c2 = EpochClock(rank, world)
    seqs = []
    for groups in rounds + [sched]:
        seq = []
        for (_, _, by_rank, owners) in groups:
            seq.append(c2.sync_args(True, True))
            c2.group_done(owners)
        c2.advance()
        seqs.append(seq)
    ok &= seqs[2] == seqs[3]
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, bool(ok)))


def test_pm_cell_shard_schedule_and_epochs_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_pm_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def test_synthetic_planes_distribution():
    from localexpstereo_b200 import synth
    import localexpstereo_b200 as L
    lay = L.LayerManager(640, 480, 20).addLayer(16)
    P = synth.synthetic_planes(lay.unitRegions, 5, 128, 7)
    assert P.shape == (5, len(lay.unitRegions), 4) and P.dtype == np.float32 and (P[..., 3] == 0).all()
    slope = np.hypot(P[0, :, 0], P[0, :, 1])  # tan(polar angle) of the normal, angle ~ U[0, pi/3)
    assert slope.max() <= np.tan(np.pi / 3) + 1e-3 and 0.3 < np.median(slope) < 0.9
    u = np.asarray(lay.unitRegions)
    cx, cy = u[:, 0] + u[:, 2] / 2, u[:, 1] + u[:, 3] / 2
    z = P[0, :, 0] * cx + P[0, :, 1] * cy + P[0, :, 2]
    assert z.min() > -40 and z.max() < 127 + 40


def test_reference_side_adapter_compiles_and_links(tmp_path):
    """include/CudaCostVolumeEnergy.h (the StereoEnergy subclass a reference maintainer adds) against a cv:: stub."""
    import subprocess
    from localexpstereo_b200 import _capi, build
    build.build()
    exe = tmp_path / "adapter_check"
    so_dir = os.path.dirname(_capi.SO_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "tests", "cxx"), os.path.join(ROOT, "tests", "cxx", "adapter_check.cpp"),
           "-o", str(exe), "-L", so_dir, "-llexp_cuda", f"-Wl,-rpath,{so_dir}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and "lexp version" in out.stdout, out.stderr


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver times beside ours) prints one JSON line with the agreed keys."""
    import json
    import subprocess
    import sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny_450x375x64_r20",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads(res.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["config"]["workload"].startswith("tiny")


def test_emulation_hooks_never_reach_the_product_library():
    """csrc carries `#ifdef LEXP_EMU` hooks for the CPU emulator of tests/emu (test infrastructure).  The product build must not
    define it, and the built library must not contain the emulator."""
    import subprocess
    from localexpstereo_b200 import build, _capi
    assert not any("LEXP_EMU" in f for f in build.NVCC_FLAGS)
    build.build()
    syms = subprocess.run(["nm", "-C", _capi.SO_PATH], capture_output=True, text=True).stdout
    assert "emu::" not in syms and "run_block" not in syms
    assert "lexp_fused_kernel" in syms  # the device kernels are what the library carries


def test_bench_cpu_baseline_block_of_the_gpu_arm():
    """bench.py's `cpu_baseline` (computed beside the GPU number at N = 1) with a stand-in for the sweep object: same
    attributes as sweep.UnarySweep's groups; runs the reference's CPU implementation on group 0 of every layer."""
    import sys
    from types import SimpleNamespace
    sys.path.insert(0, ROOT)
    import bench
    import localexpstereo_b200 as L
    from localexpstereo_b200 import synth
    W, H, D, windR = 200, 150, 16, 20
    imL, vol = bench.make_inputs(W, H, D)
    lm = L.LayerManager(W, H, windR)
    layers = [lm.addLayer(u) for u in (5, 15)]
    groups, planes = [], []
    for li, lay in enumerate(layers):
        for gj, cells in enumerate(lay.disjointRegionSets[:2]):
            K = 3 - li
            groups.append(SimpleNamespace(layer=li, group=gj, cells=list(cells), n_steps=K))
            planes.append(np.ascontiguousarray(synth.synthetic_planes(lay.unitRegions, K, D, 7 + li)[:, cells, :]))
    cpu = bench.cpu_baseline_beside(W, H, D, windR, imL, vol, False, None, groups, lambda l: layers[l], planes)
    assert cpu["value"] > 0 and cpu["kind"] in ("reference", "port") and cpu["cores"] >= 1 and "L0g0x3+L1g0x2" in cpu["sample"]
    imR = synth.synthetic_image(H, W, 43)
    from oracle import build_ref
    if build_ref.build() is None:   # the image-based energy's only CPU implementation is the compiled reference
        with pytest.raises(RuntimeError, match="no CPU implementation"):
            bench.cpu_baseline_beside(W, H, D, windR, imL, None, True, imR, groups, lambda l: layers[l], planes)
        return
    cpu = bench.cpu_baseline_beside(W, H, D, windR, imL, None, True, imR, groups, lambda l: layers[l], planes)
    assert cpu["value"] > 0 and cpu["kind"] == "reference"
