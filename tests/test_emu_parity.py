"""The GPU parity tests, run on the CPU against the kernel source itself.

tests/emu/liblexp_emu.so is localexpstereo_b200/csrc (lexp_capi.cu + lexp_kernels.cuh, unmodified) compiled with
g++ -DLEXP_EMU against tests/emu/cuda_runtime.h: every CUDA thread is a fiber, named barriers follow the PTX semantics, a
deadlock or an unbalanced barrier is an error.  The tests below are the very functions of tests/test_gpu_parity.py,
tests/test_gpu_naive.py and the golden-vector test, executed through the same Python binding and C-ABI with the emulator
swapped in as the library.  They check the kernel's logic (indices, pipeline protocol, planner) without a GPU; the `-m gpu`
suite remains the parity gate for the real device."""
import pytest

from emu import emu_lib

# the test functions and their fixtures, imported under new names so that pytest collects them here without the gpu mark
import test_gpu_parity as _p
import test_gpu_golden as _g


@pytest.fixture(scope="module", autouse=True)
def _use_emulator():
    with emu_lib.emulated():
        yield


scene = _p.scene


class _HostAsDeviceMemory:
    """On the emulator device memory is host memory: numpy arrays stand in for the device buffers."""

    @staticmethod
    def zeros(shape, fill=0.0):
        import numpy as np
        return np.full(shape, fill, np.float32)

    @staticmethod
    def upload(a):
        import numpy as np
        return np.ascontiguousarray(a)

    @staticmethod
    def ptr(t):
        return t.ctypes.data

    @staticmethod
    def download(t):
        return t


@pytest.fixture(scope="module")
def devmem():
    return _HostAsDeviceMemory()


test_emu_device_image_and_tile_outputs = _p.test_device_image_and_tile_outputs
test_emu_host_tile_output = _p.test_host_tile_output
test_emu_partially_registered_output = _p.test_partially_registered_output_takes_the_staged_path
test_emu_volume_file_disparity_map_and_pfm = _p.test_volume_file_disparity_map_and_pfm
test_emu_stats_match_oracle = _p.test_stats_match_oracle
test_emu_cells_of_a_layer = _p.test_cells_of_a_layer
test_emu_single_cell_virtuals = _p.test_single_cell_virtuals
test_emu_branches_of_the_sampler = _p.test_branches_of_the_sampler
test_emu_filter_rect_smaller_than_dependency_cone = _p.test_filter_rect_smaller_than_dependency_cone
test_emu_errors_are_reported = _p.test_errors_are_reported
test_emu_concurrent_single_cell_calls = _p.test_concurrent_single_cell_calls_like_the_openmp_loop
test_emu_other_filter_radii = _p.test_other_filter_radii
test_emu_nonzero_min_disparity_and_odd_max = _p.test_nonzero_min_disparity_and_odd_max
test_emu_golden_vectors_through_the_c_abi = _g.test_golden_vectors_through_the_c_abi
test_emu_textureless_guides = _p.test_textureless_guides
test_emu_plan_outlives_its_energy = _p.test_plan_outlives_its_energy
test_emu_volume_preparation_on_the_device = _p.test_volume_preparation_on_the_device


def test_emu_result_does_not_depend_on_the_thread_schedule(scene):
    """A missing or misplaced barrier in lexp_fused_kernel would make the result depend on the order in which the emulated
    threads run between barriers: forward, reverse and reshuffled-every-pass schedules must agree bit for bit."""
    import numpy as np
    from oracle import lexp_oracle as O
    L, E, H, W, D = (scene[k] for k in "L E H W D".split())
    lay = L.LayerManager(W, H, 20).addLayer(10)
    rng = O.CvRNG(5)
    outs = []
    for order in (0, 1, 2):
        with emu_lib.emulated(order=order):
            res = []
            for g in lay.disjointRegionSets[:3]:
                rng_g = O.CvRNG(5 + len(res))
                planes = np.stack([O.create_random_label(rng_g, *lay.unitRegions[r][:2], 0.0, D - 1.0) for r in g])
                img = np.full((H, W), -7.0, np.float32)
                E.ComputeUnaryPotentialBatch([lay.filterRegions[r] for r in g], [lay.sharedRegions[r] for r in g], img, planes, mode=0)
                res.append(img)
            outs.append(np.stack(res))
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


def test_emu_concurrent_calls_are_combined_into_batched_launches(scene):
    """lexp_eval_cell from many threads at once (the reference's unchanged OpenMP loop): calls that arrive while the device is
    busy must be served together by one launch, with exactly the results of one-call-at-a-time evaluation."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import lexp_oracle as O
    L, H, W, D = (scene[k] for k in "L H W D".split())
    imL, imR, volL, volR = _p.make_scene(H, W, D)
    prm = L.Parameters(windR=20, filterName="GF", filter_param1=1e-4, th_col=0.5)
    lay = L.LayerManager(W, H, 20).addLayer(7)
    cells = [r for g in lay.disjointRegionSets[:2] for r in g]
    rng = O.CvRNG(9)
    planes = [np.stack([O.create_random_label(rng, *lay.unitRegions[r][:2], 0.0, D - 1.0) for r in cells]) for _ in range(3)]

    def sweep(E, workers):
        outs = []
        for k in range(3):
            img = np.full((H, W), -7.0, np.float32)

            def one(i, k=k, img=img):
                f, t = lay.filterRegions[cells[i]], lay.sharedRegions[cells[i]]
                # cells of different groups overlap: give every call its own image, as they would race otherwise
                own = np.full((H, W), -7.0, np.float32)
                E.ComputeUnaryPotential(f, t, own[f[1]:f[1] + f[3], f[0]:f[0] + f[2]], planes[k][i], mode=k & 1)
                return own[t[1]:t[1] + t[3], t[0]:t[0] + t[2]].copy()

            with ThreadPoolExecutor(max_workers=workers) as ex:
                outs.append(list(ex.map(one, range(len(cells)))))
        return outs

    E0 = L.CostVolumeEnergy(imL, imR, volL, volR, prm, D - 1)
    ref = sweep(E0, 1)   # one caller at a time: every call takes the plain single-cell path
    assert E0.combine_stats == (0, 0)
    E0.close()
    E1 = L.CostVolumeEnergy(imL, imR, volL, volR, prm, D - 1)
    got = sweep(E1, 12)
    batches, calls = E1.combine_stats
    launches = E1.launch_count
    E1.close()
    for a, b in zip(ref, got):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    n = 3 * len(cells)
    assert calls > n // 4 and batches < calls, (batches, calls, n)   # calls were served in groups (typically ~280 of 288 in ~45 launches)
    print(f"{n} calls: {calls} combined into {batches} launches, {launches} kernel launches in total")


def test_emu_zero_copy_and_staged_host_paths_agree(scene):
    """lexp_plan_eval_host writes straight into a registered (mapped) cost image, and through a compact device buffer + host
    scatter otherwise: same pixels, and only costs(targetRect) is touched in both."""
    import numpy as np
    from oracle import lexp_oracle as O
    L, E, H, W, D = (scene[k] for k in "L E H W D".split())
    lay = L.LayerManager(W, H, 20).addLayer(18)
    g = lay.disjointRegionSets[0]
    fr = [lay.filterRegions[r] for r in g]
    tr = [lay.sharedRegions[r] for r in g]
    plan = E.make_plan(fr, tr)
    rng = O.CvRNG(31)
    planes = np.stack([O.create_random_label(rng, *lay.unitRegions[r][:2], 0.0, D - 1.0) for r in g])
    staged = np.full((H, W), -7.0, np.float32)
    plan.eval_host(planes, staged, True, 0)
    mapped = np.full((H, W), -7.0, np.float32)
    L.host_register(mapped)
    try:
        plan.eval_host(planes, mapped, True, 0)
    finally:
        L.host_unregister(mapped)
    assert np.array_equal(staged, mapped)
    mask = np.zeros((H, W), bool)
    for x, y, w, h in tr:
        mask[y:y + h, x:x + w] = True
    assert (staged[~mask] == -7.0).all() and (staged[mask] != -7.0).all()
    with pytest.raises(L.LexpError):
        L.host_unregister(mapped)  # not registered any more
    plan.close()
