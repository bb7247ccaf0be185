"""The diagnosis build of lexp_kernels.cuh (-DLEXP_TRACE=1) on the CPU emulator: its timing instrumentation must not change
what the kernel computes."""
import numpy as np
import pytest

from emu import emu_lib
import test_gpu_golden as _g


@pytest.mark.parametrize("variant", ["trace"])
def test_variant_reproduces_golden_vectors_and_the_shipped_kernel(variant, monkeypatch, tmp_path):
    import lexp_golden
    monkeypatch.setenv("LEXP_TRACE_FILE", str(tmp_path / "trace.txt"))  # only the `trace` (diagnosis) build writes it
    import localexpstereo_b200 as L
    from oracle import lexp_oracle as O
    with emu_lib.emulated(variant=variant):
        _g.test_golden_vectors_through_the_c_abi()
    G = lexp_golden.load()
    H, W = G["imL"].shape[:2]
    prm = L.Parameters(windR=G["windR"], filterName="GF", filter_param1=G["eps"], th_col=G["th"])
    lay = L.LayerManager(W, H, G["windR"]).addLayer(16)
    g = lay.disjointRegionSets[2]
    rng = O.CvRNG(8)
    planes = np.stack([O.create_random_label(rng, *lay.unitRegions[r][:2], 0.0, G["D"] - 1.0) for r in g])
    outs = []
    for v in ("", variant):
        with emu_lib.emulated(variant=v, order=2 if v else 0):
            E = L.CostVolumeEnergy(G["imL"], G["imR"], G["volL"], G["volR"], prm, G["D"] - 1)
            img = np.full((H, W), -3.0, np.float32)
            for k in range(2):  # two launches into the same image (write-after-write across launches)
                E.ComputeUnaryPotentialBatch([lay.filterRegions[r] for r in g], [lay.sharedRegions[r] for r in g], img, planes if k else planes[::-1].copy())
            E.close()
            outs.append(img)
    assert np.array_equal(outs[0], outs[1])
    if variant == "trace":
        lines = open(tmp_path / "trace.txt").read().strip().splitlines()
        assert len(lines) >= 3 and all(" | A total " in l and " | E total " in l for l in lines)
