"""-m gpu: the reference's own pybind surface (`rasterize_gaussians`, `rasterize_gaussians_backward`, `mark_visible`;
ext.cpp:15-19) rebuilt on top of the C ABI -- integration/rasterize_points_gsr.cpp, the file INTEGRATION.md section 3
hands a maintainer -- must give the same results as the unmodified reference extension when both are driven by the
same autograd wrapper (oracle/ref_driver.RefRasterize: the argument packing of the reference's Python package).  The
reference's results are the ones it computed on a B200 (tests/golden/ref_case_*.npz)."""
import os

import numpy as np
import pytest
import torch

import gpu_util as U
import scenes
from integration import build_binding
from oracle import ref_driver

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    mod = build_binding.load()
    if mod is None:
        pytest.skip("integration/_gsr_refbind.so not built (python integration/build_binding.py)")
    return mod


@pytest.mark.parametrize("case", "ABCD")
def test_binding_matches_reference_extension(binding, case):
    ref = np.load(os.path.join(U.GOLD, f"ref_case_{case}.npz"))
    s = scenes.scene(case)
    dev = torch.device("cuda")
    # forward AND backward of the run must go through `binding`: keep it selected for the whole run_torch call
    saved = ref_driver._mod
    ref_driver._mod = binding
    try:
        new = scenes.run_torch(s, ref_driver.rasterize, dev)
    finally:
        ref_driver._mod = saved
    for k in ("color", "depth", "median", "opacity", "radii"):
        assert np.array_equal(new[k], ref["ref_" + k]), k
    assert sorted(k for k in new if k.startswith("g_")) == sorted(k[4:] for k in ref.files if k.startswith("ref_g_"))
    for k in sorted(k for k in new if k.startswith("g_")):
        U.assert_grads_close(new[k], ref["ref_" + k], what=f"{case}:{k}")


def test_binding_mark_visible_and_empty_input(binding):
    dev = torch.device("cuda")
    s = scenes.scene("C")
    pts = torch.tensor(s["means3D"], device=dev)
    view = torch.tensor(s["viewmatrix"], device=dev); proj = torch.tensor(s["projmatrix"], device=dev)
    from gaustudio_b200 import _C
    assert torch.equal(binding.mark_visible(pts, view, proj), _C.mark_visible(pts, view, proj))
    e = torch.Tensor([])
    out = binding.rasterize_gaussians(torch.zeros(3), torch.zeros(0, 3, device=dev), e, torch.zeros(0, 1, device=dev),
                                      torch.zeros(0, 3, device=dev), torch.zeros(0, 4, device=dev), 1.0, e, view, proj,
                                      s["tanfovx"], s["tanfovy"], 32, 48, torch.zeros(0, 16, 3, device=dev), 3,
                                      torch.tensor(s["campos"], device=dev), False, False)
    assert out[0] == 0 and out[1].shape == (3, 32, 48) and float(out[1].abs().max()) == 0.0
