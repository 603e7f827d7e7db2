"""-m gpu parity tests: the CUDA path (through the reference-shaped Python API -> ctypes -> C ABI) against
 (1) what the UNMODIFIED reference extension compiled for sm_100a computed on a B200: the committed golden fixtures
     (tests/golden/ref_case_*.npz whole, tests/golden/ref_outputs_sampled.npz as digests and seeded samples),
 (2) the CPU oracle.
Tolerances: BASELINE.json -- 1e-4 max-abs on images, 1e-3 relative on gradients.  Against the reference on a B200
the forward is expected to be BIT-EXACT (same arithmetic, same order), which is asserted."""
import os

import numpy as np
import pytest
import torch

import gpu_util as U
import scenes

pytestmark = pytest.mark.gpu
GOLD = U.GOLD
FWD = ("color", "depth", "median", "opacity")


@pytest.fixture(scope="module")
def G():
    return np.load(U.SAMPLED)


def _grad_keys(r):
    return sorted(k for k in r if k.startswith("g_"))


@pytest.mark.parametrize("case", "ABCD")
def test_matches_compiled_reference(case):
    ref = np.load(os.path.join(GOLD, f"ref_case_{case}.npz"))
    s = scenes.scene(case)
    dev = torch.device("cuda")
    new = scenes.run_torch(s, U.new_rasterize, dev)
    for k in FWD + ("radii",):
        assert np.array_equal(new[k], ref["ref_" + k]), f"{k} not bit-identical to the reference"
    assert _grad_keys(new) == sorted(k[4:] for k in ref.files if k.startswith("ref_g_"))
    for k in _grad_keys(new):
        U.assert_grads_close(new[k], ref["ref_" + k], what=f"{case}:{k}")
    assert (new["radii"] > 0).any()


@pytest.mark.parametrize("case", "ABCD")
def test_matches_golden_fixture(case):
    f = os.path.join(GOLD, f"ref_case_{case}.npz")
    if not os.path.exists(f):
        pytest.skip("golden fixture missing")
    G = np.load(f)
    s = scenes.scene(case)
    for k, v in s.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, G["in_" + k]), f"scene generator drifted from the fixture ({k})"
    dev = torch.device("cuda")
    captured = {}

    def rast(rs, *a, **kw):
        res = U.new_rasterize(rs, *a, **kw)
        fn = res[0].grad_fn
        captured["R"], captured["bufs"] = fn.num_rendered, fn.saved_tensors[7:10]  # before backward frees them
        return res
    new = scenes.run_torch(s, rast, dev)
    R = captured["R"]
    assert R == int(G["ref_num_rendered"])
    assert np.array_equal(new["radii"], G["ref_radii"])
    from gaustudio_b200 import _C
    P = s["means3D"].shape[0]
    ex = _C.debug_export(P, s["W"], s["H"], R, *captured["bufs"])
    # global sort order: the reference's list minus (Gaussian, tile) pairs that cannot contribute (exact tile culling);
    # the tile boundaries of the fixture's list come from the pinned CPU oracle (its list equals the fixture's)
    from oracle.oracle import Oracle
    o = Oracle()
    o.forward(s["means3D"], s["opacities"], s["viewmatrix"], s["projmatrix"], s["campos"], s["tanfovx"], s["tanfovy"],
              s["W"], s["H"], s["D"], shs=s.get("shs"), colors_precomp=s.get("colors_precomp"), scales=s.get("scales"),
              rotations=s.get("rotations"), cov3D_precomp=s.get("cov3D_precomp"), scale_modifier=s["scale_modifier"])
    ob = o.binning()
    if np.array_equal(ob["point_list"], G["ref_point_list"]):  # (host libm may move a key by an ulp on another box)
        U.assert_binned_list_is_culled_reference_list(ex, G["ref_point_list"], ob["ranges"], s["W"], s["H"], P)
    for k in FWD:
        U.assert_images_close(new[k], G["ref_" + k], atol=1e-6, what=f"{case}:{k}")
    for k in _grad_keys(new):
        U.assert_grads_close(new[k], G["ref_" + k], what=f"{case}:{k}")


@pytest.mark.parametrize("case", "ABCD")
def test_matches_cpu_oracle(case):
    s = scenes.scene(case)
    new = scenes.run_torch(s, U.new_rasterize, torch.device("cuda"))
    orc = U.oracle_run(s)
    assert (new["radii"] != orc["radii"]).mean() < 1e-3
    for k in FWD:
        # 1e-4 max-abs; a hard-threshold flip (alpha<1/255, T<1e-4) moves a pixel by more, so a tiny budget
        U.assert_images_close(new[k], orc[k], atol=1e-4, outlier_frac=2e-3, what=f"{case}:{k}")
    for k in _grad_keys(new):
        a, b = new[k], orc[k]
        scale = np.abs(b).max()
        assert (np.abs(a - b) > 1e-3 * np.abs(b) + 2e-3 * scale).mean() < 2e-3, k


def test_sh_degrees_and_stride(G):
    """D < tensor degree: coefficients are read with stride M (quirk 13); every degree against the reference."""
    s = scenes.scene("A")
    for D in (0, 1, 2, 3):
        s["D"] = D
        new = scenes.run_torch(s, U.new_rasterize, torch.device("cuda"))
        assert U.digest(new["color"]) == G[f"sh_D{D}_color"], D
        U.assert_sample_close(new["g_shs"], G, f"sh_D{D}_g_shs")
        assert (new["g_shs"][:, (D + 1) ** 2:, :] == 0).all()


def test_medium_scene_bit_exact_and_sorted(G):
    """cfg2-shaped scene (100k Gaussians, 800x800): forward bit-exact vs the reference; the sorted list is the
    reference's minus provably inert (Gaussian, tile) pairs, in the reference's order."""
    from gaustudio_b200 import _C
    from gaustudio_b200.synthetic import build_config
    model, cams, c = build_config("cfg2", K=3)
    dev = torch.device("cuda")
    model.to(dev)
    for v, cam in enumerate(cams[:2]):
        cam.to(dev)
        with torch.no_grad():
            n = _C.rasterize_gaussians(*U.raw_args(model, cam, c, dev, 3))
        assert n[0] > 1_000_000
        ex, dropped = U.assert_reference_outputs_and_binning(G, f"medium_v{v}", n, c["W"], c["H"], c["P"])
        assert 0 < dropped < n[0] // 2 and ex["num_binned"] == n[0] - dropped


def sparse_scene():
    s = dict(scenes.scene("D"))
    rng = np.random.RandomState(21)
    P = s["means3D"].shape[0]
    xyz, sc = s["means3D"].copy(), s["scales"].copy()
    far = np.arange(P) >= 1024
    far &= rng.rand(P) < 0.7                 # the first 1024 stay as they are: dense CTAs
    xyz[far] *= rng.uniform(3.0, 9.0, size=(int(far.sum()), 1)).astype(np.float32)   # behind the camera / off screen
    big = np.where(far)[0][:40]
    sc[big] = 1.5                            # off-screen centres whose splats still reach the image
    s["means3D"], s["scales"] = xyz, sc
    return s


def test_sparse_and_dense_projection_ctas_match_reference(G):
    """A scene whose projection CTAs are a mix of dense ones (everything visible) and sparse ones (most Gaussians
    behind the camera or far off screen, some off-screen centres whose splats still reach the image) stays
    bit-identical to the compiled reference; gradients within 1e-3."""
    new = scenes.run_torch(sparse_scene(), U.new_rasterize, torch.device("cuda"))
    assert 0.2 < (new["radii"] > 0).mean() < 0.8
    for k in FWD + ("radii",):
        assert U.digest(new[k]) == G["sparse_" + k], f"{k} not bit-identical to the reference"
    assert _grad_keys(new) == sorted(k[7:-4] for k in G.files if k.startswith("sparse_g_") and k.endswith("_val"))
    for k in _grad_keys(new):
        U.assert_sample_close(new[k], G, "sparse_" + k)
