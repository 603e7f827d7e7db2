"""-m gpu parity at the FULL size of every BASELINE.json configuration a number is quoted on, in the mode it is
quoted in (VERDICT r1, next-round item 1):
  cfg 1  10k / 256x256, forward RGB           vs the CPU oracle and the compiled reference
  cfg 2  100k / 800x800, fwd+bwd              gradients vs the compiled reference
  cfg 3  1M / 1080p in bench.py's DEFAULT mode (fused activations + pipelined forward + one CUDA-graph replay per view)
         vs the compiled reference chained through the reference's torch activations
  cfg 5  5M / 1440x1080 forward only, D=3 and D=0 with M=16  vs the compiled reference (bit-exact, incl. sort order)
The reference's side is what it computed on a B200, stored in tests/golden/ref_outputs_sampled.npz: digests of the
outputs compared bit for bit, seeded samples of those compared within a tolerance.
Tolerances: BASELINE.json -- 1e-4 max-abs on images (bit-exact where the arithmetic is identical), 1e-3 relative on
gradients with a floor relative to the tensor's scale (the reference's own float atomics are order-dependent)."""
import math

import numpy as np
import pytest
import torch

import gpu_util as U

pytestmark = pytest.mark.gpu
NAMES = ("color", "depth", "median", "opacity", "radii")


@pytest.fixture(scope="module")
def G():
    return np.load(U.SAMPLED)


def _grad_bad_fraction(G, key, x, rel=1e-3, floor=1e-4):
    """Fraction of the stored sample of the reference's gradient `key` that x misses (floor relative to the whole
    reference tensor's max |value|)."""
    x, y, scale = U.load_sample(G, key, x)
    return float((np.abs(x - y) > rel * np.abs(y) + floor * scale).mean())


def _weights(c, dev, seed):
    g = torch.Generator().manual_seed(seed)
    H, W = c["H"], c["W"]
    return [torch.randn(s, H, W, generator=g).to(dev) for s in (3, 1, 1)]


def _weighted(out, w):
    return (out["render"] * w[0]).sum() + (out["rendered_depth"] * w[1]).sum() + (out["rendered_final_opacity"] * w[2]).sum()


def test_cfg1_real_size_forward_vs_oracle_and_reference(G):
    from gaustudio_b200 import _C
    from gaustudio_b200.synthetic import build_config
    from oracle.oracle import Oracle
    model, cams, c = build_config("cfg1")
    assert c["P"] == 10_000 and (c["W"], c["H"]) == (256, 256)
    dev = torch.device("cuda")
    cam = cams[0]
    o = Oracle()
    with torch.no_grad():
        orc = o.forward(model.get_attribute("xyz").numpy(), model.get_attribute("opacity").numpy(),
                        cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), cam.camera_center.numpy(),
                        math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5), 256, 256, 3, shs=model.get_features.numpy(),
                        scales=model.get_attribute("scale").numpy(), rotations=model.get_attribute("rot").numpy())
    model.to(dev); cam.to(dev)
    new = _C.rasterize_gaussians(*U.raw_args(model, cam, c, dev, 3))
    assert new[0] == int(G["cfg1_R"]) == orc["num_rendered"]
    for i, name in zip(range(1, 6), NAMES):
        assert U.digest(new[i]) == G["cfg1_" + name], name
    err = np.abs(new[1].cpu().numpy() - orc["color"])
    assert (err > 1e-4).mean() < 2e-3 and np.median(err) < 1e-6, err.max()
    assert (new[5].cpu().numpy() != orc["radii"]).mean() < 1e-3


def test_cfg2_full_size_gradients_vs_reference(G):
    from gaustudio_b200 import renderers
    from gaustudio_b200.synthetic import build_config
    model, cams, c = build_config("cfg2", K=4)
    assert c["P"] == 100_000 and (c["W"], c["H"]) == (800, 800)
    dev = torch.device("cuda")
    model.to(dev).requires_grad_(True)
    names = ("xyz", "scale", "rot", "opacity", "f_dc", "f_rest")
    for k, cam in enumerate(cams[:2]):
        cam.to(dev)
        w = _weights(c, dev, 21 + k)
        key = f"cfg2_v{k}"
        for fused in (False, True):
            for p in model.parameters_list():
                p.grad = None
            out = renderers.make({"name": "vanilla_renderer", "fused_activations": fused}).render(cam, model)
            _weighted(out, w).backward()
            if not fused:  # identical inputs -> identical forward
                assert U.digest(out["render"]) == G[key + "_render"]
                assert U.digest(out["rendered_depth"]) == G[key + "_rendered_depth"]
            for n, p in zip(names, model.parameters_list()):
                bad = _grad_bad_fraction(G, f"{key}_{n}", p.grad)
                assert bad < 1e-5, (n, fused, bad)


def test_cfg3_bench_default_mode_matches_reference(G):
    """fused activations + pipelined (fixed-capacity) forward + CUDA-graph replay: the mode bench.py times."""
    from gaustudio_b200 import _C, renderers
    from gaustudio_b200.graphs import GraphedViewStep
    from gaustudio_b200.synthetic import build_config
    model, cams, c = build_config("cfg3", K=8)
    dev = torch.device("cuda")
    model.to(dev).requires_grad_(True)
    cams = [cm.to(dev) for cm in cams[:3]]
    w = _weights(c, dev, 5)
    r = renderers.make({"name": "vanilla_renderer", "fused_activations": True})
    before = _C.pipeline_state()
    step = GraphedViewStep(r, model, lambda out: _weighted(out, w), cams)
    assert _C.pipeline_state()["enabled"] == before["enabled"] and _C.pipeline_state()["fixed"] == before["fixed"]
    names = ("xyz", "scale", "rot", "opacity", "f_dc", "f_rest")
    for v, cam in enumerate(cams[1:]):
        step(cam)                                         # one graph replay
        torch.cuda.synchronize()
        got = {k: step.out[k].detach().clone() for k in ("render", "rendered_depth", "rendered_final_opacity")}
        got_g = [g.detach().clone() for g in step.grads]
        key = f"cfg3_v{v}"
        for k in got:
            x, y, _ = U.load_sample(G, f"{key}_{k}", got[k])
            err = np.abs(x.astype(np.float64) - y)
            # fused exp / sigmoid / normalize round differently from the torch ops by ulps: a hard-threshold flip
            # (alpha < 1/255, T < 1e-4, tile rect) moves a pixel by more than 1e-4, hence a small outlier budget
            assert float((err > 1e-4).mean()) < 1e-3, (k, float(err.max()))
            assert float(np.median(err)) < 1e-6
        for n, x in zip(names, got_g):
            bad = _grad_bad_fraction(G, f"{key}_{n}", x)
            assert bad < 1e-4, (n, bad)
    assert 0 < step.max_rendered() <= step.capacity


@pytest.mark.parametrize("D", [3, 0])
def test_cfg5_full_size_forward_bit_exact_vs_reference(G, D):
    """5M Gaussians, 1440x1080, the extraction-pass shape (forward only); D = 0 reads 12 of each 192-byte SH row
    (quirk 13).  All five outputs and num_rendered are identical to the reference's; the sorted list is the reference's
    minus provably inert (Gaussian, tile) pairs, in the reference's order."""
    from gaustudio_b200 import _C
    from gaustudio_b200.synthetic import build_config
    model, cams, c = build_config("cfg5", K=8)
    assert c["P"] == 5_000_000 and (c["W"], c["H"]) == (1440, 1080)
    dev = torch.device("cuda")
    model.to(dev)
    cam = cams[1].to(dev)
    with torch.no_grad():
        new = _C.rasterize_gaussians(*U.raw_args(model, cam, c, dev, D))
    assert new[0] > 10_000_000
    ex, dropped = U.assert_reference_outputs_and_binning(G, f"cfg5_D{D}", new, c["W"], c["H"], c["P"])
    assert ex["num_binned"] == new[0] - dropped
    n = (ex["ranges"][:, 1] - ex["ranges"][:, 0]).long()
    assert int(n.max()) > 4096, int(n.max())  # the crowded-tile sort tier is exercised (larger tiers: test_gpu_api)
    del new, ex
    torch.cuda.empty_cache()
