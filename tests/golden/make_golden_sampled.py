"""Generates tests/golden/ref_outputs_sampled.npz by running the UNMODIFIED reference CUDA extension
(oracle/_ref/_refC.so, built by oracle/build_ref.py) on a B200, on the inputs of the GPU tests that compare with it
at sizes too large to store whole:

    python tests/golden/make_golden_sampled.py [OUT_DIR]      # writes OUT_DIR/ref_outputs_sampled.npz

Outputs compared bit for bit are stored as digests (gpu_util.digest); outputs compared within a tolerance as a fixed,
seeded sample (gpu_util.store_sample) with the max |value| of the whole tensor.  The reference's sorted instance list
is stored as a digest too: the tests rebuild it from the forward's geometry (gpu_util.reference_binning), and this
script checks that the rebuild equals the reference's own list.  The JSON report it prints holds, for each stored
quantity, how this package's result compares with the reference's over the WHOLE tensor.
"""
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gpu_util as U  # noqa: E402
import scenes  # noqa: E402
import test_gpu_fullsize as F  # noqa: E402
import test_gpu_parity as PAR  # noqa: E402
from gaustudio_b200 import _C, renderers  # noqa: E402
from gaustudio_b200.graphs import GraphedViewStep  # noqa: E402
from gaustudio_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer  # noqa: E402
from gaustudio_b200.synthetic import build_config  # noqa: E402
from oracle import ref_driver, ref_torch_ops  # noqa: E402

K_GRAD, K_IMG = 512, 2048
NAMES = ("color", "depth", "median", "opacity", "radii")
PARAMS = ("xyz", "scale", "rot", "opacity", "f_dc", "f_rest")
dev = torch.device("cuda")
G, report = {}, {}


def bad_fraction(x, y, rel=1e-3, floor=1e-4):
    x, y = (np.asarray(U._np(v), np.float64) for v in (x, y))
    return float((np.abs(x - y) > rel * np.abs(y) + floor * np.abs(y).max()).mean())


def put_outputs(key, ref, new):
    """num_rendered + digests of the five forward outputs of a rasterize_gaussians result."""
    G[key + "_R"] = np.int64(ref[0])
    rep = {"R_equal": int(new[0]) == int(ref[0])}
    for i, name in zip(range(1, 6), NAMES):
        G[f"{key}_{name}"] = U.digest(ref[i])
        rep[name + "_bit_exact"] = bool(torch.equal(new[i], ref[i]))
    return rep


def put_binning(key, ref, new, W, H, P):
    T = ((W + 15) // 16) * ((H + 15) // 16)
    pl = ref_driver.parse_binning(ref[7], ref[0])
    rg = ref_driver.parse_image_ranges(ref[8], W * H, T)
    G[key + "_point_list"], G[key + "_ranges"] = U.digest(pl), U.digest(rg)
    ex = _C.debug_export(P, W, H, new[0], new[6], new[7], new[8])
    rpl, rrg = U.reference_binning(ex["means2D"], new[5], ex["depths"], W, H)
    return {"rebuilt_list_equal": bool(torch.equal(rpl, pl)), "rebuilt_ranges_equal": bool(torch.equal(rrg, rg))}


def ref_step(model, cam, c, D, w):
    """The reference's op sequence: torch activations -> its CUDA extension -> loss -> backward (raw-attribute grads)."""
    for p in model.parameters_list():
        p.grad = None
    xyz, shs, opacity, scales, rotations = ref_torch_ops.gaussian_properties(model)
    rs = ref_driver.RefSettings(c["H"], c["W"], math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5),
                                torch.zeros(3, device=dev), 1.0, cam.world_view_transform, cam.full_proj_transform, D,
                                cam.camera_center, False, False)
    color, radii, depth, median, opac = ref_driver.rasterize(rs, xyz, torch.zeros_like(xyz, requires_grad=True) + 0,
                                                             opacity, shs=shs, scales=scales, rotations=rotations)
    out = {"render": color, "rendered_depth": depth, "rendered_final_opacity": opac}
    F._weighted(out, w).backward()
    return {k: v.detach().clone() for k, v in out.items()}, [p.grad.detach().clone() for p in model.parameters_list()]


def ref_case_fixtures():
    """The committed whole-array fixtures still equal what the reference computes (bit for bit in the forward)."""
    for case in "ABCD":
        f = np.load(os.path.join(U.GOLD, f"ref_case_{case}.npz"))
        s = scenes.scene(case)
        ref = scenes.run_torch(s, U.ref_rasterize, dev)
        new = scenes.run_torch(s, U.new_rasterize, dev)
        report[f"ref_case_{case}"] = {
            "fixture_eq_live_ref": {k: bool(np.array_equal(ref[k], f["ref_" + k])) for k in NAMES},
            "new_eq_fixture": {k: bool(np.array_equal(new[k], f["ref_" + k])) for k in NAMES},
            "grad_bad_new_vs_fixture": {k: bad_fraction(new[k], f["ref_" + k]) for k in new if k.startswith("g_")}}


def sh_degrees():
    s = scenes.scene("A")
    for D in (0, 1, 2, 3):
        s["D"] = D
        ref = scenes.run_torch(s, U.ref_rasterize, dev)
        new = scenes.run_torch(s, U.new_rasterize, dev)
        G[f"sh_D{D}_color"] = U.digest(ref["color"])
        U.store_sample(G, f"sh_D{D}_g_shs", ref["g_shs"], K_GRAD)
        report[f"sh_D{D}"] = {"color_bit_exact": bool(np.array_equal(new["color"], ref["color"])),
                              "g_shs_bad": bad_fraction(new["g_shs"], ref["g_shs"])}


def sparse():
    s = PAR.sparse_scene()
    ref = scenes.run_torch(s, U.ref_rasterize, dev)
    new = scenes.run_torch(s, U.new_rasterize, dev)
    rep = {}
    for k in ("color", "depth", "median", "opacity", "radii"):
        G["sparse_" + k] = U.digest(ref[k])
        rep[k + "_bit_exact"] = bool(np.array_equal(new[k], ref[k]))
    for k in sorted(k for k in ref if k.startswith("g_")):
        U.store_sample(G, "sparse_" + k, ref[k], K_GRAD)
        rep[k + "_bad"] = bad_fraction(new[k], ref[k])
    report["sparse"] = rep


def medium():
    model, cams, c = build_config("cfg2", K=3)
    model.to(dev)
    for v, cam in enumerate(cams[:2]):
        cam.to(dev)
        with torch.no_grad():
            a = U.raw_args(model, cam, c, dev, 3)
            new, ref = _C.rasterize_gaussians(*a), ref_driver.module().rasterize_gaussians(*a)
        key = f"medium_v{v}"
        report[key] = put_outputs(key, ref, new)
        report[key].update(put_binning(key, ref, new, c["W"], c["H"], c["P"]))


def cfg1():
    model, cams, c = build_config("cfg1")
    model.to(dev)
    cam = cams[0].to(dev)
    a = U.raw_args(model, cam, c, dev, 3)
    report["cfg1"] = put_outputs("cfg1", ref_driver.module().rasterize_gaussians(*a), _C.rasterize_gaussians(*a))


def cfg2():
    model, cams, c = build_config("cfg2", K=4)
    model.to(dev).requires_grad_(True)
    for k, cam in enumerate(cams[:2]):
        cam.to(dev)
        w = F._weights(c, dev, 21 + k)
        key = f"cfg2_v{k}"
        ro, rg = ref_step(model, cam, c, 3, w)
        G[key + "_render"], G[key + "_rendered_depth"] = U.digest(ro["render"]), U.digest(ro["rendered_depth"])
        rep = {}
        for n, g in zip(PARAMS, rg):
            U.store_sample(G, f"{key}_{n}", g, K_GRAD)
        for fused in (False, True):
            for p in model.parameters_list():
                p.grad = None
            out = renderers.make({"name": "vanilla_renderer", "fused_activations": fused}).render(cam, model)
            F._weighted(out, w).backward()
            if not fused:
                rep["render_bit_exact"] = bool(torch.equal(out["render"], ro["render"]))
                rep["depth_bit_exact"] = bool(torch.equal(out["rendered_depth"], ro["rendered_depth"]))
            for n, p, g in zip(PARAMS, model.parameters_list(), rg):
                rep[f"{n}_fused{int(fused)}_bad"] = bad_fraction(p.grad, g)
        report[key] = rep


def cfg3():
    model, cams, c = build_config("cfg3", K=8)
    model.to(dev).requires_grad_(True)
    cams = [cm.to(dev) for cm in cams[:3]]
    w = F._weights(c, dev, 5)
    step = GraphedViewStep(renderers.make({"name": "vanilla_renderer", "fused_activations": True}), model,
                           lambda out: F._weighted(out, w), cams)
    for v, cam in enumerate(cams[1:]):
        step(cam)
        torch.cuda.synchronize()
        got = {k: step.out[k].detach().clone() for k in ("render", "rendered_depth", "rendered_final_opacity")}
        got_g = [g.detach().clone() for g in step.grads]
        ro, rg = ref_step(model, cam, c, 3, w)
        key, rep = f"cfg3_v{v}", {}
        for k in got:
            U.store_sample(G, f"{key}_{k}", ro[k], K_IMG)
            err = (got[k] - ro[k]).abs()
            x, y, _ = U.load_sample(G, f"{key}_{k}", got[k])
            es = np.abs(x.astype(np.float64) - y)
            rep[k] = {"outlier_frac": float((err > 1e-4).float().mean()), "median": float(err.median()),
                      "sample_outlier_frac": float((es > 1e-4).mean()), "sample_median": float(np.median(es))}
        for n, x, g in zip(PARAMS, got_g, rg):
            U.store_sample(G, f"{key}_{n}", g, K_GRAD)
            rep[n + "_bad"] = bad_fraction(x, g)
        report[key] = rep


def cfg3_full():
    model, cams, c = build_config("cfg3", K=8)
    model.to(dev)
    cam = cams[0].to(dev)
    a = U.raw_args(model, cam, c, dev, 3)
    report["cfg3full"] = put_outputs("cfg3full", ref_driver.module().rasterize_gaussians(*a),
                                     _C.rasterize_gaussians(*a))
    rs = GaussianRasterizationSettings(c["H"], c["W"], math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5),
                                       torch.zeros(3, device=dev), 1.0, cam.world_view_transform,
                                       cam.full_proj_transform, 3, cam.camera_center, False, False)
    g = torch.Generator().manual_seed(11)
    wc = torch.randn(3, c["H"], c["W"], generator=g).to(dev); wd = torch.randn(1, c["H"], c["W"], generator=g).to(dev)

    def grads(fn):
        with torch.no_grad():
            leaves = [model.get_attribute("xyz").clone(), model.get_attribute("opacity").clone(),
                      model.get_attribute("scale").clone(), model.get_attribute("rot").clone(), model.get_features.clone()]
        xyz, op, sc, rot, sh = [t.requires_grad_(True) for t in leaves]
        color, radii, depth, median, opac = fn(rs, xyz, torch.zeros_like(xyz), op, shs=sh, scales=sc, rotations=rot)
        ((color * wc).sum() + (depth * wd).sum() + opac.sum()).backward()
        return [t.grad for t in (xyz, op, sc, rot, sh)]
    gn = grads(lambda rs_, *a_, **k: GaussianRasterizer(rs_)(*a_, **k))
    gr = grads(ref_driver.rasterize)
    for name, x, y in zip(("xyz", "opacity", "scale", "rot", "sh"), gn, gr):
        U.store_sample(G, "cfg3full_g_" + name, y, K_GRAD)
        report["cfg3full"][name + "_bad"] = bad_fraction(x, y)


def cfg5():
    model, cams, c = build_config("cfg5", K=8)
    model.to(dev)
    cam = cams[1].to(dev)
    for D in (3, 0):
        a = U.raw_args(model, cam, c, dev, D)
        with torch.no_grad():
            new, ref = _C.rasterize_gaussians(*a), ref_driver.module().rasterize_gaussians(*a)
        key = f"cfg5_D{D}"
        report[key] = put_outputs(key, ref, new)
        report[key].update(put_binning(key, ref, new, c["W"], c["H"], c["P"]))
        del new, ref, a
        torch.cuda.empty_cache()


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else U.GOLD
    os.makedirs(out, exist_ok=True)
    assert ref_driver.available(), "oracle/_ref/_refC.so missing: build it with oracle/build_ref.py"
    for fn in (ref_case_fixtures, sh_degrees, sparse, medium, cfg1, cfg2, cfg3, cfg3_full, cfg5):
        fn()
        print(fn.__name__, "done", flush=True)
    np.savez_compressed(os.path.join(out, "ref_outputs_sampled.npz"), **G)
    print(json.dumps({"device": torch.cuda.get_device_name(0), "report": report}, indent=1))


if __name__ == "__main__":
    main()
