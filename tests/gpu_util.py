import hashlib
import math
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# outputs of the unmodified reference extension on a B200 at sizes too large to store whole
# (generator: tests/golden/make_golden_sampled.py)
SAMPLED = os.path.join(GOLD, "ref_outputs_sampled.npz")


def _np(x):
    return x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def digest(x):
    """SHA-256 of an array's dtype, shape and bytes: a bit-exact comparison with a stored output."""
    a = np.ascontiguousarray(_np(x))
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_index(n, k):
    """Fixed, seeded flat positions at which a large output is stored."""
    return np.sort(np.random.RandomState(0).choice(n, min(n, k), replace=False))


def store_sample(G, key, x, k):
    """Put a seeded sample of x (+ its size and max |x| over ALL elements) into the dict G under `key`."""
    a = _np(x).reshape(-1)
    G[key + "_val"] = a[sample_index(a.size, k)].astype(np.float32)
    G[key + "_n"] = np.int64(a.size)
    G[key + "_absmax"] = np.float64(np.abs(a).max())


def load_sample(G, key, x):
    """-> (x at the stored positions, the stored values, max |value| of the whole stored tensor)."""
    a = _np(x).reshape(-1)
    assert a.size == int(G[key + "_n"]), (key, a.size, int(G[key + "_n"]))
    ref = G[key + "_val"]
    return a[sample_index(a.size, ref.size)], ref, float(G[key + "_absmax"])


def assert_sample_close(x, G, key, rel=1e-3, floor=1e-4):
    got, ref, scale = load_sample(G, key, x)
    assert_grads_close(got, ref, rel=rel, floor=floor, what=key, scale=scale)


def reference_binning(means2D, radii, depths, W, H):
    """The reference's sorted (tile, depth) instance list and per-tile ranges, rebuilt from a forward's geometry: every
    tile of each visible Gaussian's rect (getRect, auxiliary.h), keyed tile << 32 | depth bits, ties in Gaussian order
    (its radix sort is stable and duplicateWithKeys writes the instances in Gaussian order).
    -> (point_list int32 [R], ranges int32 [T, 2]; empty tiles (0, 0))."""
    dev = means2D.device
    gx, gy = (W + 15) // 16, (H + 15) // 16
    idx = torch.nonzero(radii > 0).squeeze(1)
    p, r = means2D[idx].float(), radii[idx].float()
    clamp = lambda v, g: torch.clamp(v.to(torch.int32), min=0, max=g).long()  # noqa: E731  (C casts truncate)
    x0, y0 = clamp((p[:, 0] - r) / 16, gx), clamp((p[:, 1] - r) / 16, gy)
    x1, y1 = clamp((p[:, 0] + r + 16 - 1) / 16, gx), clamp((p[:, 1] + r + 16 - 1) / 16, gy)  # float adds, in C order
    nx, ny = x1 - x0, y1 - y0
    cnt = nx * ny
    owner = torch.repeat_interleave(torch.arange(idx.numel(), device=dev), cnt)
    k = torch.arange(owner.numel(), device=dev) - torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    tile = (y0[owner] + k // nx[owner]) * gx + x0[owner] + k % nx[owner]
    key = (tile << 32) | depths[idx].view(torch.int32).long()[owner]
    key, order = torch.sort(key, stable=True)
    point_list = idx[owner[order]].to(torch.int32)
    n = torch.bincount(tile, minlength=gx * gy)
    end = torch.cumsum(n, 0)
    ranges = torch.stack([end - n, end], 1)
    ranges[n == 0] = 0
    return point_list, ranges.to(torch.int32)


def raw_args(model, cam, c, dev, D):
    """Arguments of `rasterize_gaussians` (the reference binding's signature) for a synthetic config's model and view."""
    e = torch.Tensor([])
    with torch.no_grad():
        return (torch.zeros(3, device=dev), model.get_attribute("xyz"), e, model.get_attribute("opacity"),
                model.get_attribute("scale"), model.get_attribute("rot"), 1.0, e, cam.world_view_transform,
                cam.full_proj_transform, math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5), c["H"], c["W"],
                model.get_features.contiguous(), D, cam.camera_center, False, False)


def assert_reference_outputs_and_binning(G, key, out, W, H, P):
    """`out` (a rasterize_gaussians result) against the reference's stored num_rendered, five outputs and sorted list:
    that list is rebuilt from the forward's geometry, checked against the reference's digest, and ours must be it minus
    provably inert (Gaussian, tile) pairs, in its order.  Returns (debug export, number of dropped pairs)."""
    from gaustudio_b200 import _C
    assert out[0] == int(G[key + "_R"])
    for i, name in zip(range(1, 6), ("color", "depth", "median", "opacity", "radii")):
        assert digest(out[i]) == G[f"{key}_{name}"], f"{name} not bit-identical to the reference"
    ex = _C.debug_export(P, W, H, out[0], out[6], out[7], out[8])
    pl, rg = reference_binning(ex["means2D"], out[5], ex["depths"], W, H)
    assert digest(pl) == G[key + "_point_list"] and digest(rg) == G[key + "_ranges"]
    return ex, assert_binned_list_is_culled_reference_list(ex, pl, rg, W, H, P)


def new_rasterize(rs, means3D, means2D, opacities, **kw):
    from gaustudio_b200.rasterizer import GaussianRasterizer
    return GaussianRasterizer(rs)(means3D, means2D, opacities, **kw)


def ref_rasterize(rs, means3D, means2D, opacities, **kw):
    from oracle import ref_driver
    return ref_driver.rasterize(rs, means3D, means2D, opacities, **kw)


def oracle_run(s):
    """CPU oracle outputs + grads in the naming of scenes.run_torch."""
    from oracle.oracle import Oracle
    o = Oracle()
    out = o.forward(s["means3D"], s["opacities"], s["viewmatrix"], s["projmatrix"], s["campos"], s["tanfovx"],
                    s["tanfovy"], s["W"], s["H"], s["D"], shs=s.get("shs"), colors_precomp=s.get("colors_precomp"),
                    scales=s.get("scales"), rotations=s.get("rotations"), cov3D_precomp=s.get("cov3D_precomp"),
                    scale_modifier=s["scale_modifier"])
    g = o.backward(s["dL_color"], s["dL_depth"][0], s["dL_median"], s["dL_opacity"][0], bg=s["bg"])
    r = dict(color=out["color"], radii=out["radii"], depth=out["depth"], median=out["median"], opacity=out["opacity"],
             num_rendered=out["num_rendered"], g_means2D=g["means2D"], g_means3D=g["means3D"],
             g_opacities=g["opacities"])
    if "shs" in s:
        r["g_shs"] = g["shs"]
    else:
        r["g_colors_precomp"] = g["colors_precomp"]
    if "scales" in s:
        r["g_scales"], r["g_rotations"] = g["scales"], g["rotations"]
    else:
        r["g_cov3D_precomp"] = g["cov3D_precomp"]
    return r


def assert_grads_close(a, b, rel=1e-3, floor=1e-4, what="", scale=None):
    """BASELINE: <= 1e-3 relative on gradients, with an absolute floor (relative to the tensor's scale, max |b| unless
    given) because the reference's float atomics make its own gradients order-dependent."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = np.abs(b).max() if scale is None else scale
    err = np.abs(a - b)
    bound = rel * np.abs(b) + floor * scale + 1e-30
    bad = err > bound
    assert not bad.any(), f"{what}: {int(bad.sum())}/{bad.size} beyond tolerance, worst {err.max():.3e} (scale {scale:.3e})"


def assert_images_close(a, b, atol=1e-4, outlier_frac=0.0, what=""):
    err = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
    frac = (err > atol).mean()
    assert frac <= outlier_frac, f"{what}: {frac:.2e} of pixels beyond {atol} (max {err.max():.3e})"


def assert_binned_list_is_culled_reference_list(ex, ref_point_list, ref_ranges, W, H, P):
    """The binning keeps a (Gaussian, tile) pair of the reference's rect only if the Gaussian can reach alpha >= 1/255 on
    some pixel of the tile (exact tile culling).  So the sorted list must be the REFERENCE's sorted list with entries
    removed -- same relative order -- and every removed entry must be provably inert: no pixel of its tile passes the
    reference's own `power <= 0 && alpha >= 1/255` test (forward.cu:349-355).  Returns the number of removed entries.
    ex: _C.debug_export dict; ref_point_list [R_ref], ref_ranges [>=T, 2]: the reference's (or the pinned oracle's)."""
    dev = ex["point_list"].device
    our_pl, our_rg = ex["point_list"].long(), ex["ranges"].long()
    T = our_rg.shape[0]
    ref_pl = torch.as_tensor(np.asarray(ref_point_list.cpu() if torch.is_tensor(ref_point_list) else ref_point_list).astype(np.int64)).to(dev)
    ref_rg = torch.as_tensor(np.asarray(ref_ranges.cpu() if torch.is_tensor(ref_ranges) else ref_ranges).astype(np.int64)).to(dev).reshape(-1, 2)[:T]
    tiles = torch.arange(T, device=dev)
    ref_tile = torch.repeat_interleave(tiles, ref_rg[:, 1] - ref_rg[:, 0])
    our_tile = torch.repeat_interleave(tiles, our_rg[:, 1] - our_rg[:, 0])
    assert ref_tile.numel() == ref_pl.numel(), "reference ranges do not cover its list"
    assert our_tile.numel() == our_pl.numel() == ex["num_binned"]
    ref_key, our_key = ref_tile * P + ref_pl, our_tile * P + our_pl
    kept = torch.isin(ref_key, our_key)
    assert int(kept.sum()) == our_key.numel(), "binned an instance the reference does not have"
    assert torch.equal(ref_key[kept], our_key), "binned list is not the reference's order"
    dt, dg = ref_tile[~kept], ref_pl[~kept]
    gx = (W + 15) // 16
    px0, py0 = ((dt % gx) * 16).float(), ((dt // gx) * 16).float()
    m2, co = ex["means2D"][dg], ex["conic_opacity"][dg]
    off = torch.arange(16, device=dev, dtype=torch.float32)
    step = 1 << 16
    for c in range(0, dg.numel(), step):
        sl = slice(c, c + step)
        X, Y = px0[sl, None, None] + off[None, None, :], py0[sl, None, None] + off[None, :, None]
        dx, dy = m2[sl, 0, None, None] - X, m2[sl, 1, None, None] - Y
        A, B, C, o = (co[sl, i, None, None] for i in range(4))
        power = -0.5 * (A * dx * dx + C * dy * dy) - B * dx * dy
        alpha = torch.clamp(o * torch.exp(power), max=0.99)
        live = (X < W) & (Y < H) & (power <= 0) & (alpha >= 1.0 / 255.0)
        assert not bool(live.any()), "a culled (Gaussian, tile) pair could have contributed"
    return int((~kept).sum())
