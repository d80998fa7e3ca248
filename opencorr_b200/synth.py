"""Synthetic speckle pairs / volumes with known displacement fields (SURVEY.md section 8(d)).

The reference ships no generator; bench.py and the tests use this one.  Gaussian-speckle model,
8-bit quantised then cast to float for 2D (the reference only ever sees 8-bit-valued floats in
2D, src/oc_image.cpp:39,56): I(x) = clip(B + (255 - B) * sum_k a_k exp(-|x - c_k|^2 / rho^2)), the
target is rendered analytically from displaced centres c_k' = c_k + u(c_k).

The background level B = 24 is a deliberate departure from SURVEY.md's formula (B = 0): the
reference treats ANY interpolated sample < 0 as "outside the image" (src/oc_icgn.cpp:251-255), and
bicubic/tricubic overshoot next to truly black pixels produces such samples, so a pattern with a
zero background makes the reference reject every POI with ZNCC = -3.
"""
import numpy as np

REF_SEED = 20260924
BACKGROUND = 24.0


def _render_torch(shape, centres, amps, rho, device):
    """Same as _render on a torch device (float64 accumulation); used for the large bench inputs."""
    import torch
    nd = len(shape)
    c = torch.as_tensor(centres, dtype=torch.float64, device=device)
    a = torch.as_tensor(amps, dtype=torch.float64, device=device)
    img = torch.zeros(int(np.prod(shape)), dtype=torch.float64, device=device)
    base = torch.floor(c).to(torch.int64)
    half = int(np.ceil(3.5 * rho))
    rng = torch.arange(-half, half + 1, device=device)
    offs = torch.stack([g.reshape(-1) for g in torch.meshgrid(*([rng] * nd), indexing="ij")], 1)
    lim = torch.tensor(shape, device=device)
    strides = torch.tensor([int(np.prod(shape[i + 1:])) for i in range(nd)], dtype=torch.int64, device=device)
    inv = 1.0 / (rho * rho)
    # centres that share a pixel cell add to the same pixel in one index_add_; on CUDA its default atomics add them in a
    # different order from run to run, and the last bit can round a pixel the other way: deterministic mode fixes the order,
    # so the same arguments render the same images every time
    was_deterministic = torch.are_deterministic_algorithms_enabled()
    was_warn_only = torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        for o in offs:
            p = base + o
            ok = ((p >= 0) & (p < lim)).all(1)
            d2 = ((p[ok].to(torch.float64) - c[ok]) ** 2).sum(1)
            img.index_add_(0, (p[ok] * strides).sum(1), a[ok] * torch.exp(-d2 * inv))
    finally:
        torch.use_deterministic_algorithms(was_deterministic, warn_only=was_warn_only)
    return img.reshape(shape).cpu().numpy()


def _render(shape, centres, amps, rho, device=None):
    """Sum of isotropic Gaussians, evaluated within +-3.5 rho of each centre (numpy, any dim)."""
    if device is not None:
        return _render_torch(shape, centres, amps, rho, device)
    nd = len(shape)
    img = np.zeros(int(np.prod(shape)), np.float64)
    base = np.floor(centres).astype(np.int64)
    half = int(np.ceil(3.5 * rho))
    rng = np.arange(-half, half + 1)
    grids = np.meshgrid(*([rng] * nd), indexing="ij")
    offs = np.stack([g.ravel() for g in grids], axis=1)  # [K, nd], order (z,)y,x
    inv = 1.0 / (rho * rho)
    strides = np.array([int(np.prod(shape[i + 1:])) for i in range(nd)], np.int64)
    for o in offs:
        p = base + o
        ok = np.all((p >= 0) & (p < np.array(shape)), axis=1)
        d2 = np.sum((p[ok] - centres[ok]) ** 2, axis=1)
        np.add.at(img, p[ok] @ strides, amps[ok] * np.exp(-d2 * inv))
    return img.reshape(shape)


def displacement_2d(x, y, width, height, second_order=False):
    """u, v at pixel positions (x, y); x~, y~ are relative to the image centre."""
    xt, yt = x - 0.5 * width, y - 0.5 * height
    u = 2.37 + 1.5e-3 * xt - 0.8e-3 * yt
    v = -1.62 + 0.6e-3 * xt + 2.1e-3 * yt
    if second_order:
        u = u + 2e-6 * xt * xt - 1e-6 * xt * yt + 1.5e-6 * yt * yt
        v = v + 1.5e-6 * xt * xt - 1e-6 * xt * yt + 2e-6 * yt * yt
    return u, v


def displacement_3d(x, y, z, dim_x, dim_y, dim_z):
    xt, yt, zt = x - 0.5 * dim_x, y - 0.5 * dim_y, z - 0.5 * dim_z
    return 1.3 + 1e-3 * xt, -0.7 + 1.2e-3 * yt, 2.4 - 1.5e-3 * zt


def speckle_pair_2d(width, height, second_order=False, rho=2.0, seed=REF_SEED, quantise=True, device=None, background=BACKGROUND):
    """(ref, tar) float32 [height, width].  background=0 is SURVEY.md's formula (truly black gaps between the speckles)."""
    rng = np.random.default_rng(seed)
    n = int(0.5 * width * height / (np.pi * rho * rho))
    cx = rng.uniform(-8, width + 8, n)
    cy = rng.uniform(-8, height + 8, n)
    amp = rng.uniform(0.4, 1.0, n)
    ref = _render((height, width), np.stack([cy, cx], 1), amp, rho, device)
    u, v = displacement_2d(cx, cy, width, height, second_order)
    tar = _render((height, width), np.stack([cy + v, cx + u], 1), amp, rho, device)
    out = []
    for im in (ref, tar):
        im = np.clip(background + (255.0 - background) * im, 0, 255)
        if quantise:
            im = np.round(im)
        out.append(im.astype(np.float32))
    return out[0], out[1]


def speckle_pair_3d(dim_x, dim_y, dim_z, rho=2.0, seed=REF_SEED, quantise=True, device=None, background=BACKGROUND):
    """(ref, tar) float32 [dim_z, dim_y, dim_x]."""
    rng = np.random.default_rng(seed)
    n = int(0.35 * dim_x * dim_y * dim_z / (4.0 / 3.0 * np.pi * rho ** 3))
    cx = rng.uniform(-8, dim_x + 8, n)
    cy = rng.uniform(-8, dim_y + 8, n)
    cz = rng.uniform(-8, dim_z + 8, n)
    amp = rng.uniform(0.4, 1.0, n)
    ref = _render((dim_z, dim_y, dim_x), np.stack([cz, cy, cx], 1), amp, rho, device)
    u, v, w = displacement_3d(cx, cy, cz, dim_x, dim_y, dim_z)
    tar = _render((dim_z, dim_y, dim_x), np.stack([cz + w, cy + v, cx + u], 1), amp, rho, device)
    out = []
    for im in (ref, tar):
        im = np.clip(background + (255.0 - background) * im, 0, 255)
        if quantise:
            im = np.round(im)
        out.append(im.astype(np.float32))
    return out[0], out[1]


def grid_2d(x0, y0, nx, ny, sx, sy):
    """POI grid, row-major over y then x like the reference examples (test_2d_dic_fftcc_icgn1.cpp:57-66)."""
    ys, xs = np.meshgrid(y0 + sy * np.arange(ny), x0 + sx * np.arange(nx), indexing="ij")
    return np.stack([xs.ravel(), ys.ravel()], 1).astype(np.float32)


def grid_3d(x0, y0, z0, nx, ny, nz, sx, sy, sz):
    zs, ys, xs = np.meshgrid(z0 + sz * np.arange(nz), y0 + sy * np.arange(ny), x0 + sx * np.arange(nx), indexing="ij")
    return np.stack([xs.ravel(), ys.ravel(), zs.ravel()], 1).astype(np.float32)


# BASELINE.json configs (SURVEY.md section 8(d)): image size, POI grid, subset radius, path
CONFIGS = {
    "A": dict(kind="2d", size=(512, 512), grid=(48, 48, 20, 10, 20, 40), r=15, order=1, conv=1e-3, stop=10),
    "B": dict(kind="2d", size=(2048, 2048), grid=(64, 64, 250, 200, 7, 9), r=16, order=1, conv=1e-3, stop=10),
    "C": dict(kind="2d", size=(2048, 2048), grid=(64, 64, 250, 200, 7, 9), r=20, order=2, conv=1e-3, stop=10),
    "D": dict(kind="3d", size=(256, 256, 256), grid=(40, 40, 40, 40, 25, 20, 4, 7, 8), r=16, order=1, conv=1e-3, stop=20),
    "E": dict(kind="2d", size=(4096, 4096), grid=(128, 128, 1000, 500, 3, 7), r=16, order=1, conv=1e-3, stop=10),
    # not a BASELINE.json config: the geometry of the reference's own DVC example (examples/test_dvc_fftcc_icgn1.cpp:
    # 61^3 subvolumes, stop 20) on a synthetic volume, for the record in profiles/
    "F": dict(kind="3d", size=(288, 288, 288), grid=(40, 40, 40, 12, 12, 12, 19, 19, 19), r=30, order=1, conv=1e-3, stop=20),
}
