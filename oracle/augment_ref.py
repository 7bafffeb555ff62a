"""numpy restatement of isa_augment (csrc/augment.cu): the same int64 fixed-point source coordinates, bilinear weights
and normalisation in float64, then the renumbering of the surviving ids and the fallback to the plain resize map.

    augment(rgb_list, label_list, params, H, W, mean, std) -> dict(image (b,H,W,3) f64, sem, ins (b,H,W) u8, n_objects)

rgb_list[i] (h,w,3) u8 and label_list[i] (h,w) u8 (ids 0..n-1, 255 = background) are the store's images; params (b,7)
int64 rows (source index, a0..a5 in Q32.32).
"""
import numpy as np

ONE = np.int64(1) << np.int64(32)


def plain_map(h, w, H, W):
    """The plain resize map as the kernel computes it: a0 = round(w 2^32 / W), a4 = round(h 2^32 / H)."""
    return np.array([((w << 33) + W) // (2 * W), 0, 0, 0, ((h << 33) + H) // (2 * H), 0], dtype=np.int64)


def coords(a, H, W):
    """-> (u, v) int64 (H, W): the source coordinate of every output pixel centre in units of 2^-33."""
    a = np.asarray(a, dtype=np.int64)
    X = (2 * np.arange(W, dtype=np.int64) + 1)[None, :]
    Y = (2 * np.arange(H, dtype=np.int64) + 1)[:, None]
    return a[0] * X + a[1] * Y + 2 * a[2], a[3] * X + a[4] * Y + 2 * a[5]


def sample(rgb, lab, a, H, W):
    """One view through map a -> (bilinear rgb (H,W,3) float64 in 0..255, nearest labels (H,W) u8)."""
    h, w = lab.shape
    u, v = coords(a, H, W)
    ix, iy = u >> 33, v >> 33
    inside = (ix >= 0) & (ix < w) & (iy >= 0) & (iy < h)
    out_lab = np.full((H, W), 255, dtype=np.uint8)
    out_lab[inside] = lab[iy[inside], ix[inside]]
    ub, vb = u - ONE, v - ONE
    x0, y0 = ub >> 33, vb >> 33
    fx = (ub & ((ONE << 1) - 1)).astype(np.float64) / 2.0 ** 33
    fy = (vb & ((ONE << 1) - 1)).astype(np.float64) / 2.0 ** 33

    def tap(xx, yy):
        ok = (xx >= 0) & (xx < w) & (yy >= 0) & (yy < h)
        t = np.zeros((H, W, 3), dtype=np.float64)
        t[ok] = rgb[yy[ok], xx[ok]]
        return t

    fx, fy = fx[..., None], fy[..., None]
    top = (1 - fx) * tap(x0, y0) + fx * tap(x0 + 1, y0)
    bot = (1 - fx) * tap(x0, y0 + 1) + fx * tap(x0 + 1, y0 + 1)
    return (1 - fy) * top + fy * bot, out_lab


def renumber(lab):
    """ids present -> 0..n-1 in ascending order of the old id; -> (labels, n)."""
    ids = np.unique(lab[lab != 255])
    lut = np.full(256, 255, dtype=np.uint8)
    lut[ids] = np.arange(len(ids), dtype=np.uint8)
    return lut[lab], len(ids)


def augment(rgb_list, label_list, params, H, W, mean, std):
    params = np.asarray(params, dtype=np.int64).reshape(-1, 7)
    b = params.shape[0]
    mean = np.asarray(mean, dtype=np.float64)
    std = np.asarray(std, dtype=np.float64)
    image = np.empty((b, H, W, 3), dtype=np.float64)
    ins = np.empty((b, H, W), dtype=np.uint8)
    n_objects = np.empty(b, dtype=np.int32)
    for i in range(b):
        src, a = int(params[i, 0]), params[i, 1:]
        rgb, lab = rgb_list[src], label_list[src]
        val, out_lab = sample(rgb, lab, a, H, W)
        if not (out_lab != 255).any():
            val, out_lab = sample(rgb, lab, plain_map(lab.shape[0], lab.shape[1], H, W), H, W)
        ins[i], n_objects[i] = renumber(out_lab)
        image[i] = (val / 255.0 - mean) / std
    return dict(image=image, sem=(ins != 255).astype(np.uint8), ins=ins, n_objects=n_objects)
