"""rt_frame_denoise restated in numpy float32 (include/rtfs_b200.h): the device filter must equal this bit for bit.

numpy evaluates every float32 operation below with IEEE round-to-nearest and without contraction, in the order written, and
the device kernels (csrc/rtfs_denoise.cu) spell each operation as an intrinsic in the same order."""
import numpy as np

from test_noise_cpu import numpy_se

F = np.float32
B3 = (1, 4, 6, 4, 1)


def edge_weight(x):
    """W(x) = 1 / (1 + x (1 + x / 2)): 1 at 0, 0 at +inf."""
    return F(1) / (F(1) + x * (F(1) + F(0.5) * x))


def gamma_lut(gamma):
    """PixelOutput.correct of every 8-bit mean (fill_gamma_lut): Math.Round (half to even) of sqrt(i / 255) * 255."""
    i = np.arange(256)
    if not gamma:
        return i.astype(np.uint8)
    return np.minimum(np.rint(np.sqrt(i / 255.0) * 255.0), 255).astype(np.uint8)


def denoise(sums, sq, albedo, normal, depth, iterations, sigma_colour, sigma_normal, sigma_albedo, sigma_depth, gamma=False,
            view_rows=None):
    """(rgb uint8 [..., 3], linear float32 [..., 3]) of a frame: sums int32 [rows, cols, 4] and Q uint64 [rows, cols] as
    rt_frame_read and rt_frame_noise give them, features as rt_frame_features gives them.  A batch of views has a leading view
    axis ([n_views, rows, cols, ...]) and is filtered as rt_frame_denoise filters its tall frame; view_rows cuts a tall frame
    given without that axis."""
    shape = np.shape(sums)[:-1]
    if len(shape) == 3:  # a batch: the tall frame, views of shape[1] rows
        view_rows = shape[1]
    rows, cols = int(np.prod(shape[:-1])), shape[-1]
    view_rows = rows if view_rows is None else view_rows
    sums = np.asarray(sums).reshape(rows, cols, 4)
    albedo = np.asarray(albedo).reshape(rows, cols, 3).astype(F)
    normal = np.asarray(normal, F).reshape(rows, cols, 3)
    z = np.asarray(depth, F).reshape(rows, cols)
    n = sums[..., 3]
    valid = n > 0
    with np.errstate(all="ignore"):
        cur = np.where(valid[..., None], sums[..., :3].astype(F) / n[..., None].astype(F), F(0)).astype(F)
        e = numpy_se(sums, np.asarray(sq).reshape(rows, cols)).astype(F)
        v = e * e
        sn, sa, sz = F(sigma_normal), F(sigma_albedo), F(sigma_depth)
        sn2, sa2 = sn * sn, sa * sa
        zscale = sz * z
        r_idx, c_idx = np.arange(rows), np.arange(cols)
        for k in range(iterations):
            step = 1 << k
            sc = F(sigma_colour) * F(2.0 ** -k)
            sc2 = sc * sc
            ws = np.zeros((rows, cols), F)
            acc = np.zeros((rows, cols, 3), F)
            for j in range(5):
                rr = r_idx + (j - 2) * step
                in_r = (rr >= 0) & (rr < rows) & (rr // view_rows == r_idx // view_rows)
                rq = np.clip(rr, 0, rows - 1)
                for i in range(5):
                    cc = c_idx + (i - 2) * step
                    in_c = (cc >= 0) & (cc < cols)
                    cq = np.clip(cc, 0, cols - 1)

                    def take(a):
                        return a[rq][:, cq]

                    m = in_r[:, None] & in_c[None, :] & take(valid)
                    c_q = take(cur)
                    dcol = cur - c_q
                    d = (dcol[..., 0] * dcol[..., 0] + dcol[..., 1] * dcol[..., 1]) + dcol[..., 2] * dcol[..., 2]
                    xc = np.where(d == 0, F(0), d / (sc2 * (v + take(v))))
                    dnv = normal - take(normal)
                    xn = ((dnv[..., 0] * dnv[..., 0] + dnv[..., 1] * dnv[..., 1]) + dnv[..., 2] * dnv[..., 2]) / sn2
                    dav = albedo - take(albedo)
                    xa = ((dav[..., 0] * dav[..., 0] + dav[..., 1] * dav[..., 1]) + dav[..., 2] * dav[..., 2]) / sa2
                    zq = take(z)
                    t = (z - zq) / zscale
                    xz = np.where(z == zq, F(0), np.where(np.isinf(z) | np.isinf(zq), F(np.inf), t * t))
                    w = F(B3[j] * B3[i]) * edge_weight(xc) * edge_weight(xn) * edge_weight(xa) * edge_weight(xz)
                    w = np.where(m, w, F(0)).astype(F)
                    ws = ws + w
                    acc = acc + w[..., None] * np.where(m[..., None], c_q, F(0))
            cur = np.where(valid[..., None], acc / ws[..., None], cur).astype(F)
    rgb = gamma_lut(gamma)[np.clip(cur, F(0), F(255)).astype(np.int64)]
    return rgb.reshape(shape + (3,)), cur.reshape(shape + (3,))
