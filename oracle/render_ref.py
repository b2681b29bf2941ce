"""NumPy restatement of the mesh overlay contract of tp_render_meshes (include/tepose_b200.h) -- TEST INFRASTRUCTURE (tests/
import it; the product never does).  Every rounding step of csrc/render.cu has its twin here, so the device's frames are pinned
bit for bit:

- project: fp32 u = (sx*(X+tx)+1)*(W/2), v = (sy*(Y+ty)+1)*(H/2), each operation rounded on its own; q = rint(256 u);
  a vertex is usable when X, Y, Z are finite and |u|, |v| <= 2^15;
- setup: a face with an unusable vertex or zero int64 area draws nothing; negative area swaps vertices 1 and 2;
- coverage: int64 edge functions at the pixel centre (256x+128, 256y+128), top-left rule ("nudge right, then down");
- visibility: the smallest key (n-1-person) << 48 | depth bits << 16 | face, depth = fp32(((w0 z0 + w1 z1) + w2 z2) * (1/area))
  in float64;
- shading in float64: unit face normals, vertex normals summed in CSR order and normalised, interpolated with the integer
  weights, normalised; colour * (0.3 + 0.7 |n_z|) * 255, clamped to [0, 255], rounded half to even.

It takes the tensors the renderer is given (faces, vertex -> face CSR, verts, orig_cam, colors) as they are.
"""
import numpy as np

GUARD = np.float32(32768.0)
EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)


def _np(a, dtype=None):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    return a if dtype is None else a.astype(dtype)


def project(verts, cam, H, W):
    """verts [V,3] fp32, cam (sx, sy, tx, ty) fp32 -> qx, qy int64 [V], z fp32 [V], ok bool [V]."""
    v = _np(verts, np.float32)
    sx, sy, tx, ty = (np.float32(c) for c in _np(cam, np.float32))
    X, Y, Z = v[:, 0], v[:, 1], v[:, 2]
    with np.errstate(all="ignore"):
        u = ((sx * (X + tx)) + np.float32(1)) * np.float32(0.5 * W)
        w = ((sy * (Y + ty)) + np.float32(1)) * np.float32(0.5 * H)
        ok = np.isfinite(X) & np.isfinite(Y) & np.isfinite(Z) & (np.abs(u) <= GUARD) & (np.abs(w) <= GUARD)
        qx = np.where(ok, np.rint(u * np.float32(256)), 0).astype(np.int64)
        qy = np.where(ok, np.rint(w * np.float32(256)), 0).astype(np.int64)
    return qx, qy, Z, ok


def _unit(n):
    """[...,3] float64 -> n / |n| where |n| is finite and > 0, else 0."""
    with np.errstate(all="ignore"):
        ln = np.sqrt((n[..., 0] * n[..., 0] + n[..., 1] * n[..., 1]) + n[..., 2] * n[..., 2])
        good = (ln > 0) & (ln <= np.finfo(np.float64).max)
        return np.where(good[..., None], n / np.where(good, ln, 1.0)[..., None], 0.0)


def vertex_normals(verts, faces, vf_offsets, vf_faces):
    """verts [V,3] fp32 -> [V,3] float64: the adjacent unit face normals summed in CSR order, normalised."""
    p = _np(verts, np.float32).astype(np.float64)
    f = _np(faces, np.int64)
    with np.errstate(all="ignore"):
        e1 = p[f[:, 1]] - p[f[:, 0]]
        e2 = p[f[:, 2]] - p[f[:, 0]]
        fn = np.stack([e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1],
                       e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2],
                       e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]], 1)
    fn = _unit(fn)
    off, ids = _np(vf_offsets, np.int64), _np(vf_faces, np.int64)
    deg = off[1:] - off[:-1]
    s = np.zeros((len(deg), 3))
    for j in range(int(deg.max(initial=0))):
        m = deg > j
        s[m] = s[m] + fn[ids[off[:-1][m] + j]]
    return _unit(s)


def _setup(qx, qy, z, ok, f):
    """faces f [m,3] of one person -> (keep, x [m,3], y [m,3], z [m,3], ids [m,3], area [m]) oriented to positive area."""
    keep = ok[f].all(1)
    x, y, zz, ids = qx[f].copy(), qy[f].copy(), z[f].copy(), f.copy()
    area = (x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (y[:, 1] - y[:, 0]) * (x[:, 2] - x[:, 0])
    keep &= area != 0
    neg = area < 0
    for a in (x, y, zz, ids):
        a[neg, 1], a[neg, 2] = a[neg, 2].copy(), a[neg, 1].copy()
    return keep, x, y, zz, ids, np.abs(area)


def _edge(ax, ay, bx, by, px, py):
    return (bx - ax) * (py - ay) - (by - ay) * (px - ax)


def _bias(ax, ay, bx, by):
    dx, dy = bx - ax, by - ay
    return np.where((dy < 0) | ((dy == 0) & (dx > 0)), 0, 1)


def weights(x, y, px, py):
    """x, y [m,3] oriented triangles, pixel centres px, py [m] (fixed point) -> w [m,3] int64, covered [m] bool."""
    w = np.stack([_edge(x[:, 1], y[:, 1], x[:, 2], y[:, 2], px, py),
                  _edge(x[:, 2], y[:, 2], x[:, 0], y[:, 0], px, py),
                  _edge(x[:, 0], y[:, 0], x[:, 1], y[:, 1], px, py)], 1)
    b = np.stack([_bias(x[:, 1], y[:, 1], x[:, 2], y[:, 2]), _bias(x[:, 2], y[:, 2], x[:, 0], y[:, 0]),
                  _bias(x[:, 0], y[:, 0], x[:, 1], y[:, 1])], 1)
    return w, ((w - b) >= 0).all(1)


def coverage(x, y, H, W):
    """Oriented triangles x, y [m,3] (fixed point, positive area) -> [m,H,W] bool coverage masks (fill-rule tests)."""
    ys, xs = np.meshgrid(np.arange(H) * 256 + 128, np.arange(W) * 256 + 128, indexing="ij")
    out = []
    for t in range(x.shape[0]):
        _, c = weights(np.repeat(x[t:t + 1], H * W, 0), np.repeat(y[t:t + 1], H * W, 0), xs.reshape(-1), ys.reshape(-1))
        out.append(c.reshape(H, W))
    return np.stack(out) if out else np.zeros((0, H, W), bool)


def _depth_bits(z):
    u = z.astype(np.float32).view(np.uint32).astype(np.uint64)
    return np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000)


def render(frame, verts, orig_cam, colors, faces, vf_offsets, vf_faces, chunk=1 << 22):
    """frame uint8 [H,W,3], verts [n,V,3] fp32, orig_cam [n,4] fp32, colors [n,3] fp32 -> uint8 [H,W,3]."""
    frame = _np(frame, np.uint8)
    H, W = frame.shape[:2]
    verts, cams, colors = _np(verts, np.float32), _np(orig_cam, np.float32), _np(colors, np.float32)
    f_all = _np(faces, np.int64)
    n = verts.shape[0]
    keys = np.full(H * W, EMPTY, np.uint64)
    projs = [project(verts[p], cams[p], H, W) for p in range(n)]
    for p in range(n):
        qx, qy, z, ok = projs[p]
        keep, x, y, zz, _, area = _setup(qx, qy, z, ok, f_all)
        bx0 = np.maximum(-((-(x.min(1) - 128)) >> 8), 0)
        bx1 = np.minimum((x.max(1) - 128) >> 8, W - 1)
        by0 = np.maximum(-((-(y.min(1) - 128)) >> 8), 0)
        by1 = np.minimum((y.max(1) - 128) >> 8, H - 1)
        keep &= (bx0 <= bx1) & (by0 <= by1)
        fid = np.nonzero(keep)[0]
        bw = (bx1 - bx0 + 1)[fid]
        cnt = bw * (by1 - by0 + 1)[fid]
        base = np.uint64(n - 1 - p) << np.uint64(48)
        start = 0
        while start < len(fid):                   # chunks of faces with at most `chunk` box pixels (at least one face)
            csum = np.cumsum(cnt[start:])
            stop = start + max(1, int(np.searchsorted(csum, chunk, side="right")))
            sl = slice(start, stop)
            c = cnt[sl]
            t = np.repeat(np.arange(stop - start), c)
            local = np.arange(int(c.sum())) - np.repeat(np.cumsum(c) - c, c)
            ff = fid[sl][t]
            py_ = by0[ff] + local // bw[sl][t]
            px_ = bx0[ff] + local % bw[sl][t]
            w, cov = weights(x[ff], y[ff], px_ * 256 + 128, py_ * 256 + 128)
            w, ff, px_, py_ = w[cov], ff[cov], px_[cov], py_[cov]
            zf = zz[ff].astype(np.float64)
            s = (w[:, 0].astype(np.float64) * zf[:, 0] + w[:, 1].astype(np.float64) * zf[:, 1]) + \
                w[:, 2].astype(np.float64) * zf[:, 2]
            with np.errstate(over="ignore"):
                d = (s * (1.0 / area[ff].astype(np.float64))).astype(np.float32)
            key = base | (_depth_bits(d) << np.uint64(16)) | ff.astype(np.uint64)
            np.minimum.at(keys, py_ * W + px_, key)
            start = stop
    out = frame.reshape(-1, 3).copy()
    hit = np.nonzero(keys != EMPTY)[0]
    if len(hit):
        k = keys[hit]
        p = (n - 1 - (k >> np.uint64(48)).astype(np.int64))
        f = (k & np.uint64(0xFFFF)).astype(np.int64)
        normals = np.zeros((n, verts.shape[1], 3))
        for q in np.unique(p):
            normals[q] = vertex_normals(verts[q], f_all, vf_offsets, vf_faces)
        qx = np.stack([pr[0] for pr in projs])
        qy = np.stack([pr[1] for pr in projs])
        ids0 = f_all[f]
        x, y = qx[p[:, None], ids0], qy[p[:, None], ids0]
        area = (x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (y[:, 1] - y[:, 0]) * (x[:, 2] - x[:, 0])
        neg = area < 0
        ids = ids0.copy()
        for a in (x, y, ids):
            a[neg, 1], a[neg, 2] = a[neg, 2].copy(), a[neg, 1].copy()
        py_, px_ = hit // W, hit % W
        w, _ = weights(x, y, px_ * 256 + 128, py_ * 256 + 128)
        N = normals[p[:, None], ids]                                    # [m,3 vertices,3]
        wd = w.astype(np.float64)
        nn = (wd[:, 0, None] * N[:, 0] + wd[:, 1, None] * N[:, 1]) + wd[:, 2, None] * N[:, 2]
        nz = _unit(nn)[:, 2]
        shade = 0.3 + 0.7 * np.abs(nz)
        v = (colors[p].astype(np.float64) * shade[:, None]) * 255.0
        out[hit] = np.rint(np.fmin(np.fmax(v, 0.0), 255.0)).astype(np.uint8)
    return out.reshape(H, W, 3)


def uv_sphere(rings=84, segments=82):
    """A closed UV sphere of radius 1: 2 poles + rings x segments vertices (84 x 82 + 2 = 6890, SMPL's count) and
    2 * segments * rings faces (13776, SMPL's count), consistently wound."""
    th = np.pi * np.arange(1, rings + 1) / (rings + 1)
    ph = 2 * np.pi * np.arange(segments) / segments
    ring = np.stack([np.sin(th)[:, None] * np.cos(ph), np.sin(th)[:, None] * np.sin(ph),
                     np.repeat(np.cos(th)[:, None], segments, 1)], -1).reshape(-1, 3)
    verts = np.concatenate([[[0, 0, 1]], ring, [[0, 0, -1]]]).astype(np.float32)
    idx = 1 + np.arange(rings * segments).reshape(rings, segments)
    nxt = np.roll(idx, -1, 1)
    south = 1 + rings * segments
    faces = [np.stack([np.zeros(segments, int), idx[0], nxt[0]], 1)]
    a, b, c, d = idx[:-1], nxt[:-1], idx[1:], nxt[1:]
    faces += [np.stack([a, c, b], -1).reshape(-1, 3), np.stack([b, c, d], -1).reshape(-1, 3)]
    faces.append(np.stack([np.full(segments, south), nxt[-1], idx[-1]], 1))
    return verts, np.concatenate(faces).astype(np.int64)
