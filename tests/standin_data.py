"""Stand-in scene assets, generated: the reference's Data folder is not part of this repository.

The scenes of tests/scenes.py and bench.py name three meshes of the reference's Data folder:
TorusKnot.obj, BlenderMonkey.obj and the textured unitychan.obj (+ unitychan.mtl + PNG textures).
Where that folder is not staged under assets/_ref/Data, `write(dir)` creates meshes of the same names
and formats from closed-form surfaces, so that every test that compares the CUDA path with the host
layer or the plain-C restatement (and bench.py) runs from the repository alone:

    TorusKnot.obj      a (2,3) torus knot tube, quads (the loader's quad split), one material-less mesh
    BlenderMonkey.obj  a lumpy closed blob, triangles
    unitychan.obj      a standing figure of eight parts (head, hair, torso, skirt, arms, legs), 21 760
                       triangles, one `usemtl` per part; unitychan.mtl maps each part to a PNG under
                       unitychan/ (RGB and RGBA, 8 bits, sizes 64..256)

The stand-ins are not the reference's models: tests/test_golden.py replays the fixtures of the reference's
own meshes where the folder is staged, else those of the stand-ins (tests/golden/standin/, written by the
plain-C restatement, not by the reference).  Deterministic: no randomness.

    python tests/standin_data.py OUT_DIR
"""
import os
import struct
import sys
import zlib

import numpy as np

NAMES = ("TorusKnot.obj", "BlenderMonkey.obj", "unitychan.obj", "unitychan.mtl")


def _grid(fn, nu, nv):
    """Vertices, normals and (u, v) of the parametric surface fn(u, v) on an (nu + 1) x (nv + 1) grid."""
    u, v = np.meshgrid(np.linspace(0.0, 1.0, nu + 1), np.linspace(0.0, 1.0, nv + 1), indexing="ij")
    p = fn(u, v)
    e = 1e-4
    du = fn(np.minimum(u + e, 1.0), v) - fn(np.maximum(u - e, 0.0), v)
    dv = fn(u, np.minimum(v + e, 1.0)) - fn(u, np.maximum(v - e, 0.0))
    n = np.cross(du, dv)
    ln = np.linalg.norm(n, axis=-1, keepdims=True)
    # poles of spheres and closed ends: the direction away from the part's centre
    radial = p - p.reshape(-1, 3).mean(0)
    n = np.where(ln > 1e-12, n / np.maximum(ln, 1e-30), radial / np.maximum(np.linalg.norm(radial, axis=-1, keepdims=True), 1e-30))
    uv = np.stack([u, v], -1)
    return p.reshape(-1, 3), n.reshape(-1, 3), uv.reshape(-1, 2)


def _faces(nu, nv, base, quads):
    """1-based corner indices of the grid's cells: one quad or two triangles per cell."""
    out = []
    for i in range(nu):
        for j in range(nv):
            a = base + i * (nv + 1) + j + 1
            b, c, d = a + (nv + 1), a + (nv + 1) + 1, a + 1
            out.append((a, b, c, d) if quads else (a, b, c))
            if not quads:
                out.append((a, c, d))
    return out


def _write_obj(path, parts, mtllib=None):
    """parts: (material name or None, vertices, normals, uvs, faces with 1-based indices into this part)."""
    lines = []
    if mtllib:
        lines.append(f"mtllib {mtllib}")
    base = 0
    body = []
    for mat, p, n, uv, faces in parts:
        lines += ["v %.6f %.6f %.6f" % tuple(x) for x in p]
        lines += ["vt %.6f %.6f" % tuple(x) for x in uv]
        lines += ["vn %.6f %.6f %.6f" % tuple(x) for x in n]
        if mat:
            body.append(f"usemtl {mat}")
        body += ["f " + " ".join(f"{k + base}/{k + base}/{k + base}" for k in f) for f in faces]
        base += len(p)
    with open(path, "w") as f:
        f.write("\n".join(lines + body) + "\n")


def _png(path, px):
    """8-bit RGB (H, W, 3) or RGBA (H, W, 4) PNG; rows alternate filters 0 (none) and 1 (sub)."""
    h, w, ch = px.shape
    raw = bytearray()
    for y in range(h):
        row = px[y].reshape(-1).astype(np.int32)
        if y % 2:
            raw.append(1)
            sub = row.copy()
            sub[ch:] -= row[:-ch]
            raw += (sub & 255).astype(np.uint8).tobytes()
        else:
            raw.append(0)
            raw += row.astype(np.uint8).tobytes()

    def chunk(kind, data):
        return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data) & 0xFFFFFFFF)

    ihdr = struct.pack(">IIBBBBB", w, h, 8, 2 if ch == 3 else 6, 0, 0, 0)
    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", ihdr) + chunk(b"IDAT", zlib.compress(bytes(raw), 9)) + chunk(b"IEND", b""))


def _texture(k, w, h, ch):
    """Part k's texture: stripes, checks and a gradient in a colour of its own (alpha varies where present)."""
    y, x = np.mgrid[0:h, 0:w]
    base = np.array([(230, 190, 170), (120, 70, 40), (240, 240, 250), (40, 50, 110), (230, 190, 170), (30, 30, 40),
                     (200, 40, 60), (250, 220, 120)][k], np.float64)
    check = ((x // (4 + k)) + (y // (6 + k))) % 2
    stripe = 0.5 + 0.5 * np.sin(2 * np.pi * (x * (k + 1) / w + y * 2.0 / h))
    shade = (0.55 + 0.3 * check + 0.15 * stripe)[..., None] * base + (x[..., None] * 37 + y[..., None] * 11 + 13 * k) % 23
    px = np.clip(shade, 0, 255).astype(np.uint8)
    if ch == 4:
        px = np.concatenate([px, (160 + (x + 3 * y) % 96)[..., None].astype(np.uint8)], -1)
    return px


def _torus_knot(u, v):
    t, a = 2 * np.pi * u, 2 * np.pi * v
    p, q, R, r, tube = 2, 3, 1.2, 0.5, 0.32

    def centre(t):
        rr = R + r * np.cos(q * t)
        return np.stack([rr * np.cos(p * t), rr * np.sin(p * t), -r * np.sin(q * t)], -1)

    c = centre(t)
    tan = centre(t + 1e-3) - centre(t - 1e-3)
    tan /= np.linalg.norm(tan, axis=-1, keepdims=True)
    ref = np.broadcast_to(np.array([0.0, 0.0, 1.0]), tan.shape)
    nrm = np.cross(tan, ref)
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    bin_ = np.cross(tan, nrm)
    return c + tube * (np.cos(a)[..., None] * nrm + np.sin(a)[..., None] * bin_)


def _blob(u, v):
    th, ph = np.pi * u, 2 * np.pi * v
    rad = 1.3 + 0.18 * np.sin(3 * th) * np.cos(4 * ph) + 0.1 * np.cos(5 * ph + th)
    return np.stack([rad * np.sin(th) * np.cos(ph) * 1.1, rad * np.cos(th) * 0.9 + 0.2, rad * np.sin(th) * np.sin(ph)], -1)


def _ellipsoid(c, r, th0=0.0, th1=1.0):
    def f(u, v):
        th, ph = np.pi * (th0 + (th1 - th0) * u), 2 * np.pi * v
        return np.stack([c[0] + r[0] * np.sin(th) * np.cos(ph), c[1] + r[1] * np.cos(th), c[2] + r[2] * np.sin(th) * np.sin(ph)], -1)
    return f


def _limb(top, bottom, r0, r1):
    top, bottom = np.array(top, np.float64), np.array(bottom, np.float64)
    axis = bottom - top
    side = np.cross(axis, [0.0, 0.0, 1.0])
    if np.linalg.norm(side) < 1e-9:
        side = np.array([1.0, 0.0, 0.0])
    side /= np.linalg.norm(side)
    front = np.cross(side, axis / np.linalg.norm(axis))

    def f(u, v):
        ph = 2 * np.pi * v
        # rounded ends: the radius closes to 0 over the first and last 8 % of the length
        s = np.clip(u, 0.0, 1.0)
        rad = (r0 + (r1 - r0) * s) * np.sqrt(np.clip(1 - ((np.abs(s - 0.5) - 0.42) / 0.08).clip(0) ** 2, 0, 1))
        return (top + s[..., None] * axis + rad[..., None] * (np.cos(ph)[..., None] * side + np.sin(ph)[..., None] * front))
    return f


def _figure():
    """(name, surface, nu, nv, texture size, channels) of the eight parts; 21 760 triangles in all."""
    return [
        ("face", _ellipsoid((0.0, 1.35, 0.0), (0.42, 0.48, 0.42)), 40, 48, (128, 128), 3),
        ("hair", _ellipsoid((0.0, 1.42, -0.04), (0.47, 0.5, 0.47), 0.0, 0.62), 32, 48, (256, 128), 4),
        ("body", _ellipsoid((0.0, 0.35, 0.0), (0.38, 0.62, 0.26)), 40, 40, (128, 256), 3),
        ("skirt", _limb((0.0, 0.05, 0.0), (0.0, -0.55, 0.0), 0.3, 0.62), 24, 64, (64, 64), 4),
        ("arm_l", _limb((0.45, 0.8, 0.0), (0.95, -0.2, 0.25), 0.11, 0.08), 40, 20, (64, 128), 3),
        ("arm_r", _limb((-0.45, 0.8, 0.0), (-0.9, -0.15, 0.3), 0.11, 0.08), 40, 20, (64, 128), 3),
        ("leg_l", _limb((0.16, -0.3, 0.0), (0.22, -1.98, 0.1), 0.14, 0.1), 56, 24, (128, 64), 3),
        ("leg_r", _limb((-0.16, -0.3, 0.0), (-0.2, -1.98, 0.05), 0.14, 0.1), 56, 24, (128, 64), 4),
    ]


def write(out_dir):
    """Writes the stand-in Data folder into out_dir (created if needed) and returns out_dir."""
    os.makedirs(os.path.join(out_dir, "unitychan"), exist_ok=True)
    p, n, uv = _grid(_torus_knot, 256, 16)
    _write_obj(os.path.join(out_dir, "TorusKnot.obj"), [(None, p, n, uv, _faces(256, 16, 0, True))])
    p, n, uv = _grid(_blob, 24, 48)
    _write_obj(os.path.join(out_dir, "BlenderMonkey.obj"), [(None, p, n, uv, _faces(24, 48, 0, False))])
    parts, mtl = [], []
    for k, (name, fn, nu, nv, (tw, th), ch) in enumerate(_figure()):
        p, n, uv = _grid(fn, nu, nv)
        parts.append((name, p, n, uv, _faces(nu, nv, 0, False)))
        tex = f"unitychan/{name}.png"
        _png(os.path.join(out_dir, tex), _texture(k, tw, th, ch))
        mtl += [f"newmtl {name}", "Kd 1.000000 1.000000 1.000000", f"map_Kd {tex}", ""]
    _write_obj(os.path.join(out_dir, "unitychan.obj"), parts, mtllib="unitychan.mtl")
    with open(os.path.join(out_dir, "unitychan.mtl"), "w") as f:
        f.write("\n".join(mtl))
    return out_dir


if __name__ == "__main__":
    write(sys.argv[1])
