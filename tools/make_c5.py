"""BASELINE configs[4]: a generated OBJ of translated (and uniformly scaled) copies of a reference mesh on an
nx x ny grid that fills the default frustum (eye (0,0,7), dir_z -0.5).  The reference has no instancing or
transforms (MeshShape.cpp:101-110 uses file coordinates), so the copies are baked into the file and go through
the ordinary loader.  Deterministic: no randomness.

    python tools/make_c5.py SRC.obj OUT.obj COPIES [aspect]

`usemtl`/`mtllib` lines are kept; the .mtl and its textures are expected next to OUT.obj (this script symlinks
the source's .mtl and texture directory when they exist)."""
import hashlib
import math
import os
import sys


def cached_name(src, copies, aspect=16.0 / 9.0):
    """File name for the generated OBJ in a cache directory: keyed by the source mesh's and this script's
    contents, the copy count and the aspect, so that a changed input never reuses an old file."""
    h = hashlib.sha256()
    for path in (src, os.path.abspath(__file__)):
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(f"{copies}:{float(aspect)!r}".encode())
    return f"{os.path.splitext(os.path.basename(src))[0]}_x{copies}_{h.hexdigest()[:16]}.obj"


def main(src, out, copies, aspect=16.0 / 9.0):
    v, vt, vn, faces, mtllib = [], [], [], [], None
    with open(src) as f:
        for line in f:
            t = line.split()
            if not t:
                continue
            if t[0] == "v":
                v.append(tuple(float(x) for x in t[1:4]))
            elif t[0] == "vt":
                vt.append(line.rstrip("\n"))
            elif t[0] == "vn":
                vn.append(line.rstrip("\n"))
            elif t[0] in ("f", "usemtl"):
                faces.append(t)
            elif t[0] == "mtllib":
                mtllib = line.rstrip("\n")
    xs, ys, zs = zip(*v)
    cx, cy, cz = (min(xs) + max(xs)) / 2, (min(ys) + max(ys)) / 2, (min(zs) + max(zs)) / 2
    ex, ey = max(xs) - min(xs), max(ys) - min(ys)
    nx = max(1, int(round(math.sqrt(copies * aspect * ey / ex))))
    ny = (copies + nx - 1) // nx
    # frustum at z = 0: |x| <= 3.5 * aspect, |y| <= 3.5 (RayTracerProgram.cpp:141-142,164); use 90 % of it
    cell_w, cell_h = 2 * 3.5 * aspect * 0.9 / nx, 2 * 3.5 * 0.9 / ny
    scale = 0.9 * min(cell_w / ex, cell_h / ey)
    with open(out, "w") as o:
        if mtllib:
            o.write(mtllib + "\n")
        # texcoords / normals are shared by every copy (translation and uniform scale keep them)
        o.write("\n".join(vt) + "\n")
        o.write("\n".join(vn) + "\n")
        done = 0
        for j in range(ny):
            for i in range(nx):
                if done >= copies:
                    break
                ox = (i + 0.5) * cell_w - 3.5 * aspect * 0.9
                oy = (j + 0.5) * cell_h - 3.5 * 0.9
                o.write("".join("v %.6f %.6f %.6f\n" % ((x - cx) * scale + ox, (y - cy) * scale + oy, (z - cz) * scale) for x, y, z in v))
                base = done * len(v)
                lines = []
                for t in faces:
                    if t[0] == "usemtl":
                        lines.append(" ".join(t))
                        continue
                    corners = []
                    for c in t[1:]:
                        a = c.split("/")
                        a[0] = str(int(a[0]) + base)
                        corners.append("/".join(a))
                    lines.append("f " + " ".join(corners))
                o.write("\n".join(lines) + "\n")
                done += 1
    # assets next to the output
    sdir, odir = os.path.dirname(os.path.abspath(src)), os.path.dirname(os.path.abspath(out))
    # the loader opens <obj name>.mtl (MeshShape.cpp:202-210) and resolves map_Kd relative to the OBJ's directory
    stem = os.path.splitext(os.path.basename(src))[0]
    src_mtl = os.path.join(sdir, stem + ".mtl")
    out_mtl = os.path.splitext(os.path.abspath(out))[0] + ".mtl"
    if os.path.exists(src_mtl) and not os.path.exists(out_mtl):
        os.symlink(src_mtl, out_mtl)
    if sdir != odir and os.path.isdir(os.path.join(sdir, stem)) and not os.path.exists(os.path.join(odir, stem)):
        os.symlink(os.path.join(sdir, stem), os.path.join(odir, stem))
    return nx, ny, scale


if __name__ == "__main__":
    nx, ny, scale = main(sys.argv[1], sys.argv[2], int(sys.argv[3]), float(sys.argv[4]) if len(sys.argv) > 4 else 16.0 / 9.0)
    print(f"grid {nx} x {ny}, scale {scale:.5f}")
