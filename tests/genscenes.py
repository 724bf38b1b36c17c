"""Scenes generated from a seed, for the tests that need scale the committed snapshots do not have: a
large displaced mesh ("bigmesh"), a large HDR probe with a small, very bright sun ("bigenv") and a few
meshes instanced many times under glass and metal ("instances").  They stand in for tinsel's ajax, env
and table scenes, whose snapshots are converted from tinsel's scene data and are not in the repository.

`path(name)` returns scenes/<name>.tsnap for a committed scene and, for a generated one, a snapshot
written on first use into a temporary directory that is removed at exit.  Everything is built on the
CPU: mesh BVHs are balanced trees over Morton-ordered triangles (any valid BVH gives the CUDA path and
the CPU restatement the same walk), the scene BVH is fuzzscene's median split."""
import atexit
import ctypes as C
import os
import shutil
import tempfile

import numpy as np

import tinsel_b200 as tb
from tinsel_b200 import abi
import fuzzscene

LEAF = fuzzscene.LEAF
_dir = None
_keep = []


def _morton_bvh(lo, hi):
    """Balanced binary BVH over items with bounds lo/hi (n,3), split at the middle of the Morton order.
    Returns a (BvhNode array, node count); node 0 is the root, leaves hold one item."""
    n = lo.shape[0]
    c = (lo + hi) * 0.5
    cmin, cmax = c.min(0), c.max(0)
    q = ((c - cmin) / np.maximum(cmax - cmin, 1e-12) * 1023.0).astype(np.uint64)
    code = np.zeros(n, np.uint64)
    for b in range(10):
        for a in range(3):
            code |= ((q[:, a] >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b + a)
    order = np.argsort(code, kind="stable")
    slo = np.vstack([lo[order], np.full((1, 3), np.inf, np.float32)])
    shi = np.vstack([hi[order], np.full((1, 3), -np.inf, np.float32)])
    nodes = (abi.BvhNode * (2 * n - 1))()
    start, end, ids = np.array([0]), np.array([n]), np.array([0])
    count = 1
    while start.size:
        pairs = np.stack([start, end], 1).ravel()
        blo = np.minimum.reduceat(slo, pairs, axis=0)[::2]
        bhi = np.maximum.reduceat(shi, pairs, axis=0)[::2]
        leaf = end - start == 1
        inner = ~leaf
        k = int(inner.sum())
        left = count + 2 * np.arange(k)
        mid = (start[inner] + end[inner]) // 2
        lefts = np.zeros(start.size, np.int64)
        rights = np.zeros(start.size, np.int64)
        lefts[inner], rights[inner] = left, left + 1
        lefts[leaf], rights[leaf] = order[start[leaf]], LEAF
        for i, node in enumerate(ids):
            nd = nodes[int(node)]
            nd.lower[:] = [float(x) for x in blo[i]]
            nd.upper[:] = [float(x) for x in bhi[i]]
            nd.left, nd.right_leaf = int(lefts[i]), int(rights[i])
        count += 2 * k
        start = np.stack([start[inner], mid], 1).ravel()
        end = np.stack([mid, end[inner]], 1).ravel()
        ids = np.stack([left, left + 1], 1).ravel()
    return nodes, count


def _grid_mesh(nu, nv, surface):
    """Triangulated (u, v) grid; surface(u, v) -> (nu*nv, 3) positions.  Smooth vertex normals."""
    u, v = np.meshgrid(np.linspace(0.0, 1.0, nu), np.linspace(0.0, 1.0, nv), indexing="xy")
    pos = surface(u.ravel(), v.ravel()).astype(np.float32)
    i = np.arange(nv - 1)[:, None] * nu + np.arange(nu - 1)[None, :]
    i = i.ravel()
    tri = np.concatenate([np.stack([i, i + nu, i + 1], 1), np.stack([i + 1, i + nu, i + nu + 1], 1)]).astype(np.int32)
    return pos, tri


def _mesh(pos, tri):
    """A tb200 mesh (arrays kept alive in _keep) with vertex normals, area CDF and BVH."""
    p0, p1, p2 = pos[tri[:, 0]], pos[tri[:, 1]], pos[tri[:, 2]]
    fn = np.cross(p1 - p0, p2 - p0)
    area = 0.5 * np.linalg.norm(fn, axis=1)
    nrm = np.zeros_like(pos)
    for k in range(3):
        np.add.at(nrm, tri[:, k], fn)
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-20)
    nrm = nrm.astype(np.float32)
    cdf = (np.cumsum(area, dtype=np.float64) / max(float(area.sum()), 1e-20)).astype(np.float32)
    nodes, count = _morton_bvh(np.minimum(np.minimum(p0, p1), p2), np.maximum(np.maximum(p0, p1), p2))
    pos, tri = np.ascontiguousarray(pos), np.ascontiguousarray(tri.ravel())
    _keep.extend([pos, nrm, tri, cdf, nodes])
    m = abi.Mesh()
    m.positions = pos.ctypes.data_as(C.POINTER(C.c_float))
    m.normals = nrm.ctypes.data_as(C.POINTER(C.c_float))
    m.indices = tri.ctypes.data_as(C.POINTER(C.c_int32))
    m.nodes = C.cast(nodes, C.POINTER(abi.BvhNode))
    m.cdf = cdf.ctypes.data_as(C.POINTER(C.c_float))
    m.numVertices, m.numIndices, m.numNodes = pos.shape[0], tri.size, count
    m.area = float(area.sum())
    return m, pos.reshape(-1, 3)


def _blob(nu, nv, radius, bumps, seed):
    rng = np.random.RandomState(seed)
    f = rng.randint(3, 9, size=(4, 2))
    a = rng.uniform(0.03, 0.1, 4) * bumps

    def surface(u, v):
        th, ph = v * np.pi, u * 2.0 * np.pi
        r = radius * (1.0 + sum(a[k] * np.sin(f[k, 0] * th + k) * np.cos(f[k, 1] * ph + 2 * k) for k in range(4)))
        return np.stack([r * np.sin(th) * np.cos(ph), r * np.cos(th), r * np.sin(th) * np.sin(ph)], 1)
    return _grid_mesh(nu, nv, surface)


def _box():
    c = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], np.float32) * 0.5
    q = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    tri = np.array([t for a, b, c2, d in q for t in ((a, b, c2), (a, c2, d))], np.int32)
    return c, tri


def _prism():
    ang = np.array([0.0, 2.0 * np.pi / 3.0, 4.0 * np.pi / 3.0])
    ring = np.stack([0.5 * np.cos(ang), np.zeros(3), 0.5 * np.sin(ang)], 1)
    pos = np.vstack([ring + [0.0, -0.5, 0.0], ring + [0.0, 0.5, 0.0]]).astype(np.float32)
    tri = np.array([(0, 2, 1), (3, 4, 5), (0, 1, 4), (0, 4, 3), (1, 2, 5), (1, 5, 4), (2, 0, 3), (2, 3, 5)], np.int32)
    return pos, tri


def _xf(t, p, q=(0.0, 0.0, 0.0, 1.0), s=1.0):
    t.p[:] = [float(x) for x in p]
    t.r[:] = [float(x) for x in q]
    t.s = float(s)


def _write(path, prims, bounds, meshes, sky, cam_pos, fov, maxdepth=4, clamp=None):
    tree = fuzzscene._build_bvh(bounds)
    nodes = (abi.BvhNode * len(tree))()
    for i, (lo, hi, left, right) in enumerate(tree):
        nodes[i].lower[:] = [float(x) for x in lo]
        nodes[i].upper[:] = [float(x) for x in hi]
        nodes[i].left, nodes[i].right_leaf = int(left), int(right)
    arr = (abi.Primitive * len(prims))(*prims)
    marr = (abi.Mesh * max(len(meshes), 1))(*meshes)
    scene = abi.Scene()
    scene.primitives, scene.numPrimitives = C.cast(arr, C.POINTER(abi.Primitive)), len(prims)
    scene.meshes, scene.numMeshes = C.cast(marr, C.POINTER(abi.Mesh)), len(meshes)
    scene.bvhNodes, scene.numBvhNodes = C.cast(nodes, C.POINTER(abi.BvhNode)), len(tree)
    scene.sky = sky
    base = tb.Snapshot(tb.scene_path("cornell"))
    cam, opt = abi.copy_struct(base.camera), abi.copy_struct(base.options)
    base.close()
    cam.position[:] = [float(x) for x in cam_pos]
    cam.rotation[:] = [0.0, 0.0, 0.0, 1.0]
    cam.fov = float(np.radians(fov))
    cam.shutterStart, cam.shutterEnd = 0.0, 1.0
    opt.width, opt.height, opt.maxDepth = 256, 256, maxdepth
    if clamp is not None:
        opt.clamp = clamp
    if tb.load_library().tb200_snapshot_save(path.encode(), C.byref(scene), C.byref(cam), C.byref(opt)) != 0:
        raise RuntimeError(tb.last_error())


def _plane(eq, color):
    p = abi.Primitive()
    p.type, p.mesh = abi.PLANE, -1
    p.plane[:] = [float(x) for x in eq]
    _xf(p.start, (0, 0, 0))
    _xf(p.end, (0, 0, 0))
    p.material = abi.Material.default()
    p.material.color[:] = list(color)
    return p, (np.full(3, -1.0e8, np.float32), np.full(3, 1.0e8, np.float32))


def _sphere(pos, radius, material, light_samples=0):
    p = abi.Primitive()
    p.type, p.mesh, p.radius = abi.SPHERE, -1, float(radius)
    _xf(p.start, pos)
    _xf(p.end, pos)
    p.material, p.lightSamples = material, light_samples
    r = np.float32(radius * 1.001 + 1e-4)
    return p, (np.asarray(pos, np.float32) - r, np.asarray(pos, np.float32) + r)


def _instance(mesh_index, verts, pos, q, s, material):
    p = abi.Primitive()
    p.type, p.mesh = abi.MESH, mesh_index
    _xf(p.start, pos, q, s)
    _xf(p.end, pos, q, s)
    p.material = material
    # bounds of the transformed vertices (rotation by the unit quaternion q, then scale and offset)
    x, y, z, w = q
    rot = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                    [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                    [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    v = verts @ rot.T * s + np.asarray(pos)
    pad = 1e-3 * (1.0 + np.abs(v).max())
    return p, ((v.min(0) - pad).astype(np.float32), (v.max(0) + pad).astype(np.float32))


def _mat(color, **kw):
    m = abi.Material.default()
    m.color[:] = list(color)
    for k, val in kw.items():
        if isinstance(val, (list, tuple)):
            getattr(m, k)[:] = list(val)
        else:
            setattr(m, k, val)
    return m


def _gradient_sky():
    sky = abi.Sky()
    sky.horizon[:] = [0.35, 0.4, 0.5]
    sky.zenith[:] = [0.1, 0.15, 0.35]
    return sky


def make_bigmesh(path):
    """82k-triangle displaced blob (ajax's role: a mesh far larger than the flat scene program takes,
    walked by the inline and the offloaded mesh walk) on a floor, one sphere light, gradient sky."""
    pos, tri = _blob(257, 161, 1.0, 1.0, seed=1)
    mesh, verts = _mesh(pos, tri)
    floor, fb = _plane((0.0, 1.0, 0.0, 1.05), (0.6, 0.6, 0.55))
    blob, bb = _instance(0, verts, (0.0, 0.0, 0.0), (0.0, 0.0, 0.0, 1.0), 1.0, _mat((0.7, 0.5, 0.3), roughness=0.35, specular=0.5))
    light, lb = _sphere((1.5, 3.0, 2.0), 0.4, _mat((0.0, 0.0, 0.0), emission=[30.0, 28.0, 24.0], specular=0.0), 1)
    _write(path, [floor, blob, light], [fb, bb, lb], [mesh], _gradient_sky(), (0.0, 0.3, 4.2), 40.0)


def make_bigenv(path):
    """Lit only by a 1024x512 HDR probe with a small sun of radiance 4000 (env's role: probe importance
    sampling over a large, very uneven table) -- metal, glass and diffuse spheres and a blob on a floor."""
    w, h = 1024, 512
    v, u = np.meshgrid((np.arange(h) + 0.5) / h, (np.arange(w) + 0.5) / w, indexing="ij")
    rng = np.random.RandomState(7)
    sky = np.stack([0.25 + 0.6 * (1.0 - v), 0.3 + 0.5 * (1.0 - v), 0.45 + 0.4 * (1.0 - v)], -1)
    sky *= 1.0 + 0.3 * np.sin(u * 40.0)[..., None] * np.sin(v * 25.0)[..., None]
    sky[v > 0.5] *= 0.2
    sun = ((u - 0.3) ** 2 * 4.0 + (v - 0.22) ** 2) < 0.012 ** 2
    sky[sun] = [4000.0, 3600.0, 3000.0]
    sky += rng.uniform(0.0, 0.02, sky.shape)
    data = np.zeros((h * w + 1, 4), np.float32)
    data[:-1, :3] = sky.reshape(-1, 3)
    _keep.append(data)
    s = _gradient_sky()
    s.probeValid, s.probeWidth, s.probeHeight = 1, w, h
    s.probeData = data.ctypes.data_as(C.POINTER(C.c_float))
    pos, tri = _blob(97, 65, 0.5, 1.5, seed=2)
    mesh, verts = _mesh(pos, tri)
    floor, fb = _plane((0.0, 1.0, 0.0, 0.6), (0.5, 0.5, 0.5))
    prims = [floor,
             _sphere((-1.2, 0.0, 0.0), 0.6, _mat((0.95, 0.8, 0.6), metallic=1.0, roughness=0.15)),
             _sphere((0.0, -0.1, 0.8), 0.5, _mat((1.0, 1.0, 1.0), transmission=1.0, eta=1.5, roughness=0.02)),
             _instance(0, verts, (1.2, 0.0, -0.2), (0.0, 0.0, 0.0, 1.0), 1.0, _mat((0.3, 0.6, 0.3), roughness=0.6))]
    bounds = [fb] + [b for _, b in prims[1:]]
    prims = [floor] + [p for p, _ in prims[1:]]
    _write(path, prims, bounds, [mesh], s, (0.0, 0.4, 4.5), 45.0, maxdepth=5)


def make_instances(path):
    """Three meshes (box, prism, small blob), 14 instances with rotations and scales, glass, metal and
    diffuse (table's role), a sphere light and a quad-free room of two planes."""
    rng = np.random.RandomState(3)
    shapes = [_box(), _prism(), _blob(17, 13, 0.5, 1.0, seed=4)]
    meshes, verts = [], []
    for p, t in shapes:
        m, v = _mesh(p, t)
        meshes.append(m)
        verts.append(v)
    floor, fb = _plane((0.0, 1.0, 0.0, 0.0), (0.55, 0.5, 0.45))
    wall, wb = _plane((0.0, 0.0, 1.0, 3.0), (0.5, 0.55, 0.6))
    prims, bounds = [floor, wall], [fb, wb]
    mats = [_mat((1.0, 1.0, 1.0), transmission=1.0, eta=1.45, roughness=0.01, absorption=[0.2, 0.05, 0.1]),
            _mat((0.9, 0.9, 0.95), metallic=1.0, roughness=0.08),
            _mat((0.7, 0.3, 0.2), roughness=0.5, clearcoat=1.0, clearcoatGloss=0.8),
            _mat((0.2, 0.4, 0.7), roughness=0.9, sheen=1.0)]
    for k in range(14):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        s = float(rng.uniform(0.35, 0.8))
        pos = (float(rng.uniform(-2.0, 2.0)), s * 0.6, float(rng.uniform(-2.0, 1.0)))
        p, b = _instance(k % 3, verts[k % 3], pos, q, s, mats[k % 4])
        prims.append(p)
        bounds.append(b)
    light, lb = _sphere((0.0, 3.5, 1.0), 0.5, _mat((0.0, 0.0, 0.0), emission=[20.0, 20.0, 20.0], specular=0.0), 2)
    prims.append(light)
    bounds.append(lb)
    _write(path, prims, bounds, meshes, _gradient_sky(), (0.0, 1.4, 5.5), 45.0, maxdepth=6)


GENERATED = {"bigmesh": make_bigmesh, "bigenv": make_bigenv, "instances": make_instances}


def path(name):
    global _dir
    if name not in GENERATED:
        return tb.scene_path(name)
    if _dir is None:
        _dir = tempfile.mkdtemp(prefix="tinsel_b200_scenes_")
        atexit.register(shutil.rmtree, _dir, True)
    p = os.path.join(_dir, name + ".tsnap")
    if not os.path.exists(p):
        GENERATED[name](p)
        del _keep[:]
    return p
