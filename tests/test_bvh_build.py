"""GPU BVH build (tb200_bvh_build, tinsel_b200/csrc/bvh_build.cu; SURVEY.md 8f rank 3).

A different tree is a different -- equally valid -- input to the same traversal, so the criteria are:
  * structure: the reference's node format, root at 0, every triangle in exactly one leaf, every
    interior box the exact union of its children's, leaf boxes = the triangle's bounds (mesh.cpp:320-331);
  * parity: hand the GPU-built tree to the oracle AS the mesh's BVH and compare the CUDA renderer on
    that same tree per sample, bit for bit;
  * quality: node visits per ray (instrumented oracle, reference traversal order) within 10 % of the
    reference's SAH tree; and the build time."""
import ctypes as C
import os
import time

import numpy as np
import pytest

import tinsel_b200 as tb
from tinsel_b200 import abi
import refdrv
import genscenes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPORT = os.path.join(ROOT, "gpurun_out", "bvh_build.txt")


def _mesh_arrays(mesh):
    nv, ni = mesh.numVertices, mesh.numIndices
    pos = np.ctypeslib.as_array(mesh.positions, shape=(nv * 3,)).reshape(nv, 3)
    idx = np.ctypeslib.as_array(mesh.indices, shape=(ni,)).reshape(ni // 3, 3)
    return pos, idx


def _check_structure(nodes, pos, idx):
    ntri = idx.shape[0]
    assert nodes.shape[0] == 2 * ntri - 1
    lo = np.stack([nodes["lower"][:, k] for k in range(3)], 1)
    hi = np.stack([nodes["upper"][:, k] for k in range(3)], 1)
    leaf = (nodes["right_leaf"] >> 31) != 0
    left = nodes["left"].astype(np.int64)
    right = (nodes["right_leaf"] & 0x7FFFFFFF).astype(np.int64)
    assert not leaf[0] or ntri == 1
    # leaves: every triangle exactly once, box = triangle bounds
    tris = left[leaf]
    assert np.array_equal(np.sort(tris), np.arange(ntri))
    tp = pos[idx[tris]]                       # (n, 3 verts, 3)
    assert np.array_equal(lo[leaf], tp.min(1)) and np.array_equal(hi[leaf], tp.max(1))
    # interior: children in range, every node except the root referenced exactly once, box = exact union
    inner = ~leaf
    li, ri = left[inner], right[inner]
    assert (li >= 0).all() and (li < nodes.shape[0]).all() and (ri < nodes.shape[0]).all()
    refs = np.bincount(np.concatenate([li, ri]), minlength=nodes.shape[0])
    assert refs[0] == 0 and (refs[1:] == 1).all()
    assert np.array_equal(lo[inner], np.minimum(lo[li], lo[ri])) and np.array_equal(hi[inner], np.maximum(hi[li], hi[ri]))
    # depth (iterative): the walkers and the reference's own stack[32] want <= 32
    depth = np.zeros(nodes.shape[0], np.int32)
    order = [0]
    maxd = 0
    frontier = np.array([0])
    d = 0
    while frontier.size:
        d += 1
        f = frontier[~leaf[frontier]]
        frontier = np.concatenate([left[f], right[f]]) if f.size else np.array([], np.int64)
    return d


NODE_DTYPE = np.dtype([("lower", np.float32, 3), ("upper", np.float32, 3), ("left", np.uint32), ("right_leaf", np.uint32)])


def _build(mesh):
    pos, idx = _mesh_arrays(mesh)
    nodes = np.zeros(2 * idx.shape[0] - 1, NODE_DTYPE)
    info = tb.bvh_build(pos, idx, nodes)
    return pos, idx, nodes, info


def _scene_with_nodes(snap, mesh_index, nodes):
    """A copy of the snapshot's tb200_scene whose mesh `mesh_index` uses `nodes` as its BVH."""
    base = snap.scene.contents
    sc = abi.Scene()
    C.memmove(C.byref(sc), C.byref(base), C.sizeof(abi.Scene))
    meshes = (abi.Mesh * base.numMeshes)()
    C.memmove(meshes, base.meshes, C.sizeof(meshes))
    meshes[mesh_index].nodes = nodes.ctypes.data_as(C.POINTER(abi.BvhNode))
    meshes[mesh_index].numNodes = nodes.shape[0]
    sc.meshes = C.cast(meshes, C.POINTER(abi.Mesh))
    return sc, meshes


def _biggest_mesh(scene):
    best, tris = -1, 0
    for m in range(scene.numMeshes):
        if scene.meshes[m].numIndices // 3 > tris:
            best, tris = m, scene.meshes[m].numIndices // 3
    return best


@pytest.mark.parametrize("name,size", [("glass", (128, 128)), ("meshlight", (128, 128)), ("table", (160, 100)), ("ajax", (192, 192)),
                                       ("instances", (160, 100)), ("bigmesh", (192, 192))])
def test_gpu_built_bvh_structure_and_parity(name, size):
    if not os.path.exists(genscenes.path(name)):
        pytest.skip("snapshot scenes/%s.tsnap not present" % name)
    os.environ["TINSEL_B200_PIPELINE"] = "wavefront"
    snap = tb.Snapshot(genscenes.path(name))
    cam, opt = snap.camera, snap.options
    opt.width, opt.height = size
    m = _biggest_mesh(snap.scene.contents)
    pos, idx, nodes, info = _build(snap.scene.contents.meshes[m])
    depth = _check_structure(nodes, pos, idx)
    sc, keep = _scene_with_nodes(snap, m, nodes)
    oracle = refdrv.PortScene(C.pointer(sc), cam, opt, keepalive=(snap, keep, nodes))
    oracle.set_size(*size)
    r = tb.Renderer(C.pointer(sc))
    r.Init(*size)
    for frame in (0, 3):
        rad, ras = r.trace_frame(cam, opt, frame)
        orad, oras = oracle.trace_frame(frame, 8)
        assert np.array_equal(ras, oras)
        same = (rad.view(np.uint32) == orad.view(np.uint32)).all(-1) | (np.isnan(rad).any(-1) & np.isnan(orad).any(-1))
        assert bool(same.all()), "%s frame %d: %d samples differ on the GPU-built tree" % (name, frame, int((~same).sum()))
    msg = "%-10s %7d triangles: build %.2f ms on the GPU (%d rounds, %d launches), depth %d" % (
        name, idx.shape[0], info.buildMs, info.rounds, info.kernelLaunches, depth)
    print(msg)
    try:
        os.makedirs(os.path.dirname(REPORT), exist_ok=True)
        with open(REPORT, "a") as f:
            f.write(msg + "\n")
    except OSError:
        pass
    r.close()
    oracle.close()
    snap.close()


def _visits(scene_ptr, cam, opt, size, keep):
    """Interior-node visits and triangle tests per ray on the reference traversal order (instrumented oracle)."""
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "count"])
    lib = C.CDLL(os.path.join(ROOT, "oracle", "libtinsel_oracle_count.so"))
    lib.oracle_create.restype = C.c_void_p
    lib.oracle_create.argtypes = [C.POINTER(abi.Scene)]
    lib.oracle_render_seeded.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.POINTER(abi.Options), C.c_int, C.c_int,
                                         C.POINTER(C.c_float), C.c_int]
    lib.oracle_counters.argtypes = [C.POINTER(C.c_ulonglong), C.c_int]
    lib.oracle_destroy.argtypes = [C.c_void_p]
    h = C.c_void_p(lib.oracle_create(scene_ptr))
    o = abi.copy_struct(opt)
    o.width, o.height = size
    out = np.zeros((size[1], size[0], 4), np.float32)
    buf = (C.c_ulonglong * 16)()
    lib.oracle_counters(buf, 1)
    lib.oracle_render_seeded(h, C.byref(cam), C.byref(o), 0, 1, out.ctypes.data_as(C.POINTER(C.c_float)), 8)
    lib.oracle_counters(buf, 1)
    lib.oracle_destroy(h)
    names = ["V_int", "T_tri", "T_prim", "H_mesh", "H", "B_nee", "B_probe", "B_miss", "P_fb", "rays", "samples"]
    c = dict(zip(names, [int(x) for x in buf[:len(names)]]))
    return c["V_int"] / c["rays"], c["T_tri"] / c["rays"]


def test_gpu_built_bvh_quality_and_build_time():
    """ajax: node visits per ray within 10 % of the reference's SAH tree (bvh.h:30-263), build < 50 ms
    (reference: 1.33 s on one host core, SURVEY 8f)."""
    if not os.path.exists(tb.scene_path("ajax")):
        pytest.skip("snapshot scenes/ajax.tsnap not present")
    snap = tb.Snapshot(tb.scene_path("ajax"))
    cam, opt = snap.camera, snap.options
    m = _biggest_mesh(snap.scene.contents)
    pos, idx, nodes, info = _build(snap.scene.contents.meshes[m])   # first call pays CUDA context + cub set-up
    pos, idx, nodes, info = _build(snap.scene.contents.meshes[m])
    size = (256, 256)
    v_ref, t_ref = _visits(snap.scene, cam, opt, size, None)
    sc, keep = _scene_with_nodes(snap, m, nodes)
    v_gpu, t_gpu = _visits(C.pointer(sc), cam, opt, size, keep)
    msg = "ajax quality: interior visits/ray %.2f (GPU PLOC tree) vs %.2f (reference SAH tree) = %.3f; triangle tests/ray %.2f vs %.2f; build %.2f ms" % (
        v_gpu, v_ref, v_gpu / v_ref, t_gpu, t_ref, info.buildMs)
    print(msg)
    try:
        os.makedirs(os.path.dirname(REPORT), exist_ok=True)
        with open(REPORT, "a") as f:
            f.write(msg + "\n")
    except OSError:
        pass
    assert info.buildMs < 50.0, msg
    assert v_gpu <= 1.10 * v_ref, msg
    snap.close()


def test_bvh_build_rejects_bad_input_and_handles_tiny_meshes():
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.5]], np.float32)
    one = np.array([[0, 1, 2]], np.int32)
    nodes = np.zeros(1, NODE_DTYPE)
    tb.bvh_build(pos, one, nodes)
    assert (nodes["right_leaf"][0] >> 31) == 1 and nodes["left"][0] == 0
    two = np.array([[0, 1, 2], [1, 3, 2]], np.int32)
    nodes = np.zeros(3, NODE_DTYPE)
    tb.bvh_build(pos, two, nodes)
    _check_structure(nodes, pos, two)
    bad = np.array([[0, 1, 9]], np.int32)
    with pytest.raises(tb.TinselB200Error):
        tb.bvh_build(pos, bad, np.zeros(1, NODE_DTYPE))
