"""Multi-GPU behind the reference interface (tb200_create_multi, what CreateGpuWavefrontRenderer builds
for TINSEL_GPUS=N; SURVEY.md 8e): owner-computes row slabs, every device delivers its own rows to the
host, no reduction.  The slab machinery is tested on ONE GPU too (slab renderers side by side, and a
group whose members share the device), so the driver's single-GPU box exercises all of the host code;
the tests that need distinct devices skip there."""
import os

import numpy as np
import pytest

import tinsel_b200 as tb
from tinsel_b200 import abi, sharding
import refdrv
import genscenes

pytestmark = pytest.mark.gpu


def _gpus():
    import torch
    return torch.cuda.device_count()


def _scene(name, size):
    if not os.path.exists(genscenes.path(name)):
        pytest.skip("snapshot scenes/%s.tsnap not present" % name)
    os.environ["TINSEL_B200_PIPELINE"] = "wavefront"
    snap = tb.Snapshot(genscenes.path(name))
    cam, opt = snap.camera, snap.options
    opt.width, opt.height = size
    return snap, cam, opt


def _single(snap, cam, opt, spp):
    r = tb.Renderer(snap.scene)
    r.Init(opt.width, opt.height)
    out = np.zeros((opt.height, opt.width, 4), np.float32)
    for _ in range(spp):
        r.Render(cam, opt, out)
    r.close()
    return out


@pytest.mark.parametrize("name,size,parts", [("cornell", (200, 150), 3), ("veach", (160, 90), 2), ("cornell", (64, 9), 4),
                                             ("ajax", (96, 96), 3), ("bigmesh", (96, 96), 3)])
def test_row_slabs_compose_the_image_on_one_device(name, size, parts):
    """tb200_set_slab: `parts` renderers, each owning one slab, all Render() into the SAME host buffer;
    every row is written by its owner only, and the composed image is the unsharded one (same
    contributions per pixel -- halo samples are bit-identical duplicates -- in another summation order)."""
    snap, cam, opt = _scene(name, size)
    spp = 3
    full = _single(snap, cam, opt, spp)
    out = np.full((opt.height, opt.width, 4), -7.0, np.float32)
    samples = 0
    for k in range(parts):
        row0, rows = sharding.slab_rows(opt.height, k, parts)
        r = tb.Renderer(snap.scene)
        r.Init(opt.width, opt.height)
        r.set_slab(row0, rows)
        before = out.copy()
        for _ in range(spp):
            r.Render(cam, opt, out)
        # rows outside the slab are untouched by this renderer
        mask = np.ones(opt.height, bool)
        mask[row0:row0 + rows] = False
        assert np.array_equal(out[mask], before[mask])
        samples += r.stats().samples
        r.close()
    assert samples == spp * opt.width * opt.height
    assert np.allclose(out, full, rtol=2e-6, atol=1e-6), float(np.abs(out - full).max())
    snap.close()


def _check_group(devices, name="cornell", size=(256, 192)):
    snap, cam, opt = _scene(name, size)
    spp = 4
    full = _single(snap, cam, opt, spp)
    m = tb.Renderer(snap.scene, devices=devices)
    assert m.num_devices() == len(devices)
    m.Init(opt.width, opt.height)
    out = np.full((opt.height, opt.width, 4), -1.0, np.float32)
    m.pin_output(out)
    for _ in range(spp):
        m.Render(cam, opt, out)
    assert np.allclose(out, full, rtol=2e-6, atol=1e-6), float(np.abs(out - full).max())
    assert m.stats().samples == spp * opt.width * opt.height and m.stats().frames == spp
    # the accumulators stay distributed; read_accumulator gathers the owned rows, bit for bit what Render delivered
    assert np.array_equal(m.read_accumulator().view(np.uint32), out.view(np.uint32))
    # finish step: slabs gathered onto the head device first
    f, b = m.finish(1.0, 1.5)
    fo = refdrv.port_finish(out, 1.0)
    assert ((f.view(np.uint32) == fo.view(np.uint32)) | (np.isnan(f) & np.isnan(fo))).all()
    # batch call and one more frame on top
    m.render_n(cam, opt, 2, out)
    ref2 = _single(snap, cam, opt, spp + 2)
    assert np.allclose(out, ref2, rtol=2e-6, atol=1e-6)
    # eNormals: every pixel from its own primary ray -> identical bits whoever renders the row
    opt.mode = abi.MODE_NORMALS
    nm = np.zeros_like(out)
    m.Render(cam, opt, nm)
    r1 = tb.Renderer(snap.scene)
    r1.Init(opt.width, opt.height)
    n1 = np.zeros_like(out)
    r1.Render(cam, opt, n1)
    assert np.array_equal(nm.view(np.uint32), n1.view(np.uint32))
    opt.mode = abi.MODE_PATHTRACE
    # per-sample probe still covers the whole frame, and single-device-only calls are refused
    rad, ras = m.trace_frame(cam, opt, 1)
    rad1, ras1 = r1.trace_frame(cam, opt, 1)
    assert np.array_equal(rad.view(np.uint32), rad1.view(np.uint32)) and np.array_equal(ras, ras1)
    with pytest.raises(tb.TinselB200Error):
        m.set_shard(0, 2)
    # destroying the group must not touch the caller's buffer (a worker thread once re-ran its last job on the
    # way out and rendered one more frame into it)
    m.Render(cam, opt, out)
    before = out.copy()
    m.unpin_output()
    m.close()
    assert np.array_equal(out.view(np.uint32), before.view(np.uint32))
    r1.close()
    snap.close()


def test_group_of_renderers_sharing_one_device():
    """The whole multi-device host path (worker threads, slabs, per-member streamed read-back, gather)
    on a one-GPU box: a group whose three members all sit on device 0 (test hook)."""
    os.environ["TINSEL_B200_TEST_DUP_DEVICES"] = "1"
    try:
        _check_group([0, 0, 0])
        _check_group([0, 0], name="veach", size=(200, 110))
    finally:
        del os.environ["TINSEL_B200_TEST_DUP_DEVICES"]


def test_multi_device_renderer_equals_single_device():
    n = _gpus()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    _check_group(list(range(min(n, 8))))
    _check_group([1, 0], name="ajax", size=(160, 160))   # head on device 1: per-device kernel configuration


def test_second_device_alone():
    """A renderer on a device other than 0 (the shared-memory opt-in of the wavefront kernel is per device)."""
    if _gpus() < 2:
        pytest.skip("needs at least 2 GPUs")
    snap, cam, opt = _scene("cornell", (128, 96))
    a = _single(snap, cam, opt, 2)
    r = tb.Renderer(snap.scene, device=1)
    r.Init(opt.width, opt.height)
    out = np.zeros_like(a)
    for _ in range(2):
        r.Render(cam, opt, out)
    assert np.allclose(out, a, rtol=2e-6, atol=1e-6)
    r.close()
    snap.close()


def test_pinned_and_unpinned_outputs_and_caller_streams():
    import torch
    snap, cam, opt = _scene("cornell", (160, 120))
    r = tb.Renderer(snap.scene)
    r.Init(opt.width, opt.height)
    a = np.zeros((opt.height, opt.width, 4), np.float32)
    b = np.zeros_like(a)
    r.Render(cam, opt, a)            # pageable buffer: the driver's staged copy
    r.Render(cam, opt, a)            # the same pointer again is NOT pinned behind the caller's back
    r.pin_output(b)
    r.pin_output(b)                  # idempotent
    r.Render(cam, opt, b)
    dev = r.read_accumulator()
    assert np.array_equal(b.view(np.uint32), dev.view(np.uint32))
    r.unpin_output()
    r.unpin_output()
    del b                            # freeing after unpin is the contract
    # caller streams, including CUDA's legacy default stream (handle 0)
    for handle in (0, torch.cuda.Stream().cuda_stream):
        r.set_stream(handle)
        r.render_device(cam, opt, 1)
    r.set_stream(None)
    out = r.read_accumulator()
    full = _single(snap, cam, opt, 5)
    assert np.allclose(out, full, rtol=2e-6, atol=1e-6)
    r.close()
    snap.close()


def test_normals_and_trace_frame_respect_shards():
    """eNormals under tb200_set_shard writes only the shard's tile rows (summing the shards gives the image
    once), and tb200_trace_frame returns zeros -- not stale scratch -- for pixels of other shards."""
    snap, cam, opt = _scene("cornell", (96, 70))
    r = tb.Renderer(snap.scene)
    r.Init(opt.width, opt.height)
    opt.mode = abi.MODE_NORMALS
    whole = np.zeros((opt.height, opt.width, 4), np.float32)
    r.Render(cam, opt, whole)
    opt.mode = abi.MODE_PATHTRACE
    rad_all, _ = r.trace_frame(cam, opt, 0)
    total = np.zeros_like(whole)
    for shard in range(3):
        rs = tb.Renderer(snap.scene)
        rs.Init(opt.width, opt.height)
        rs.set_shard(shard, 3)
        opt.mode = abi.MODE_NORMALS
        part = np.zeros_like(whole)
        rs.Render(cam, opt, part)
        opt.mode = abi.MODE_PATHTRACE
        rows = sharding.shard_rows(opt.height, shard, 3)
        other = sorted(set(range(opt.height)) - set(rows))
        assert not part[other].any()
        total += part
        rad, ras = rs.trace_frame(cam, opt, 0)
        assert not rad[other].any() and not ras[other].any()
        assert np.array_equal(rad[rows].view(np.uint32), rad_all[rows].view(np.uint32))
        rs.close()
    assert np.array_equal(total.view(np.uint32), whole.view(np.uint32))
    r.close()
    snap.close()
