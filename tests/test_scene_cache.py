"""Scene cache (tb200_scene_cache_save / tb200_create_cached, SURVEY.md 8f rank 4): the device layouts of
a scene -- BVH pair records, pre-gathered triangles, primitive records, the probe with its four CDF/PDF
tables -- on disk, loaded straight into device memory.  CPU: the file is written without a GPU, is
deterministic, and damaged files are refused with an error (never a crash).  GPU: a renderer created from
the cache is bit-identical to one created from the loader's scene."""
import os

import numpy as np
import pytest

import tinsel_b200 as tb
import genscenes


def _cache(tmp_path, name):
    if not os.path.exists(genscenes.path(name)):
        pytest.skip("snapshot scenes/%s.tsnap not present" % name)
    snap = tb.Snapshot(genscenes.path(name))
    path = str(tmp_path / (name + ".tcache"))
    tb.scene_cache_save(snap.scene, path)
    return snap, path


def test_cache_is_written_without_a_gpu_and_is_deterministic(tmp_path):
    snap, path = _cache(tmp_path, "glass")
    a = open(path, "rb").read()
    assert a[:8] == b"TB2CACHE" and len(a) > 1280 * (64 + 96)   # pairs + gathered triangles of the 1280-triangle mesh
    path2 = str(tmp_path / "again.tcache")
    tb.scene_cache_save(snap.scene, path2)
    assert open(path2, "rb").read() == a
    snap.close()


def test_probe_tables_are_in_the_cache(tmp_path):
    """envmini's 128x64 probe: data + pdfX + cdfX (n+1 floats each) + pdfY + cdfY (h+1) are stored, so loading needs no BuildCDF."""
    snap, path = _cache(tmp_path, "envmini")
    n = 128 * 64
    assert os.path.getsize(path) >= (n + 1) * 16 + 2 * (n + 1) * 4 + 2 * 65 * 4
    snap.close()


def test_damaged_cache_files_are_refused(tmp_path):
    import torch
    snap, path = _cache(tmp_path, "glass")
    snap.close()
    data = open(path, "rb").read()
    lib = tb.load_library()

    def attempt(blob):
        p = str(tmp_path / "bad.tcache")
        open(p, "wb").write(blob)
        h = lib.tb200_create_cached(p.encode(), 0)
        if h:
            lib.tb200_destroy(h)
        return bool(h), tb.last_error()

    ok, err = attempt(data[: len(data) // 2])
    assert not ok and "truncated" in err
    ok, err = attempt(b"NOTCACHE" + data[8:])
    assert not ok
    stamp = bytearray(data)
    stamp[12] ^= 0xFF                      # sizeof(DPrim) in the layout stamp
    ok, err = attempt(bytes(stamp))
    assert not ok and "another build" in err
    huge = bytearray(data)
    huge[24:32] = (2 ** 62).to_bytes(8, "little")   # first array count far beyond the file
    ok, err = attempt(bytes(huge))
    assert not ok
    assert not attempt(b"")[0]
    ok, err = attempt(data)                # the intact file: fails only for want of a GPU
    if not torch.cuda.is_available():
        assert not ok and "no CUDA device" in err


@pytest.mark.gpu
@pytest.mark.parametrize("name,size", [("glass", (128, 128)), ("envmini", (128, 96)), ("ajax", (160, 160)), ("veach", (192, 108)),
                                       ("env", (256, 256)), ("bigmesh", (160, 160)), ("bigenv", (256, 256))])
def test_renderer_from_cache_is_bit_identical(tmp_path, name, size):
    snap, path = _cache(tmp_path, name)
    os.environ["TINSEL_B200_PIPELINE"] = "wavefront"
    cam, opt = snap.camera, snap.options
    opt.width, opt.height = size
    a = tb.Renderer(snap.scene)
    b = tb.Renderer(None, cache=path)
    for r in (a, b):
        r.Init(*size)
    for frame in (0, 2):
        ra, sa = a.trace_frame(cam, opt, frame)
        rb, sb = b.trace_frame(cam, opt, frame)
        assert np.array_equal(sa, sb)
        assert np.array_equal(ra.view(np.uint32), rb.view(np.uint32)), "%s frame %d" % (name, frame)
    oa = np.zeros((size[1], size[0], 4), np.float32)
    ob = np.zeros_like(oa)
    for _ in range(2):
        a.Render(cam, opt, oa)
        b.Render(cam, opt, ob)
    assert np.allclose(oa, ob, rtol=2e-6, atol=1e-6)
    assert b.stats().h2dBytes == a.stats().h2dBytes    # the same arrays went to the device
    a.close()
    b.close()
    snap.close()
