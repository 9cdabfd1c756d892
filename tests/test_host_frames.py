"""Host paths of the frame runtime that the parity tests do not reach: arena overflow in the middle of a stream, a blocking
call while streamed frames are in flight, read-back bands with and without CUDA graphs, and a group's host destination
leaving its renderers' own settings alone. Every frame is compared with the same frame from a blocking render."""
import ctypes as C

import numpy as np
import pytest

from vello_b200 import scenes
from vello_b200.config import AA_MSAA16, RenderParams
from vello_b200.encoding import BLACK, resolve

pytestmark = pytest.mark.gpu

P1024 = RenderParams(BLACK, 1024, 1024, AA_MSAA16)
# paths per frame: every scene needs more line / tile arena than its own first guess and than the grown arenas of the one before
GROWING = (300, 1500, 4000, 8000, 14000)


def _paris(n, seed, size=1024):
    return resolve(scenes.paris_like(n, size, seed=seed).encoding)


def _blocking(packed_frames, params):
    """The frames through blocking vb_render on a renderer warmed by each frame once; and the retries of those first calls."""
    from vello_b200.renderer import Renderer
    r = Renderer()
    frames, retries = [], 0
    for pk in packed_frames:
        r.render_to_texture(pk, params)
        retries += int(r.last_stats.retries)
        frames.append(r.render_to_texture(pk, params))
    r.close()
    return frames, retries


@pytest.mark.parametrize("n_frames", [1, 2, 3, 5])
def test_stream_overflow_midstream(n_frames):
    """render_stream on a renderer sized by one tiny frame: with 5 growing scenes the arenas overflow at the rasterisation
    check and the frame is re-run together with the younger frame enqueued behind it; 1-3 frames only go through the
    vb_readback_wait tail. Every frame equals the blocking render."""
    from vello_b200.renderer import Renderer
    seq = [_paris(n, 20 + k) for k, n in enumerate(GROWING[:n_frames])]
    r = Renderer()
    r.render_to_texture(_paris(20, 1, size=64), RenderParams(BLACK, 64, 64, AA_MSAA16))
    got = list(r.render_stream(seq, P1024))
    r.close()
    want, retries = _blocking(seq, P1024)
    if n_frames == 5:
        assert retries > 0, "the growing scenes were meant to overflow the arenas"
    assert len(got) == n_frames
    for k, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), k


def test_blocking_call_drains_streamed_frames():
    """Two frames begun through vb_render_begin, then a blocking vb_render: on its return both streamed host buffers are
    complete and equal the blocking frames."""
    from vello_b200.renderer import Renderer, _Layout, _params_struct, FrameStats
    seq = [_paris(1500, 31), _paris(1500, 32), _paris(1500, 33)]
    want, _ = _blocking(seq, P1024)
    r = Renderer()
    keep, outs = [], []
    for pk in seq[:2]:
        scene = np.ascontiguousarray(pk.scene, dtype=np.uint32)
        ramps = np.ascontiguousarray(pk.ramps, dtype=np.uint32)
        atlas = np.ascontiguousarray(pk.atlas, dtype=np.uint8)
        lay = _Layout(*[int(v) for v in pk.layout.as_array()])
        ps = _params_struct(P1024)
        out = np.zeros((1024, 1024, 4), dtype=np.uint8)
        keep.append((scene, ramps, atlas, lay, ps))
        outs.append(out)
        rc = r.lib.vb_render_begin(r.handle, scene.ctypes.data, scene.nbytes, C.byref(lay), ramps.ctypes.data if ramps.size else None,
                                   512, ramps.shape[0], atlas.ctypes.data, atlas.shape[1], atlas.shape[0], C.byref(ps),
                                   out.ctypes.data, C.byref(FrameStats()))
        r._check(rc, "vb_render_begin")
    last = r.render_to_texture(seq[2], P1024)
    assert np.array_equal(outs[0], want[0])
    assert np.array_equal(outs[1], want[1])
    assert np.array_equal(last, want[2])
    r.close()


def test_readback_bands_and_graphs():
    """A blocking host render of a 64-tile-row frame with 1, 3 and 8 read-back bands, graphs on and off: identical pixels,
    and a kernel_launches count that is the same for every repeated frame of a configuration. Fine is one launch per band.
    The graph path of a banded frame runs one more k_publish_bump than the direct path: the captured part ends with one and
    the banded fine ends with another."""
    from vello_b200.renderer import Renderer
    packed = _paris(3000, 7)
    r = Renderer()
    want = r.render_to_texture(packed, P1024)
    host = {}
    for graph in (False, True):
        r.set_cuda_graph(graph)
        for bands in (1, 3, 8):
            assert r.lib.vb_set_readback_bands(r.handle, bands) == 0
            counts = []
            for _ in range(3):
                assert np.array_equal(r.render_to_texture(packed, P1024), want), (graph, bands)
                counts.append(int(r.last_stats.kernel_launches))
            assert len(set(counts)) == 1, (graph, bands, counts)
            host[graph, bands] = counts[0]
    r.upload(packed)
    dev = {}
    for graph in (False, True):
        r.set_cuda_graph(graph)
        counts = [int(r.render_resident(P1024).kernel_launches) for _ in range(3)]
        assert len(set(counts)) == 1, (graph, counts)
        dev[graph] = counts[0]
        assert np.array_equal(r.download_target(P1024), want)
    r.close()
    assert dev[False] == dev[True]
    assert host[False, 1] == host[True, 1] == dev[False]
    for bands in (3, 8):
        assert host[False, bands] == dev[False] + bands - 1
        assert host[True, bands] == host[False, bands] + 1


def test_group_host_destination_keeps_renderer_settings():
    """After a host-destination vb_group_render, a renderer of the group renders a 64-tile-row host frame like a fresh
    renderer: same pixels and the same kernel_launches (its read-back band setting was not overwritten by the group)."""
    from vello_b200.renderer import Renderer, RendererGroup

    class Borrowed(Renderer):  # a renderer owned by the group: never freed from here
        def __init__(self, lib, handle):
            self.lib, self.handle, self.last_stats, self._keep = lib, C.c_void_p(handle), None, None

        def close(self):
            pass

    g = RendererGroup([0, 0])
    g.render_to_texture(_paris(500, 3, size=512), RenderParams(BLACK, 512, 512, AA_MSAA16))
    packed = _paris(2000, 9)
    sub = Borrowed(g.lib, g.lib.vb_group_renderer(g.handle, 0))
    fresh = Renderer()
    for _ in range(2):
        got = sub.render_to_texture(packed, P1024)
        want = fresh.render_to_texture(packed, P1024)
    assert np.array_equal(got, want)
    assert int(sub.last_stats.kernel_launches) == int(fresh.last_stats.kernel_launches)
    fresh.close()
    g.close()
