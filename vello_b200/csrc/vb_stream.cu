// vb_stream.cu -- streaming read-back: vb_render_begin / vb_readback_wait and the ring of frames in flight.
//
// Back-to-back frames with HOST buffers (a viewer / exporter reading every frame back, examples/headless/src/main.rs:188-210).
// Three frames are in flight: vb_render_begin(k) uploads frame k's scene into the free scene slot on the upload stream and
// enqueues its rasterisation and read-back; it then makes sure frame k-1 was RASTERISED without an arena overflow and that
// frame k-2's PIXELS are on the host. In steady state the GPU sees  upload(k+1) | raster(k) | read-back(k-1)  side by side and a
// frame costs max(raster, read-back) instead of their sum. On return every frame before the previous one is complete in its
// out_host and `stats` describes frame k-2 (zeros while there is none); vb_readback_wait completes the rest. THREE alternating
// out_host buffers are needed. An arena overflow is found at the rasterisation check; that frame (and the one enqueued behind
// it) is then re-run synchronously with grown arenas -- rare (first frames of a new scene size) and exact.
#include <string.h>

#include "vb_internal.h"

// A streamed frame's destination: its scene slot's target, the whole read-back in one band (it overlaps the next frames,
// there is no reason to split fine).
static FrameDest stream_dest(void *out_host, uint32_t slot) { return FrameDest{nullptr, out_host, 1u, slot, false}; }

static int rerun_frame_sync(vb_renderer *r, uint32_t q, vb_frame_stats *stats) {
    r->cur_slot = r->ring[q].slot;
    return render_attempts(r, &r->ring[q].params, stream_dest(r->ring[q].out_host, r->ring[q].slot), stats);
}

// Frame in ring entry q: wait for its kernels, look at its bump counters, re-run on overflow (together with the younger frame
// enqueued behind it, ring entry `younger`, or -1).
static int check_raster(vb_renderer *r, uint32_t q, int younger) {
    vb_renderer::RingFrame &f = r->ring[q];
    if (!f.pending || f.raster_checked) return VB_OK;
    const uint32_t keep = r->cur_slot;
    CK(r->err, cudaEventSynchronize(r->raster_done[f.slot]));
    r->cur_slot = f.slot;
    int rc = VB_OK;
    if (r->cur().h_bump->failed != 0u) {
        CK(r->err, cudaStreamSynchronize(r->stream));
        CK(r->err, cudaStreamSynchronize(r->copy_stream));
        grow_arenas(r);
        rc = rerun_frame_sync(r, q, &f.stats);
        CK(r->err, cudaEventRecord(r->copy_done[q], r->copy_stream));
        if (rc == VB_OK && younger >= 0 && r->ring[younger].pending) {
            r->cur_slot = r->ring[younger].slot;
            if (r->cur().h_bump->failed != 0u) {
                rc = rerun_frame_sync(r, (uint32_t)younger, &r->ring[younger].stats);
                CK(r->err, cudaEventRecord(r->raster_done[r->ring[younger].slot], r->stream));
                CK(r->err, cudaEventRecord(r->copy_done[younger], r->copy_stream));
            }
        }
    } else {
        r->retries = 0;
        fill_stats(r, &f.stats);
    }
    f.raster_checked = true;
    r->cur_slot = keep;
    return rc;
}

static int complete_host(vb_renderer *r, uint32_t q, vb_frame_stats *stats) {
    vb_renderer::RingFrame &f = r->ring[q];
    if (!f.pending) return VB_OK;
    int rc = check_raster(r, q, -1);
    CK(r->err, cudaEventSynchronize(r->copy_done[q]));
    if (stats) *stats = f.stats;
    f.pending = false;
    return rc;
}

extern "C" int vb_render_begin(vb_renderer *r, const uint8_t *scene, size_t scene_len, const vb_layout *layout, const uint32_t *ramps,
                               uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h,
                               const vb_params *p, void *out_host, vb_frame_stats *stats) {
    if (!r || !p || !out_host) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    if (stats) memset(stats, 0, sizeof *stats);
    const uint64_t k = r->stream_seq;
    const uint32_t slot = (uint32_t)(k & 1u), q = (uint32_t)(k % 3u), q1 = (uint32_t)((k + 2u) % 3u), q2 = (uint32_t)((k + 1u) % 3u);
    // frame k-2 (same scene slot, same device target) was checked by the previous call; frame k-3 (ring entry q) is complete
    r->cur_slot = slot;
    int rc = upload_on(r, r->upload_stream, scene, scene_len, layout, ramps, ramp_w, ramp_h, atlas, atlas_w, atlas_h);
    if (rc) return rc;
    CK(r->err, cudaEventRecord(r->upload_done[slot], r->upload_stream));
    CK(r->err, cudaStreamWaitEvent(r->stream, r->upload_done[slot], 0));
    if (k >= 2u && r->ring[q2].pending) CK(r->err, cudaStreamWaitEvent(r->stream, r->copy_done[q2], 0)); // its read-back still reads this target
    rc = frame_prepare(r, p, stream_dest(out_host, slot));
    if (rc == VB_OK) rc = frame_launch(r);
    if (rc) return rc;
    CK(r->err, cudaEventRecord(r->raster_done[slot], r->stream));
    CK(r->err, cudaEventRecord(r->copy_done[q], r->copy_stream));
    r->ring[q] = vb_renderer::RingFrame{true, false, *p, out_host, slot, {}};
    r->stream_seq = k + 1u;
    r->stream_pending = true;
    // frame k-1: rasterised without overflow?  frame k-2: pixels on the host?
    if (k >= 1u) rc = check_raster(r, q1, (int)q);
    if (k >= 2u) {
        const int rc2 = complete_host(r, q2, stats);
        if (rc == VB_OK) rc = rc2;
    }
    return rc;
}

extern "C" int vb_readback_wait(vb_renderer *r) {
    if (!r) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    int rc = VB_OK;
    const uint64_t k = r->stream_seq; // the next frame number: complete k-3 .. k-1 in order
    for (uint64_t j = k >= 3u ? k - 3u : 0u; j < k; j++) {
        const uint32_t q = (uint32_t)(j % 3u);
        const int younger = j + 1u < k ? (int)((j + 1u) % 3u) : -1;
        int rc1 = check_raster(r, q, younger);
        if (rc1 == VB_OK) rc1 = complete_host(r, q, nullptr);
        if (rc == VB_OK) rc = rc1;
    }
    CK(r->err, cudaStreamSynchronize(r->copy_stream));
    r->stream_pending = false;
    return rc;
}
