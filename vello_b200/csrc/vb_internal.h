// vb_internal.h -- the renderer as the host files share it: vb_api.cu (lifetime, upload, frames, graphs), vb_stream.cu
// (vb_render_begin / vb_readback_wait) and vb_group.cu (vb_group_*). Not installed.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/vello_b200.h"
#include "vb_types.h"

#define CK(err, call)                                                                             \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            (err) = std::string(#call) + ": " + cudaGetErrorString(e_);                           \
            return VB_E_CUDA;                                                                     \
        }                                                                                         \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0; // bytes
};

// key of a captured frame: everything a launch argument is derived from (see enqueue)
struct GraphKey {
    VbConfig cfg;
    const void *ptrs[32];
    uint64_t ctl_words;
    uint32_t aa, cull, last;
    uint32_t xen, xrows[9];
    const void *xpeer[8];
};
struct GraphSlot {
    GraphKey key;
    cudaGraphExec_t exec = nullptr;
    uint32_t launches = 0;
};

struct FrameDest {        // where one frame's pixels go
    void *out_dev;        // caller's device buffer, or nullptr = the renderer's target
    void *host_out;       // rows copied here on copy_stream (nullptr = none)
    uint32_t bands;       // fine launches when host_out is set (1..8)
    uint32_t target;      // 0 = target, 1 = target_alt (streaming)
    bool zero_fine_queue; // vb_run_stages starting after stage 0
};

// An uploaded scene. Streaming (vb_render_begin) keeps TWO frames in flight: while frame k is rasterised, frame k+1's scene
// is uploaded into the other slot on its own stream and frame k-1's pixels drain to the host.
struct SceneSlot {
    DevBuf scene, ramps, atlas;
    VbLayout layout{};
    size_t scene_words = 0;
    uint32_t n_ramps = 0, atlas_w = 0, atlas_h = 0;
    bool have_scene = false;
    VbBump *h_bump = nullptr;     // pinned + mapped: the device writes the counters straight into host memory
    VbBump *h_bump_dev = nullptr; // device-side address of h_bump
};

struct vb_renderer {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool timing = false;
    uint32_t max_retries = 6;
    std::string err;
    int sm_count = 148;

    SceneSlot slot[2];
    uint32_t cur_slot = 0; // the slot frames are prepared and launched from
    SceneSlot &cur() { return slot[cur_slot]; }
    DevBuf mask8, mask16;

    // fixed-size intermediates
    DevBuf tag_monoids, path_bboxes, draw_monoids, info_bin_data, clip_inp, clip_bboxes, clip_scratch, draw_bboxes, bin_headers, paths,
        ctl, target, target_alt, tile_start, cls_list;
    // bump arenas (capacities in elements live in cap_*)
    DevBuf resolve_tmp; // patches, ramp descriptors and stops of vb_scene_upload_streams
    DevBuf lines, line_scratch, flatten_jobs, flatten_parts, tiles, seg_counts, segments, ptcl, blend_spill;
    uint32_t cap_lines = 0, cap_binning = 0, cap_tiles = 0, cap_seg_counts = 0, cap_segments = 0, cap_blend = 0, cap_ptcl = 0;

    // per-frame
    VbConfig cfg{};
    vb_params params{};
    FrameDest dest{}; // the prepared frame's (frame_prepare writes it, frame_launch reads it)
    uint32_t retries = 0, launches = 0;
    size_t ctl_words = 0;
    bool use_graph = true; // replay whole frames as CUDA graphs (see enqueue)
    GraphSlot graphs[4];
    uint32_t graph_next = 0;
    uint32_t readback_bands = 8; // fine launches per frame when vb_render's pixels go to the host
    uint32_t occlusion_cull = 1; // fine starts each tile at its last opaque full-tile cover
    uint32_t parts_pathtag = 0, parts_flatten = 0, parts_draw = 0, parts_tile = 0;
    size_t off_lb_pathtag = 0, off_lb_flatten = 0, off_lb_draw = 0, off_lb_tile = 0, off_lb_clip = 0;
    cudaEvent_t ev[VB_N_STAGE_IDS + 1]{};
    cudaEvent_t frame_ev[2]{}; // around every whole frame (vb_last_frame_ms: the signal stripe balancing uses)
    bool frame_timed = false;
    // read-back of a host destination: fine runs in row bands, each band's D2H copy overlaps the next band
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t band_ev[8]{};

    // streaming read-back (vb_render_begin): frames alternate between the two scene slots and the two targets, so that the
    // copy of frame n can still be draining while frame n+1 is rasterised
    bool stream_pending = false;
    cudaEvent_t copy_done[3]{};
    cudaStream_t upload_stream = nullptr;
    cudaEvent_t upload_done[2]{}, raster_done[2]{};
    struct RingFrame { // a streamed frame between vb_render_begin and its completion on the host
        bool pending = false, raster_checked = false;
        vb_params params{};
        void *out_host = nullptr;
        uint32_t slot = 0;
        vb_frame_stats stats{};
    } ring[3];
    uint64_t stream_seq = 0;

    // multi-GPU exchange (flatten sharded by tag range; k_exchange.cu)
    struct Exchange {
        bool configured = false, enabled = false;
        uint32_t rank = 0, world = 1, lines_cap = 0, n_paths = 0;
        size_t half_bytes = 0;
        DevBuf arena;
        void *peer[8] = {};
        uint32_t rows[9] = {};
    } xc;
};

// ---- defined in vb_api.cu for the other host files; not exported ---------------------------------------------------------
#define VB_HIDDEN __attribute__((visibility("hidden")))
// Upload a scene into the current slot, copies on stream `st`.
VB_HIDDEN int upload_on(vb_renderer *r, cudaStream_t st, const uint8_t *scene, size_t scene_len, const vb_layout *layout,
                        const uint32_t *ramps, uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h);
// A frame is enqueued in two steps: everything that may allocate, free or otherwise synchronise with the device (config,
// arenas, the output target), then the launches. vb_group runs step 1 for ALL its renderers before step 2 of any: with the
// exchange on, a renderer's frame contains a kernel that waits for its peers, and a peer that shares the device (tests)
// must not be stuck in a cudaFree behind that kernel.
VB_HIDDEN int frame_prepare(vb_renderer *r, const vb_params *p, const FrameDest &d);
VB_HIDDEN int frame_launch(vb_renderer *r);
// The same frame in two submissions (plain launches): up to and including flatten + the sending half of the exchange, then
// the rest. Used by vb_group when renderers share a device, see k_exchange.cu.
VB_HIDDEN int frame_launch_half(vb_renderer *r, int half);
// One frame, complete on return: launched, waited for, and after an arena overflow grown and re-run. The copies to a host
// destination are finished whatever the result. Does not drain streamed frames: public entry points do that, internal
// callers (the stream and the group themselves) must not.
VB_HIDDEN int render_attempts(vb_renderer *r, const vb_params *p, const FrameDest &d, vb_frame_stats *stats);
// Wait for the host-destination copies on copy_stream; an earlier error `rc` wins.
VB_HIDDEN int wait_copies(vb_renderer *r, int rc);
// After a failed attempt: enlarge whatever overflowed, using the counters the kernels kept counting.
VB_HIDDEN void grow_arenas(vb_renderer *r);
VB_HIDDEN void fill_stats(vb_renderer *r, vb_frame_stats *s);
