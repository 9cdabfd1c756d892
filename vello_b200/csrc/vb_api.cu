// vb_api.cu -- host orchestration + the extern "C" ABI declared in include/vello_b200.h.
//
// Replaces vello/src/render.rs (graph: stage order, bindings, buffer lifetimes) and
// vello/src/wgpu_engine.rs (engine) with a CUDA-stream pipeline. Unlike the reference
// (config.rs:398-408 fixed `1 << 21` arenas; lib.rs:762 "TODO: re-run on overflow") every
// bump-allocated arena is sized from the scene and grown + re-run when a frame overflows.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "vb_device.cuh"
#include "vb_internal.h"

// ---- stage launchers (k_*.cu) --------------------------------------------------------------
extern "C" {
void vb_launch_pathtag(const VbConfig *, const uint32_t *, VbTagMonoid *, uint32_t *, uint32_t, cudaStream_t);
uint32_t vb_pathtag_parts(uint32_t);
void vb_launch_flatten(const VbConfig *, const uint32_t *, const VbTagMonoid *, VbPathBbox *, VbBump *, VbLineSoup *, void *, void *, uint32_t *,
                       uint32_t *, uint32_t, int, uint32_t, uint32_t, cudaStream_t);
uint32_t vb_flatten_parts(uint32_t);
void vb_flatten_arena_bytes(uint32_t, size_t *, size_t *);
void vb_launch_draw(const VbConfig *, const uint32_t *, const VbPathBbox *, VbDrawMonoid *, uint32_t *, VbClipInp *, uint32_t *, uint32_t,
                    cudaStream_t);
uint32_t vb_draw_parts(uint32_t);
void vb_launch_clip(uint32_t, const VbClipInp *, const VbPathBbox *, VbDrawMonoid *, VbBbox4 *, int32_t *, uint32_t *, cudaStream_t);
uint32_t vb_clip_parts(uint32_t);
size_t vb_clip_scratch_words(uint32_t);
void vb_launch_binning(const VbConfig *, const VbDrawMonoid *, const VbPathBbox *, const VbBbox4 *, VbBbox4 *, VbBump *, uint32_t *,
                       VbBinHeader *, cudaStream_t);
void vb_launch_tile_alloc(const VbConfig *, const uint32_t *, const VbBbox4 *, VbBump *, VbPath *, VbTile *, uint32_t *, uint32_t,
                          cudaStream_t);
uint32_t vb_tile_alloc_parts(uint32_t);
void vb_launch_backdrop(const VbConfig *, VbBump *, const VbPath *, VbTile *, cudaStream_t);
void vb_launch_path_count(const VbConfig *, VbBump *, const VbLineSoup *, const VbPath *, VbTile *, VbSegmentCount *, uint32_t,
                          cudaStream_t);
void vb_launch_coarse(const VbConfig *, const uint32_t *, const VbDrawMonoid *, const VbBinHeader *, const uint32_t *, const VbPath *,
                      VbTile *, VbBump *, uint32_t *, uint32_t *, void *, uint32_t, cudaStream_t);
void vb_launch_path_tiling(const VbConfig *, VbBump *, const VbSegmentCount *, const VbLineSoup *, const VbPath *, const VbTile *,
                           VbSegment *, uint32_t, cudaStream_t);
void vb_launch_fine(const VbConfig *, int, const VbBump *, const VbSegment *, const uint32_t *, const uint32_t *, uint32_t *, uint32_t *,
                    const uint32_t *, const uint8_t *, const uint32_t *, const uint32_t *, const uint32_t *, uint32_t, uint32_t *, const void *,
                    const uint32_t *, uint32_t, int, cudaStream_t);
}

extern "C" int vb_fine_init_constants(void);
// k_exchange.cu: flatten sharded by tag range, lines / path boxes exchanged through peer memory
struct XPeersHost { // == XPeers in k_exchange.cu
    unsigned char *base[8];
    uint32_t rows[9];
    uint32_t world, rank, n_paths, lines_cap;
    unsigned long long half_bytes;
};
extern "C" size_t vb_exchange_half_bytes(uint32_t n_paths, uint32_t lines_cap);
extern "C" size_t vb_exchange_peers_bytes(void);
extern "C" uint32_t vb_exchange_epoch_word(void);
extern "C" void vb_launch_exchange_send(const void *, VbBump *, uint32_t, VbLineSoup *, uint32_t *, VbPathBbox *, int, cudaStream_t);
extern "C" void vb_launch_exchange_recv(const void *, VbBump *, uint32_t, VbLineSoup *, VbPathBbox *, int, cudaStream_t);
extern "C" void vb_launch_resolve_finish(uint32_t *, uint32_t, uint32_t, uint32_t, uint32_t, const void *, uint32_t, cudaStream_t);
extern "C" void vb_launch_make_ramps(const void *, const void *, uint32_t, uint32_t *, cudaStream_t);

// path_tiling_setup.wgsl:21-26 flags a failed frame to fine through ptcl[0] = ~0. That word is also tile 0's blend offset
// and is only rewritten when coarse visits tile 0 -- which a stripe window with bin_row0 > 0 never does, so the flag of a
// failed attempt would outlive the successful re-run and every later frame of that renderer. fine therefore reads
// bump.failed (zeroed with the control block at the start of every attempt) directly; ptcl[0] is not used as a flag.

// Statistics for the roofline of `fine`: PTCL words each tile's interpreter reads and segments it
// references (one thread per tile walks its command stream, as fine does).
__global__ void k_ptcl_stats(VbConfig cfg, const uint32_t *__restrict__ ptcl, const uint32_t *__restrict__ tile_start,
                             unsigned long long *out) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t wt = cfg.width_in_tiles, rows = cfg.win_ty1 - cfg.win_ty0;
    if (t >= wt * rows) return;
    uint32_t tile_ix = (cfg.win_ty0 + t / wt) * wt + t % wt;
    uint32_t ix = tile_ix * VB_PTCL_INITIAL_ALLOC + 1u;
    unsigned long long words = 1, segs = 0, fills = 0;
    if (tile_start && tile_start[tile_ix]) { // occlusion start: the interpreter begins at the tile's last opaque cover
        ix = tile_start[tile_ix];
        words += 1;
    }
    for (uint32_t guard = 0; guard < (1u << 24); guard++) {
        uint32_t tag = ptcl[ix];
        uint32_t size = 1;
        if (tag == VB_CMD_END) { words += 1; break; }
        if (tag == VB_CMD_JUMP) { words += 2; ix = ptcl[ix + 1]; continue; }
        if (tag == VB_CMD_FILL) { size = 4; segs += ptcl[ix + 1] >> 1; fills++; }
        else if (tag == VB_CMD_COLOR || tag == VB_CMD_IMAGE) size = 2;
        else if (tag == VB_CMD_LIN_GRAD || tag == VB_CMD_RAD_GRAD || tag == VB_CMD_SWEEP_GRAD || tag == VB_CMD_END_CLIP || tag == VB_CMD_BLUR_RECT) size = 3;
        words += size;
        ix += size;
    }
    atomicAdd(out, words);
    atomicAdd(out + 1, segs);
    atomicAdd(out + 2, fills);
}

// Frame start: zero the control block (bump counters, look-back descriptors, fine's tile queues) and reset the path bounding
// boxes (bbox_clear.wgsl: (+INT_MAX, -INT_MAX)) -- one launch; blocks past the control block clear 256 boxes each.
__global__ void k_frame_init(uint32_t *ctl, uint32_t words, uint32_t ctl_blocks, VbPathBbox *path_bboxes, uint32_t n_paths, uint32_t *xepoch) {
    if (xepoch != nullptr && blockIdx.x == 0u && threadIdx.x == 0u) *xepoch += 1u; // multi-GPU exchange: this attempt's epoch
    if (blockIdx.x < ctl_blocks) {
        for (uint32_t i = blockIdx.x * 1024u + threadIdx.x; i < min(words, (blockIdx.x + 1u) * 1024u); i += 256u) ctl[i] = 0u;
    } else {
        const uint32_t i = (blockIdx.x - ctl_blocks) * 256u + threadIdx.x;
        if (i < n_paths) {
            VbPathBbox b;
            b.x0 = 0x7fffffff; b.y0 = 0x7fffffff; b.x1 = (int32_t)0x80000000; b.y1 = (int32_t)0x80000000;
            b.draw_flags = 0; b.trans_ix = 0;
            path_bboxes[i] = b;
        }
    }
}
__global__ void k_publish_bump(const VbBump *bump, VbBump *host) {
    if (threadIdx.x < sizeof(VbBump) / 4u) {
        reinterpret_cast<volatile uint32_t *>(host)[threadIdx.x] = reinterpret_cast<const uint32_t *>(bump)[threadIdx.x];
        __threadfence_system();
    }
}

static int ensure(vb_renderer *r, DevBuf &b, size_t bytes) {
    if (bytes < 256) bytes = 256;
    if (b.cap >= bytes) return VB_OK;
    if (b.p) CK(r->err, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = (bytes + 255) & ~(size_t)255;
    CK(r->err, cudaMalloc(&b.p, want));
    b.cap = want;
    return VB_OK;
}
// Every device buffer of a renderer except the scene slots, resolve_tmp and the exchange arena: what vb_frame_stats.arena_bytes
// counts (with both slots' scene, ramps and atlas). `key`: its address is part of a captured graph's key; the targets are
// not, the frame's destination is.
using BufMember = DevBuf vb_renderer::*;
static const struct {
    BufMember buf;
    bool key;
} kBuffers[] = {
    {&vb_renderer::mask8, true},        {&vb_renderer::mask16, true},        {&vb_renderer::tag_monoids, true},
    {&vb_renderer::path_bboxes, true},  {&vb_renderer::draw_monoids, true},  {&vb_renderer::info_bin_data, true},
    {&vb_renderer::clip_inp, true},     {&vb_renderer::clip_bboxes, true},   {&vb_renderer::clip_scratch, true},
    {&vb_renderer::draw_bboxes, true},  {&vb_renderer::bin_headers, true},   {&vb_renderer::paths, true},
    {&vb_renderer::ctl, true},          {&vb_renderer::target, false},       {&vb_renderer::target_alt, false},
    {&vb_renderer::tile_start, true},   {&vb_renderer::cls_list, true},      {&vb_renderer::lines, true},
    {&vb_renderer::line_scratch, true}, {&vb_renderer::flatten_jobs, true},  {&vb_renderer::flatten_parts, true},
    {&vb_renderer::tiles, true},        {&vb_renderer::seg_counts, true},    {&vb_renderer::segments, true},
    {&vb_renderer::ptcl, true},         {&vb_renderer::blend_spill, true},
};

static size_t arena_bytes(const vb_renderer *r) {
    size_t s = 0;
    for (const SceneSlot &sl : r->slot) s += sl.scene.cap + sl.ramps.cap + sl.atlas.cap;
    for (const auto &b : kBuffers) s += (r->*b.buf).cap;
    return s;
}

// mask LUTs: vello_encoding/src/mask.rs:10-98 (f64 maths like the reference)
static uint32_t one_mask(double slope, double translation, bool is_pos, const uint8_t *pattern, int n) {
    if (is_pos) translation = 1. - translation;
    uint32_t result = 0;
    for (int i = 0; i < n; i++) {
        double y = (i + 0.5) * (1.0 / n);
        double x = (pattern[i] + 0.5) * (1.0 / n);
        if (!is_pos) y = 1. - y;
        if ((x - (1.0 - translation)) * (1. - slope) - (y - translation) * slope >= 0.) result |= 1u << i;
    }
    return result;
}
static void make_mask_luts(std::vector<uint32_t> &l8, std::vector<uint32_t> &l16) {
    static const uint8_t P8[8] = {0, 5, 3, 7, 1, 4, 6, 2};
    static const uint8_t P16[16] = {1, 8, 4, 11, 15, 7, 3, 12, 0, 9, 5, 13, 2, 10, 6, 14};
    l8.assign(256, 0);
    l16.assign(2048, 0);
    for (int i = 0; i < 32 * 32; i++) {
        int u = i % 32, v = i / 32;
        l8[i / 4] |= one_mask(((v % 16) + 0.5) * (1.0 / 16), (u + 0.5) * (1.0 / 32), v >= 16, P8, 8) << ((i % 4) * 8);
    }
    for (int i = 0; i < 64 * 64; i++) {
        int u = i % 64, v = i / 64;
        l16[i / 2] |= one_mask(((v % 32) + 0.5) * (1.0 / 32), (u + 0.5) * (1.0 / 64), v >= 32, P16, 16) << ((i % 2) * 16);
    }
}

extern "C" int vb_renderer_new(const vb_options *opt, vb_renderer **out) {
    if (!out) return VB_E_INVALID;
    vb_renderer *r = new vb_renderer();
    r->device = opt ? opt->device : 0;
    r->timing = opt && opt->timing;
    if (opt && opt->max_retries) r->max_retries = opt->max_retries;
    cudaError_t e = cudaSetDevice(r->device);
    if (e != cudaSuccess) {
        fprintf(stderr, "vello_b200: cudaSetDevice(%d): %s\n", r->device, cudaGetErrorString(e));
        vb_renderer_free(r);
        return VB_E_CUDA;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, r->device) == cudaSuccess) r->sm_count = prop.multiProcessorCount;
    bool ok = cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&r->upload_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&r->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    for (SceneSlot &s : r->slot) {
        ok = ok && cudaHostAlloc((void **)&s.h_bump, sizeof(VbBump), cudaHostAllocMapped) == cudaSuccess &&
             cudaHostGetDevicePointer((void **)&s.h_bump_dev, s.h_bump, 0) == cudaSuccess;
        if (ok) memset(s.h_bump, 0, sizeof(VbBump));
    }
    for (auto &ev : r->upload_done) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto &ev : r->raster_done) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto &ev : r->ev) cudaEventCreate(&ev);
    for (auto &ev : r->frame_ev) cudaEventCreate(&ev);
    for (auto &ev : r->band_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto &ev : r->copy_done) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (getenv("VELLO_B200_NO_GRAPH")) r->use_graph = false;
    std::vector<uint32_t> l8, l16;
    make_mask_luts(l8, l16);
    if (!ok || vb_fine_init_constants() != 0 || ensure(r, r->mask8, l8.size() * 4) || ensure(r, r->mask16, l16.size() * 4)) {
        vb_renderer_free(r);
        return VB_E_CUDA;
    }
    cudaMemcpy(r->mask8.p, l8.data(), l8.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(r->mask16.p, l16.data(), l16.size() * 4, cudaMemcpyHostToDevice);
    *out = r;
    return VB_OK;
}

template <size_t N> static void destroy_events(cudaEvent_t (&evs)[N]) {
    for (cudaEvent_t ev : evs)
        if (ev) cudaEventDestroy(ev);
}

// Also frees a partly built renderer (vb_renderer_new's error paths): whatever was not created is null.
extern "C" void vb_renderer_free(vb_renderer *r) {
    if (!r) return;
    cudaSetDevice(r->device);
    if (r->stream) cudaStreamSynchronize(r->stream);
    for (const auto &b : kBuffers)
        if ((r->*b.buf).p) cudaFree((r->*b.buf).p);
    for (SceneSlot &s : r->slot) {
        for (DevBuf *b : {&s.scene, &s.ramps, &s.atlas})
            if (b->p) cudaFree(b->p);
        if (s.h_bump) cudaFreeHost(s.h_bump);
    }
    for (DevBuf *b : {&r->resolve_tmp, &r->xc.arena})
        if (b->p) cudaFree(b->p);
    destroy_events(r->ev);
    destroy_events(r->frame_ev);
    destroy_events(r->band_ev);
    destroy_events(r->copy_done);
    destroy_events(r->upload_done);
    destroy_events(r->raster_done);
    for (auto &gs : r->graphs)
        if (gs.exec) cudaGraphExecDestroy(gs.exec);
    for (cudaStream_t st : {r->copy_stream, r->upload_stream, r->stream})
        if (st) cudaStreamDestroy(st);
    delete r;
}

extern "C" const char *vb_strerror(int code) {
    switch (code) {
    case VB_OK: return "ok";
    case VB_E_INVALID: return "invalid argument";
    case VB_E_CUDA: return "CUDA error (see vb_last_error)";
    case VB_E_BUMP_OVERFLOW: return "bump arena overflow persisted after grow-and-retry";
    case VB_E_NO_SCENE: return "no scene uploaded";
    case VB_E_UNKNOWN_BUFFER: return "unknown buffer name";
    default: return "unknown error";
    }
}
extern "C" const char *vb_last_error(vb_renderer *r) { return r ? r->err.c_str() : ""; }
extern "C" void *vb_stream(vb_renderer *r) { return r ? (void *)r->stream : nullptr; }
extern "C" void *vb_target(vb_renderer *r, size_t *bytes) {
    if (!r) return nullptr;
    if (bytes) *bytes = r->target.cap;
    return r->target.p;
}
extern "C" int vb_copy_to_host(vb_renderer *r, const void *src_device, void *dst_host, size_t bytes) {
    if (!r || !src_device || !dst_host) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost, r->stream));
    CK(r->err, cudaStreamSynchronize(r->stream));
    return VB_OK;
}

int upload_on(vb_renderer *r, cudaStream_t st, const uint8_t *scene, size_t scene_len, const vb_layout *layout, const uint32_t *ramps,
              uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h) {
    if (!r || !layout || (scene_len && !scene) || (scene_len & 3)) return VB_E_INVALID;
    if (ramp_h && ramp_w != 512) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    SceneSlot &s = r->cur();
    memcpy(&s.layout, layout, sizeof(VbLayout));
    s.scene_words = scene_len / 4;
    int rc;
    if ((rc = ensure(r, s.scene, scene_len + 64))) return rc;
    if (scene_len) CK(r->err, cudaMemcpyAsync(s.scene.p, scene, scene_len, cudaMemcpyHostToDevice, st));
    s.n_ramps = ramp_h;
    if ((rc = ensure(r, s.ramps, (size_t)ramp_h * 512 * 4))) return rc;
    if (ramp_h) CK(r->err, cudaMemcpyAsync(s.ramps.p, ramps, (size_t)ramp_h * 512 * 4, cudaMemcpyHostToDevice, st));
    s.atlas_w = atlas ? atlas_w : 0;
    s.atlas_h = atlas ? atlas_h : 0;
    if ((rc = ensure(r, s.atlas, (size_t)s.atlas_w * s.atlas_h * 4))) return rc;
    if (s.atlas_w && s.atlas_h)
        CK(r->err, cudaMemcpyAsync(s.atlas.p, atlas, (size_t)s.atlas_w * s.atlas_h * 4, cudaMemcpyHostToDevice, st));
    s.have_scene = true;
    return VB_OK;
}

// A public entry point other than the streaming pair, used while streamed frames are still in flight, completes them first.
static int drain_stream(vb_renderer *r) { return r->stream_pending ? vb_readback_wait(r) : VB_OK; }

extern "C" int vb_scene_upload(vb_renderer *r, const uint8_t *scene, size_t scene_len, const vb_layout *layout, const uint32_t *ramps,
                               uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h) {
    if (!r) return VB_E_INVALID;
    int rc = drain_stream(r);
    if (rc) return rc;
    return upload_on(r, r->stream, scene, scene_len, layout, ramps, ramp_w, ramp_h, atlas, atlas_w, atlas_h);
}

static uint32_t grow(uint32_t need) {
    uint64_t g = (uint64_t)need + need / 4 + 1024;
    return g > 0xfffffff0ull ? 0xfffffff0u : (uint32_t)g;
}

// Compute the config for these params, size the fixed buffers, and (first time / after growth) the arenas.
static int prepare(vb_renderer *r, const vb_params *p) {
    // RenderParams sanity (the reference panics / produces nothing on these; here they are argument errors)
    if (p->width == 0u || p->height == 0u || p->aa > 2u || p->width > 65536u || p->height > 65536u) {
        r->err = "vb_params: width/height must be 1..65536 and aa 0..2";
        return VB_E_INVALID;
    }
    {
        const uint64_t nt = (uint64_t)((p->width + 15u) / 16u) * ((p->height + 15u) / 16u);
        if (nt * VB_PTCL_INITIAL_ALLOC + nt * (VB_PTCL_INCREMENT / 8u) + 65536u > 0xf0000000ull) {
            r->err = "vb_params: tile count * PTCL allocation exceeds 32-bit word offsets";
            return VB_E_INVALID;
        }
    }
    VbConfig &c = r->cfg;
    memset(&c, 0, sizeof c);
    c.width_in_tiles = (p->width + 15u) / 16u;
    c.height_in_tiles = (p->height + 15u) / 16u;
    c.target_width = p->width;
    c.target_height = p->height;
    c.base_color = p->base_color;
    const SceneSlot &s = r->cur();
    c.layout = s.layout;
    const uint32_t hb = (c.height_in_tiles + 15u) / 16u, wb = (c.width_in_tiles + 15u) / 16u;
    c.win_by0 = 0;
    c.win_by1 = hb;
    if (p->bin_row1 > p->bin_row0) {
        c.win_by0 = p->bin_row0 < hb ? p->bin_row0 : hb;
        c.win_by1 = p->bin_row1 < hb ? p->bin_row1 : hb;
    }
    c.win_ty0 = c.win_by0 * 16u;
    c.win_ty1 = c.win_by1 * 16u < c.height_in_tiles ? c.win_by1 * 16u : c.height_in_tiles;
    if (p->tile_row1 > p->tile_row0) {
        // stripe in tile rows: binning / coarse cover the bins that contain it, tile_alloc clamps every path to its rows
        // (so the extra tiles of a partly covered bin row hold empty command lists), fine paints exactly the stripe
        c.win_ty0 = p->tile_row0 < c.height_in_tiles ? p->tile_row0 : c.height_in_tiles;
        c.win_ty1 = p->tile_row1 < c.height_in_tiles ? p->tile_row1 : c.height_in_tiles;
        c.win_by0 = c.win_ty0 / 16u;
        c.win_by1 = (c.win_ty1 + 15u) / 16u;
    }
    c.win_cull = (c.win_ty0 > 0u || c.win_ty1 < c.height_in_tiles) ? 1u : 0u;
    c.n_tag_words = s.layout.path_data_base - s.layout.path_tag_base;
    c.scene_words = (uint32_t)s.scene_words;
    c.n_ramps = s.n_ramps;
    c.atlas_w = s.atlas_w;
    c.atlas_h = s.atlas_h;
    c.out_pitch_px = p->width;
    c.out_row0 = c.win_ty0 * 16u;
    r->params = *p;

    const VbLayout &L = s.layout;
    const uint32_t n_draw = L.n_draw_objects, n_paths = L.n_paths, n_clips = L.n_clips;
    const uint32_t n_tiles = c.width_in_tiles * c.height_in_tiles;
    const uint32_t n_bins = wb * hb, aligned_n_bins = (n_bins + 255u) & ~255u;
    int rc;
    if ((rc = ensure(r, r->tag_monoids, (size_t)c.n_tag_words * sizeof(VbTagMonoid)))) return rc;
    if ((rc = ensure(r, r->path_bboxes, (size_t)n_paths * sizeof(VbPathBbox)))) return rc;
    if ((rc = ensure(r, r->draw_monoids, (size_t)n_draw * sizeof(VbDrawMonoid)))) return rc;
    if ((rc = ensure(r, r->clip_inp, (size_t)n_clips * sizeof(VbClipInp)))) return rc;
    if ((rc = ensure(r, r->clip_bboxes, (size_t)n_clips * sizeof(VbBbox4)))) return rc;
    if ((rc = ensure(r, r->clip_scratch, vb_clip_scratch_words(n_clips) * 4))) return rc;
    if ((rc = ensure(r, r->draw_bboxes, (size_t)n_draw * sizeof(VbBbox4)))) return rc;
    if ((rc = ensure(r, r->bin_headers, (size_t)((n_draw + 255u) / 256u) * aligned_n_bins * sizeof(VbBinHeader)))) return rc;
    if ((rc = ensure(r, r->paths, (size_t)((n_draw + 255u) & ~255u) * sizeof(VbPath)))) return rc;
    if ((rc = ensure(r, r->tile_start, ((size_t)n_tiles + 256) * 4))) return rc;
    if ((rc = ensure(r, r->cls_list, (size_t)VB_FINE_CLASSES * n_tiles * 8))) return rc; // fine's cost-ordered tile lists

    // first-guess arena capacities (elements); they only ever grow
    const uint32_t n_tags = c.n_tag_words * 4u;
    auto atleast = [](uint32_t &cap, uint64_t v) {
        if (v > 0xfffffff0ull) v = 0xfffffff0ull;
        if (cap < (uint32_t)v) cap = (uint32_t)v;
    };
    atleast(r->cap_lines, (uint64_t)n_tags * 2 + 4096);
    atleast(r->cap_binning, (uint64_t)n_draw * 4 + 4096);
    atleast(r->cap_tiles, (uint64_t)n_draw * 16 + 4096);
    atleast(r->cap_seg_counts, (uint64_t)r->cap_lines * 2);
    atleast(r->cap_segments, (uint64_t)r->cap_seg_counts);
    atleast(r->cap_blend, 256);
    atleast(r->cap_ptcl, (uint64_t)n_tiles * VB_PTCL_INITIAL_ALLOC + (uint64_t)VB_PTCL_INCREMENT * (64 + n_tiles / 8));
    if (r->cap_ptcl < n_tiles * VB_PTCL_INITIAL_ALLOC + VB_PTCL_INCREMENT)
        r->cap_ptcl = n_tiles * VB_PTCL_INITIAL_ALLOC + VB_PTCL_INCREMENT;
    if ((rc = ensure(r, r->lines, (size_t)r->cap_lines * sizeof(VbLineSoup)))) return rc;
    {
        size_t lit_bytes, job_bytes;
        vb_flatten_arena_bytes(r->cap_lines, &lit_bytes, &job_bytes);
        if ((rc = ensure(r, r->line_scratch, lit_bytes))) return rc;
        if ((rc = ensure(r, r->flatten_jobs, job_bytes))) return rc;
    }
    if ((rc = ensure(r, r->info_bin_data, ((size_t)L.bin_data_start + r->cap_binning) * 4))) return rc;
    if ((rc = ensure(r, r->tiles, (size_t)r->cap_tiles * sizeof(VbTile)))) return rc;
    if ((rc = ensure(r, r->seg_counts, (size_t)r->cap_seg_counts * sizeof(VbSegmentCount)))) return rc;
    if ((rc = ensure(r, r->segments, (size_t)r->cap_segments * sizeof(VbSegment)))) return rc;
    if ((rc = ensure(r, r->blend_spill, (size_t)r->cap_blend * 4))) return rc;
    if ((rc = ensure(r, r->ptcl, (size_t)r->cap_ptcl * 4 + 512))) return rc; // + slack for fine's 256-byte command windows
    c.lines_size = r->cap_lines;
    c.binning_size = r->cap_binning;
    c.tiles_size = r->cap_tiles;
    c.seg_counts_size = r->cap_seg_counts;
    c.segments_size = r->cap_segments;
    c.blend_size = r->cap_blend;
    c.ptcl_size = r->cap_ptcl;

    // control block: [bump (8 words, padded to 16)] [look-back states]
    r->parts_pathtag = vb_pathtag_parts(c.n_tag_words);
    r->parts_flatten = vb_flatten_parts(c.n_tag_words);
    r->parts_draw = vb_draw_parts(n_draw);
    r->parts_tile = vb_tile_alloc_parts(n_draw);
    size_t off = VB_CTL_HEADER_WORDS;
    r->off_lb_pathtag = off; off += vb_lookback_words(r->parts_pathtag, 5);
    r->off_lb_flatten = off; // flatten: [0] literal-record counter, [1] job counter, [4..] look-back state of its partition scan
    off += 4 + vb_lookback_words((r->parts_flatten + 8191u) / 8192u, 1);
    r->off_lb_draw = off; off += vb_lookback_words(r->parts_draw, 4);
    r->off_lb_tile = off; off += vb_lookback_words(r->parts_tile, 1);
    r->off_lb_clip = off; off += vb_lookback_words(vb_clip_parts(n_clips), 1);
    r->ctl_words = off;
    if ((rc = ensure(r, r->ctl, off * 4))) return rc;
    if ((rc = ensure(r, r->flatten_parts, ((size_t)r->parts_flatten * 34 + 8) * 4))) return rc;
    return VB_OK;
}

static void xpeers_of(const vb_renderer *r, XPeersHost *X) {
    memset(X, 0, sizeof *X);
    for (uint32_t i = 0; i < r->xc.world; i++) X->base[i] = (unsigned char *)r->xc.peer[i];
    for (uint32_t i = 0; i <= r->xc.world; i++) X->rows[i] = r->xc.rows[i];
    X->world = r->xc.world; X->rank = r->xc.rank; X->n_paths = r->xc.n_paths; X->lines_cap = r->xc.lines_cap; X->half_bytes = r->xc.half_bytes;
}

static void rec(vb_renderer *r, int i) {
    if (r->timing) cudaEventRecord(r->ev[i], r->stream);
}

// grid of the kernels that stride over a bump arena: from its capacity, at most 16 blocks per SM
static uint32_t arena_grid(const vb_renderer *r, uint32_t cap) {
    const uint64_t blocks = ((uint64_t)cap + 255) / 256;
    return (uint32_t)(blocks < (uint64_t)r->sm_count * 16 ? blocks : (uint64_t)r->sm_count * 16);
}

// Queue the device->host copy of the destination's tile rows ty0..ty1 on copy_stream, behind what `stream` has enqueued so far.
static int queue_readback(vb_renderer *r, const FrameDest &d, uint32_t ty0, uint32_t ty1, uint32_t band) {
    const VbConfig &c = r->cfg;
    size_t y0 = (size_t)ty0 * 16u, y1 = (size_t)ty1 * 16u;
    if (y1 > c.target_height) y1 = c.target_height;
    if (y1 <= y0) return VB_OK;
    const size_t off = (y0 - c.out_row0) * c.out_pitch_px * 4u, bytes = (y1 - y0) * c.out_pitch_px * 4u;
    CK(r->err, cudaEventRecord(r->band_ev[band], r->stream));
    CK(r->err, cudaStreamWaitEvent(r->copy_stream, r->band_ev[band], 0));
    CK(r->err, cudaMemcpyAsync((char *)d.host_out + off, (const char *)d.out_dev + off, bytes, cudaMemcpyDeviceToHost, r->copy_stream));
    return VB_OK;
}

// Enqueue stages first..last. Does not synchronise.
static int enqueue_direct(vb_renderer *r, int first, int last, const FrameDest &d) {
    const VbConfig &c = r->cfg;
    const SceneSlot &s = r->cur();
    cudaStream_t st = r->stream;
    uint32_t *ctl = (uint32_t *)r->ctl.p;
    VbBump *bump = (VbBump *)ctl;
    uint32_t launches = 0;
    const uint32_t n_draw = c.layout.n_draw_objects;
    if (first == 0) {
        // a kernel, not cudaMemsetAsync: small memsets / copies are served by a copy engine and would queue behind a
        // 64 MiB read-back still draining from the previous frame (measured: +1.2 ms per streamed frame)
        const unsigned ctl_blocks = (unsigned)((r->ctl_words + 1023) / 1024), bb_blocks = (c.layout.n_paths + 255u) / 256u;
        uint32_t *xepoch = r->xc.enabled ? (uint32_t *)r->xc.arena.p + vb_exchange_epoch_word() : nullptr;
        k_frame_init<<<ctl_blocks + bb_blocks, 256, 0, st>>>(ctl, (uint32_t)r->ctl_words, ctl_blocks, (VbPathBbox *)r->path_bboxes.p, c.layout.n_paths,
                                                             xepoch);
        launches++;
    }
    else if (d.zero_fine_queue) {
        // vb_run_stages starting after stage 0: the control block is not zeroed, but fine's tile queues must start at 0 and
        // coarse must append to empty class lists
        if (last >= VB_STAGE_ID_FINE) CK(r->err, cudaMemsetAsync(ctl + VB_CTL_FINE_QUEUE, 0, 8 * sizeof(uint32_t), st));
        if (first <= VB_STAGE_ID_COARSE && last >= VB_STAGE_ID_COARSE)
            CK(r->err, cudaMemsetAsync(ctl + VB_CTL_FINE_CLASS, 0, VB_FINE_CLASSES * sizeof(uint32_t), st));
    }
    rec(r, 0);
    for (int stage = first; stage <= last; stage++) {
        switch (stage) {
        case VB_STAGE_ID_PATHTAG:
            vb_launch_pathtag(&c, (const uint32_t *)s.scene.p, (VbTagMonoid *)r->tag_monoids.p, ctl + r->off_lb_pathtag, r->parts_pathtag, st);
            launches += r->parts_pathtag ? 1 : 0;
            break;
        case VB_STAGE_ID_FLATTEN: {
            // With the exchange on, this GPU flattens its share of the tag stream (no stripe culling: the lines are for
            // everybody), then the lines and path boxes are exchanged through peer memory (k_exchange.cu).
            VbConfig cf = c;
            uint32_t p0 = 0u, p1 = r->parts_flatten;
            if (r->xc.enabled) {
                const uint32_t P = r->parts_flatten, G = r->xc.world, k = r->xc.rank;
                cf.win_cull = 0u;
                p0 = (uint32_t)((uint64_t)P * k / G) & ~7u;
                p1 = k + 1u == G ? P : ((uint32_t)((uint64_t)P * (k + 1u) / G) & ~7u);
            }
            vb_launch_flatten(&cf, (const uint32_t *)s.scene.p, (const VbTagMonoid *)r->tag_monoids.p, (VbPathBbox *)r->path_bboxes.p, bump,
                              (VbLineSoup *)r->lines.p, r->line_scratch.p, r->flatten_jobs.p, (uint32_t *)r->flatten_parts.p,
                              ctl + r->off_lb_flatten, r->parts_flatten, first != 0 ? 1 : 0, p0, p1, st);
            if (r->xc.enabled) {
                XPeersHost X;
                xpeers_of(r, &X);
                vb_launch_exchange_send(&X, bump, c.lines_size, (VbLineSoup *)r->lines.p, ctl + VB_CTL_XCHG_SCRATCH,
                                        (VbPathBbox *)r->path_bboxes.p, r->sm_count, st);
                launches += (r->parts_flatten ? 3 : 0) + 4;
            } else {
                launches += (first != 0 && c.layout.n_paths ? 1 : 0) + (r->parts_flatten ? 3 : 0);
            }
            break;
        }
        case VB_STAGE_ID_DRAW:
            if (r->xc.enabled) { // second half of the exchange: my lines and the complete path boxes arrive before draw_leaf reads them
                XPeersHost X;
                xpeers_of(r, &X);
                vb_launch_exchange_recv(&X, bump, c.lines_size, (VbLineSoup *)r->lines.p, (VbPathBbox *)r->path_bboxes.p, r->sm_count, st);
                launches += 3;
            }
            vb_launch_draw(&c, (const uint32_t *)s.scene.p, (const VbPathBbox *)r->path_bboxes.p, (VbDrawMonoid *)r->draw_monoids.p,
                           (uint32_t *)r->info_bin_data.p, (VbClipInp *)r->clip_inp.p, ctl + r->off_lb_draw, r->parts_draw, st);
            launches += r->parts_draw ? 1 : 0;
            break;
        case VB_STAGE_ID_CLIP:
            vb_launch_clip(c.layout.n_clips, (const VbClipInp *)r->clip_inp.p, (const VbPathBbox *)r->path_bboxes.p,
                           (VbDrawMonoid *)r->draw_monoids.p, (VbBbox4 *)r->clip_bboxes.p, (int32_t *)r->clip_scratch.p,
                           ctl + r->off_lb_clip, st);
            launches += c.layout.n_clips ? 3 : 0;
            break;
        case VB_STAGE_ID_BINNING:
            vb_launch_binning(&c, (const VbDrawMonoid *)r->draw_monoids.p, (const VbPathBbox *)r->path_bboxes.p,
                              (const VbBbox4 *)r->clip_bboxes.p, (VbBbox4 *)r->draw_bboxes.p, bump, (uint32_t *)r->info_bin_data.p,
                              (VbBinHeader *)r->bin_headers.p, st);
            launches += n_draw ? 1 : 0;
            break;
        case VB_STAGE_ID_TILE_ALLOC:
            vb_launch_tile_alloc(&c, (const uint32_t *)s.scene.p, (const VbBbox4 *)r->draw_bboxes.p, bump, (VbPath *)r->paths.p,
                                 (VbTile *)r->tiles.p, ctl + r->off_lb_tile, r->parts_tile, st);
            launches += r->parts_tile ? 2 : 0;
            break;
        case VB_STAGE_ID_PATH_COUNT: // the kernel strides over bump.lines read on the device
            vb_launch_path_count(&c, bump, (const VbLineSoup *)r->lines.p, (const VbPath *)r->paths.p, (VbTile *)r->tiles.p,
                                 (VbSegmentCount *)r->seg_counts.p, arena_grid(r, c.lines_size), st);
            launches += 1;
            break;
        case VB_STAGE_ID_BACKDROP:
            vb_launch_backdrop(&c, bump, (const VbPath *)r->paths.p, (VbTile *)r->tiles.p, st);
            launches += n_draw ? 1 : 0;
            break;
        case VB_STAGE_ID_COARSE:
            vb_launch_coarse(&c, (const uint32_t *)s.scene.p, (const VbDrawMonoid *)r->draw_monoids.p, (const VbBinHeader *)r->bin_headers.p,
                             (const uint32_t *)r->info_bin_data.p, (const VbPath *)r->paths.p, (VbTile *)r->tiles.p, bump,
                             (uint32_t *)r->ptcl.p, (uint32_t *)r->tile_start.p, r->cls_list.p, c.width_in_tiles * c.height_in_tiles, st);
            launches += 1;
            break;
        case VB_STAGE_ID_PATH_TILING:
            vb_launch_path_tiling(&c, bump, (const VbSegmentCount *)r->seg_counts.p, (const VbLineSoup *)r->lines.p,
                                  (const VbPath *)r->paths.p, (const VbTile *)r->tiles.p, (VbSegment *)r->segments.p,
                                  arena_grid(r, c.seg_counts_size), st);
            launches += 1;
            break;
        case VB_STAGE_ID_FINE: {
            // With a host destination fine is launched in up to d.bands bands of tile rows and each band's device->host copy
            // is queued on a second stream behind an event, so the read-back of band k overlaps the rasterisation of band
            // k+1 (only the last band's copy is exposed).
            const uint32_t rows = c.win_ty1 - c.win_ty0;
            const uint32_t n_bands = (d.host_out && rows >= 64u) ? d.bands : 1u;
            const uint32_t band_rows = (rows + n_bands - 1u) / n_bands;
            for (uint32_t b = 0; b < n_bands; b++) {
                VbConfig cb = c;
                cb.win_ty0 = c.win_ty0 + b * band_rows;
                cb.win_ty1 = cb.win_ty0 + band_rows < c.win_ty1 ? cb.win_ty0 + band_rows : c.win_ty1;
                if (cb.win_ty0 >= cb.win_ty1) break;
                vb_launch_fine(&cb, (int)r->params.aa, bump, (const VbSegment *)r->segments.p, (const uint32_t *)r->ptcl.p,
                               (const uint32_t *)r->info_bin_data.p, (uint32_t *)r->blend_spill.p, (uint32_t *)d.out_dev,
                               (const uint32_t *)s.ramps.p, (const uint8_t *)s.atlas.p, (const uint32_t *)r->mask8.p,
                               (const uint32_t *)r->mask16.p, (const uint32_t *)r->tile_start.p, r->occlusion_cull,
                               ctl + VB_CTL_FINE_QUEUE + b, r->cls_list.p, n_bands == 1u ? ctl + VB_CTL_FINE_CLASS : nullptr,
                               c.width_in_tiles * c.height_in_tiles, r->sm_count, st);
                launches += 1;
                if (d.host_out) {
                    const int rc = queue_readback(r, d, cb.win_ty0, cb.win_ty1, b);
                    if (rc) return rc;
                }
            }
            break;
        }
        default: return VB_E_INVALID;
        }
        rec(r, stage + 1);
    }
    k_publish_bump<<<1, 32, 0, st>>>(bump, s.h_bump_dev); // zero-copy store to mapped host memory (no copy engine)
    launches++;
    CK(r->err, cudaGetLastError());
    r->launches = launches;
    return VB_OK;
}

// ---- whole-frame CUDA graphs ---------------------------------------------------------------------------------------------
// A frame is ~20 kernel launches. Each launch makes the GPU fetch a command buffer from host memory over PCIe; while a
// 64 MiB read-back of the previous frame is streaming the other way that fetch queues behind it (measured with
// tools/e2e_probe.py: every stage of a streamed frame started ~10 us late per launch, +0.3 ms per frame). In steady state
// the launches of a frame are identical -- same kernels, grids, arena pointers, config -- so they are captured once into a
// graph and replayed with ONE submission. The key is everything a launch argument is derived from; growing an arena or
// changing the scene layout / frame size / window simply misses the cache and re-captures.
static void graph_key(vb_renderer *r, int last, const void *out_dev, GraphKey *k) {
    memset(k, 0, sizeof *k);
    k->cfg = r->cfg;
    const SceneSlot &s = r->cur();
    size_t n = 0;
    for (const DevBuf *b : {&s.scene, &s.ramps, &s.atlas}) k->ptrs[n++] = b->p;
    for (const auto &b : kBuffers)
        if (b.key) k->ptrs[n++] = (r->*b.buf).p;
    k->ptrs[n++] = out_dev;
    k->ptrs[n++] = s.h_bump_dev;
    k->ctl_words = r->ctl_words;
    k->aa = r->params.aa;
    k->cull = r->occlusion_cull;
    k->last = (uint32_t)last;
    k->xen = r->xc.enabled ? 1u + r->xc.rank + (r->xc.world << 8) : 0u;
    if (r->xc.enabled) {
        memcpy(k->xrows, r->xc.rows, sizeof k->xrows);
        memcpy(k->xpeer, r->xc.peer, sizeof k->xpeer);
    }
}

// Enqueue stages first..last: through a cached graph for whole frames, directly otherwise.
static int enqueue(vb_renderer *r, int first, int last, const FrameDest &d) {
    const VbConfig &c = r->cfg;
    if (!r->use_graph || r->timing || first != 0 || last != VB_N_STAGE_IDS - 1) return enqueue_direct(r, first, last, d);
    // with a host destination split into bands, fine and its interleaved copies stay outside the graph
    const uint32_t rows = c.win_ty1 - c.win_ty0;
    const bool banded = d.host_out && rows >= 64u && d.bands > 1u;
    const int g_last = banded ? VB_STAGE_ID_FINE - 1 : last;
    GraphKey key;
    graph_key(r, g_last, d.out_dev, &key);
    GraphSlot *slot = nullptr;
    for (GraphSlot &gs : r->graphs)
        if (gs.exec && memcmp(&gs.key, &key, sizeof key) == 0) slot = &gs;
    // Any refusal along the way (a tool or driver that does not allow capture here) turns graph replay off for this renderer
    // and the frame is launched kernel by kernel: graphs are an optimisation, never a requirement.
    auto without_graph = [&]() {
        cudaGetLastError();
        r->use_graph = false;
        return enqueue_direct(r, first, last, d);
    };
    if (!slot) {
        slot = &r->graphs[r->graph_next++ % (sizeof r->graphs / sizeof r->graphs[0])];
        if (slot->exec) {
            cudaGraphExecDestroy(slot->exec);
            slot->exec = nullptr;
        }
        if (cudaStreamBeginCapture(r->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) return without_graph();
        FrameDest captured = d;
        captured.host_out = nullptr; // the captured fine is one launch; its read-back is queued after the graph, below
        const int rc = enqueue_direct(r, 0, g_last, captured);
        cudaGraph_t g = nullptr;
        const cudaError_t e = cudaStreamEndCapture(r->stream, &g);
        if (rc != VB_OK || e != cudaSuccess || !g) {
            if (g) cudaGraphDestroy(g);
            return without_graph();
        }
        const cudaError_t ei = cudaGraphInstantiate(&slot->exec, g, 0);
        cudaGraphDestroy(g);
        if (ei != cudaSuccess) {
            slot->exec = nullptr;
            return without_graph();
        }
        slot->key = key;
        slot->launches = r->launches;
    }
    if (cudaGraphLaunch(slot->exec, r->stream) != cudaSuccess) {
        cudaGetLastError();
        cudaGraphExecDestroy(slot->exec);
        slot->exec = nullptr;
        return without_graph();
    }
    r->launches = slot->launches;
    if (banded) {
        const int rc = enqueue_direct(r, VB_STAGE_ID_FINE, VB_STAGE_ID_FINE, d);
        r->launches += slot->launches;
        return rc;
    }
    if (d.host_out) return queue_readback(r, d, c.win_ty0, c.win_ty1, 0);
    return VB_OK;
}

// Resolve a destination without a device buffer to the renderer's target, sized for the configured window.
static int pick_out(vb_renderer *r, FrameDest &d) {
    if (d.out_dev) return VB_OK;
    const VbConfig &c = r->cfg;
    size_t rows = (size_t)(c.win_ty1 - c.win_ty0) * 16u;
    DevBuf &t = d.target ? r->target_alt : r->target;
    int rc = ensure(r, t, (size_t)c.out_pitch_px * 4u * rows);
    d.out_dev = t.p;
    return rc;
}

int frame_prepare(vb_renderer *r, const vb_params *p, const FrameDest &d) {
    if (!r || !p) return VB_E_INVALID;
    if (!r->cur().have_scene) return VB_E_NO_SCENE;
    CK(r->err, cudaSetDevice(r->device));
    FrameDest dest = d;
    int rc = prepare(r, p);
    if (rc == VB_OK) rc = pick_out(r, dest);
    if (rc == VB_OK) r->dest = dest;
    return rc;
}
int frame_launch(vb_renderer *r) {
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaEventRecord(r->frame_ev[0], r->stream));
    int rc = enqueue(r, 0, VB_N_STAGE_IDS - 1, r->dest);
    if (rc == VB_OK) CK(r->err, cudaEventRecord(r->frame_ev[1], r->stream));
    r->frame_timed = rc == VB_OK;
    return rc;
}

int frame_launch_half(vb_renderer *r, int half) {
    CK(r->err, cudaSetDevice(r->device));
    if (half == 0) {
        CK(r->err, cudaEventRecord(r->frame_ev[0], r->stream));
        return enqueue_direct(r, 0, VB_STAGE_ID_FLATTEN, r->dest);
    }
    uint32_t first_half = r->launches;
    int rc = enqueue_direct(r, VB_STAGE_ID_DRAW, VB_N_STAGE_IDS - 1, r->dest);
    r->launches += first_half;
    // (with a host destination enqueue_direct queues the read-back behind fine itself)
    if (rc == VB_OK) CK(r->err, cudaEventRecord(r->frame_ev[1], r->stream));
    r->frame_timed = rc == VB_OK;
    return rc;
}

extern "C" int vb_render_enqueue(vb_renderer *r, const vb_params *p, void *out_device) {
    int rc = frame_prepare(r, p, FrameDest{out_device, nullptr, 1u, 0u, false});
    if (rc) return rc;
    return frame_launch(r);
}

void fill_stats(vb_renderer *r, vb_frame_stats *s) {
    if (!s) return;
    memset(s, 0, sizeof *s);
    memcpy(s, r->cur().h_bump, sizeof(VbBump));
    s->retries = r->retries;
    s->kernel_launches = r->launches;
    s->arena_bytes = arena_bytes(r);
    if (r->timing) {
        for (int i = 0; i < VB_N_STAGE_IDS; i++) cudaEventElapsedTime(&s->stage_ms[i], r->ev[i], r->ev[i + 1]);
        cudaEventElapsedTime(&s->total_ms, r->ev[0], r->ev[VB_N_STAGE_IDS]);
    }
}

void grow_arenas(vb_renderer *r) {
    const VbBump &b = *r->cur().h_bump;
    const VbConfig &c = r->cfg;
    if (b.lines > r->cap_lines) r->cap_lines = grow(b.lines);
    if (b.binning > r->cap_binning) r->cap_binning = grow(b.binning);
    if (b.tile > r->cap_tiles) r->cap_tiles = grow(b.tile);
    if (b.seg_counts > r->cap_seg_counts) r->cap_seg_counts = grow(b.seg_counts);
    if (b.segments > r->cap_segments) r->cap_segments = grow(b.segments);
    if (b.blend > r->cap_blend) r->cap_blend = grow(b.blend);
    uint64_t ptcl_need = (uint64_t)c.width_in_tiles * c.height_in_tiles * VB_PTCL_INITIAL_ALLOC + b.ptcl + VB_PTCL_INCREMENT;
    if (ptcl_need > r->cap_ptcl) r->cap_ptcl = grow((uint32_t)(ptcl_need > 0xf0000000ull ? 0xf0000000ull : ptcl_need));
    if (r->cap_seg_counts < r->cap_lines) r->cap_seg_counts = r->cap_lines;
    if (r->cap_segments < r->cap_seg_counts && (b.failed & VB_STAGE_PATH_COUNT)) r->cap_segments = r->cap_seg_counts;
}

extern "C" int vb_frame_finish(vb_renderer *r, vb_frame_stats *stats) {
    if (!r) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    fill_stats(r, stats);
    return r->cur().h_bump->failed ? VB_E_BUMP_OVERFLOW : VB_OK;
}

int wait_copies(vb_renderer *r, int rc) {
    const cudaError_t e = cudaStreamSynchronize(r->copy_stream);
    if (rc == VB_OK && e != cudaSuccess) {
        r->err = std::string("copy stream: ") + cudaGetErrorString(e);
        return VB_E_CUDA;
    }
    return rc;
}

int render_attempts(vb_renderer *r, const vb_params *p, const FrameDest &d, vb_frame_stats *stats) {
    r->retries = 0;
    for (uint32_t attempt = 0;; attempt++) {
        int rc = frame_prepare(r, p, d);
        if (rc == VB_OK) rc = frame_launch(r);
        if (rc == VB_OK) rc = vb_frame_finish(r, stats);
        if (rc == VB_E_BUMP_OVERFLOW) {
            if (r->xc.enabled) {
                // every attempt of an exchanged frame is a collective step (all GPUs advance their epoch together): grow what
                // overflowed here and let the caller re-issue the frame on every GPU
                grow_arenas(r);
                r->err = "bump overflow in an exchanged frame: re-issue the frame on every GPU";
            } else if (attempt >= r->max_retries) {
                r->err = "bump overflow persisted";
            } else {
                grow_arenas(r);
                r->retries++;
                continue;
            }
        }
        // a re-run after an arena overflow simply copies again
        return d.host_out ? wait_copies(r, rc) : rc;
    }
}

extern "C" int vb_render_resident(vb_renderer *r, const vb_params *p, void *out_device, vb_frame_stats *stats) {
    if (!r || !p) return VB_E_INVALID;
    int rc = drain_stream(r);
    if (rc) return rc;
    return render_attempts(r, p, FrameDest{out_device, nullptr, 1u, 0u, false}, stats);
}

extern "C" int vb_render_uploaded(vb_renderer *r, const vb_params *p, void *out, uint32_t out_is_device, vb_frame_stats *stats) {
    if (!r || !p || !out) return VB_E_INVALID;
    int rc = drain_stream(r);
    if (rc) return rc;
    const FrameDest d{out_is_device ? out : nullptr, out_is_device ? nullptr : out, r->readback_bands, 0u, false};
    return render_attempts(r, p, d, stats);
}

extern "C" int vb_render(vb_renderer *r, const uint8_t *scene, size_t scene_len, const vb_layout *layout, const uint32_t *ramps,
                         uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h, const vb_params *p,
                         void *out, uint32_t out_is_device, vb_frame_stats *stats) {
    if (!r || !p || !out) return VB_E_INVALID;
    int rc = vb_scene_upload(r, scene, scene_len, layout, ramps, ramp_w, ramp_h, atlas, atlas_w, atlas_h);
    if (rc) return rc;
    return vb_render_uploaded(r, p, out, out_is_device, stats);
}

extern "C" int vb_run_stages(vb_renderer *r, const vb_params *p, int first, int last, void *out_device) {
    if (!r || !p || first < 0 || last >= VB_N_STAGE_IDS || first > last) return VB_E_INVALID;
    if (!r->cur().have_scene) return VB_E_NO_SCENE;
    CK(r->err, cudaSetDevice(r->device));
    int rc = prepare(r, p);
    if (rc) return rc;
    FrameDest d{nullptr, nullptr, 1u, 0u, true};
    if (last == VB_STAGE_ID_FINE) {
        d.out_dev = out_device;
        if ((rc = pick_out(r, d))) return rc;
    }
    if ((rc = enqueue(r, first, last, d))) return rc;
    CK(r->err, cudaStreamSynchronize(r->stream));
    return VB_OK;
}

struct NamedBuf {
    const char *name;
    DevBuf *buf;
    size_t bytes;
};
static std::vector<NamedBuf> named(vb_renderer *r) {
    const VbConfig &c = r->cfg;
    const VbLayout &L = r->cur().layout;
    const VbBump &b = *r->cur().h_bump;
    auto mn = [](uint64_t a, uint64_t b2) { return a < b2 ? a : b2; };
    const uint32_t wb = (c.width_in_tiles + 15u) / 16u, hb = (c.height_in_tiles + 15u) / 16u;
    const uint32_t aligned_n_bins = (wb * hb + 255u) & ~255u;
    uint64_t ptcl_words = mn((uint64_t)c.width_in_tiles * c.height_in_tiles * VB_PTCL_INITIAL_ALLOC + b.ptcl, c.ptcl_size);
    return {
        {"tag_monoids", &r->tag_monoids, (size_t)c.n_tag_words * sizeof(VbTagMonoid)},
        {"path_bboxes", &r->path_bboxes, (size_t)L.n_paths * sizeof(VbPathBbox)},
        {"lines", &r->lines, (size_t)mn(b.lines, c.lines_size) * sizeof(VbLineSoup)},
        {"draw_monoids", &r->draw_monoids, (size_t)L.n_draw_objects * sizeof(VbDrawMonoid)},
        {"info_bin_data", &r->info_bin_data, ((size_t)L.bin_data_start + mn(b.binning, c.binning_size)) * 4},
        {"clip_inp", &r->clip_inp, (size_t)L.n_clips * sizeof(VbClipInp)},
        {"clip_bboxes", &r->clip_bboxes, (size_t)L.n_clips * sizeof(VbBbox4)},
        {"draw_bboxes", &r->draw_bboxes, (size_t)L.n_draw_objects * sizeof(VbBbox4)},
        {"bin_headers", &r->bin_headers, (size_t)((L.n_draw_objects + 255u) / 256u) * aligned_n_bins * sizeof(VbBinHeader)},
        {"paths", &r->paths, (size_t)L.n_draw_objects * sizeof(VbPath)},
        {"tiles", &r->tiles, (size_t)mn(b.tile, c.tiles_size) * sizeof(VbTile)},
        {"seg_counts", &r->seg_counts, (size_t)mn(b.seg_counts, c.seg_counts_size) * sizeof(VbSegmentCount)},
        {"segments", &r->segments, (size_t)mn(b.segments, c.segments_size) * sizeof(VbSegment)},
        {"ptcl", &r->ptcl, (size_t)ptcl_words * 4},
        {"blend_spill", &r->blend_spill, (size_t)mn(b.blend, c.blend_size) * 4},
    };
}

extern "C" int vb_debug_download(vb_renderer *r, const char *name, void *dst, size_t cap, size_t *bytes) {
    if (!r || !name) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    if (!strcmp(name, "bump")) {
        if (bytes) *bytes = sizeof(VbBump);
        if (dst && cap >= sizeof(VbBump)) CK(r->err, cudaMemcpy(dst, r->ctl.p, sizeof(VbBump), cudaMemcpyDeviceToHost));
        return VB_OK;
    }
    if (!strcmp(name, "seg_holes")) { // reserved-but-unused segment slots of the last frame (k_coarse.cu)
        if (bytes) *bytes = 4;
        if (dst && cap >= 4) CK(r->err, cudaMemcpy(dst, (const uint32_t *)r->ctl.p + VB_CTL_SEG_HOLES, 4, cudaMemcpyDeviceToHost));
        return VB_OK;
    }
    if (!strcmp(name, "scene") || !strcmp(name, "ramps") || !strcmp(name, "atlas")) { // the uploaded / device-resolved inputs
        const SceneSlot &s = r->cur();
        const DevBuf &b = name[0] == 's' ? s.scene : (name[0] == 'r' ? s.ramps : s.atlas);
        const size_t n = name[0] == 's' ? s.scene_words * 4 : (name[0] == 'r' ? (size_t)s.n_ramps * 512 * 4 : (size_t)s.atlas_w * s.atlas_h * 4);
        if (bytes) *bytes = n;
        const size_t c = n < cap ? n : cap;
        if (dst && c) CK(r->err, cudaMemcpy(dst, b.p, c, cudaMemcpyDeviceToHost));
        return VB_OK;
    }
    if (!strcmp(name, "config")) {
        if (bytes) *bytes = sizeof(VbConfig);
        if (dst && cap >= sizeof(VbConfig)) memcpy(dst, &r->cfg, sizeof(VbConfig));
        return VB_OK;
    }
    for (auto &nb : named(r))
        if (!strcmp(name, nb.name)) {
            if (bytes) *bytes = nb.bytes;
            size_t n = nb.bytes < cap ? nb.bytes : cap;
            if (dst && n) CK(r->err, cudaMemcpy(dst, nb.buf->p, n, cudaMemcpyDeviceToHost));
            return VB_OK;
        }
    return VB_E_UNKNOWN_BUFFER;
}

extern "C" int vb_set_timing(vb_renderer *r, int on) {
    if (!r) return VB_E_INVALID;
    r->timing = on != 0;
    return VB_OK;
}

extern "C" int vb_set_cuda_graph(vb_renderer *r, int on) {
    if (!r) return VB_E_INVALID;
    r->use_graph = on != 0;
    return VB_OK;
}

extern "C" int vb_set_readback_bands(vb_renderer *r, uint32_t n) {
    if (!r || n < 1u || n > 8u) return VB_E_INVALID;
    r->readback_bands = n;
    return VB_OK;
}

extern "C" int vb_set_occlusion_cull(vb_renderer *r, int on) {
    if (!r) return VB_E_INVALID;
    r->occlusion_cull = on ? 1u : 0u;
    return VB_OK;
}

extern "C" int vb_debug_fine_traffic(vb_renderer *r, uint64_t *ptcl_words, uint64_t *segment_refs, uint64_t *fill_cmds) {
    if (!r) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    unsigned long long *d = nullptr, h[3] = {0, 0, 0};
    CK(r->err, cudaMalloc(&d, sizeof h));
    CK(r->err, cudaMemset(d, 0, sizeof h));
    uint32_t n = r->cfg.width_in_tiles * (r->cfg.win_ty1 - r->cfg.win_ty0);
    if (n) k_ptcl_stats<<<(n + 127) / 128, 128, 0, r->stream>>>(r->cfg, (const uint32_t *)r->ptcl.p,
                                                                r->occlusion_cull ? (const uint32_t *)r->tile_start.p : nullptr, d);
    CK(r->err, cudaStreamSynchronize(r->stream));
    CK(r->err, cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost));
    cudaFree(d);
    if (ptcl_words) *ptcl_words = h[0];
    if (segment_refs) *segment_refs = h[1];
    if (fill_cmds) *fill_cmds = h[2];
    return VB_OK;
}

extern "C" int vb_debug_upload(vb_renderer *r, const char *name, const void *src, size_t bytes) {
    if (!r || !name || !src) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    if (!strcmp(name, "lines")) {
        uint32_t n = (uint32_t)(bytes / sizeof(VbLineSoup));
        if (n > r->cap_lines) {
            r->cap_lines = grow(n);
            int rc = ensure(r, r->lines, (size_t)r->cap_lines * sizeof(VbLineSoup));
            if (rc) return rc;
        }
        CK(r->err, cudaMemcpy(r->lines.p, src, (size_t)n * sizeof(VbLineSoup), cudaMemcpyHostToDevice));
        VbBump *bump = (VbBump *)r->ctl.p;
        CK(r->err, cudaMemcpy(&bump->lines, &n, 4, cudaMemcpyHostToDevice));
        r->cur().h_bump->lines = n;
        return VB_OK;
    }
    if (!strcmp(name, "path_bboxes")) {
        if (bytes > r->path_bboxes.cap) return VB_E_INVALID;
        CK(r->err, cudaMemcpy(r->path_bboxes.p, src, bytes, cudaMemcpyHostToDevice));
        return VB_OK;
    }
    return VB_E_UNKNOWN_BUFFER;
}


extern "C" float vb_last_frame_ms(vb_renderer *r) {
    if (!r || !r->frame_timed) return 0.0f;
    cudaSetDevice(r->device);
    float ms = 0.0f;
    if (cudaEventSynchronize(r->frame_ev[1]) != cudaSuccess || cudaEventElapsedTime(&ms, r->frame_ev[0], r->frame_ev[1]) != cudaSuccess) {
        cudaGetLastError();
        return 0.0f;
    }
    return ms;
}

// ---- CUDA IPC helpers (one process per GPU: the frame buffer of rank 0 mapped into the other ranks) ----------------------
extern "C" int vb_frame_alloc(vb_renderer *r, size_t bytes, void **device_ptr) {
    if (!r || !device_ptr || !bytes) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaMalloc(device_ptr, bytes));
    return VB_OK;
}
extern "C" int vb_frame_free(vb_renderer *r, void *device_ptr) {
    if (!r) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    if (device_ptr) CK(r->err, cudaFree(device_ptr));
    return VB_OK;
}
extern "C" int vb_ipc_export(vb_renderer *r, void *device_ptr, uint8_t handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!r || !device_ptr || !handle) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    cudaIpcMemHandle_t h;
    CK(r->err, cudaIpcGetMemHandle(&h, device_ptr));
    memcpy(handle, &h, 64);
    return VB_OK;
}
extern "C" int vb_ipc_open(vb_renderer *r, const uint8_t handle[64], void **device_ptr) {
    if (!r || !handle || !device_ptr) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CK(r->err, cudaIpcOpenMemHandle(device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return VB_OK;
}
extern "C" int vb_ipc_close(vb_renderer *r, void *device_ptr) {
    if (!r || !device_ptr) return VB_E_INVALID;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    CK(r->err, cudaIpcCloseMemHandle(device_ptr));
    return VB_OK;
}


// ---- Resolver::resolve on the device (resolve.rs:183-399): see include/vello_b200.h and k_resolve.cu ---------------------------
extern "C" int vb_scene_upload_streams(vb_renderer *r, const vb_encoding_streams *e, vb_layout *layout_out) {
    if (!r || !e) return VB_E_INVALID;
    if ((e->n_path_tags && !e->path_tags) || (e->n_path_data && !e->path_data) || (e->n_draw_tags && !e->draw_tags) ||
        (e->n_draw_data && !e->draw_data) || (e->n_transforms && !e->transforms) || (e->n_styles && !e->styles) ||
        (e->n_ramp_patches && !e->ramp_patches) || (e->n_image_patches && !e->image_patches))
        return VB_E_INVALID;
    int rc = drain_stream(r);
    if (rc) return rc;
    CK(r->err, cudaSetDevice(r->device));
    cudaStream_t st = r->stream;
    SceneSlot &sl = r->cur();
    struct Patch { uint32_t word, value; };
    struct Ramp { uint32_t first_stop, n_stops, premul, pad; };
    std::vector<Patch> patches;
    std::vector<Ramp> ramps;
    std::vector<vb_ramp_stop> stops;
    std::vector<const vb_ramp_patch *> ramp_of;
    // layout: sizes only (resolve.rs:107-154)
    VbLayout L;
    memset(&L, 0, sizeof L);
    L.n_paths = e->n_paths;
    L.n_clips = e->n_clips;
    L.n_draw_objects = e->n_paths;
    const uint32_t n_tags = e->n_path_tags + e->n_open_clips;
    const uint32_t padded = (n_tags + 1023u) & ~1023u; // 4 * PATH_REDUCE_WG bytes (resolve.rs:625, config.rs:237)
    uint32_t off = padded / 4u;
    L.path_tag_base = 0;
    L.path_data_base = off; off += e->n_path_data;
    L.draw_tag_base = off; off += e->n_draw_tags + e->n_open_clips;
    L.draw_data_base = off; off += e->n_draw_data;
    L.transform_base = off; off += e->n_transforms * 6u;
    L.style_base = off; off += e->n_styles * 2u;
    const size_t total_words = off;
    uint32_t info = 0;
    for (uint32_t i = 0; i < e->n_draw_tags; i++) info += (e->draw_tags[i] >> 6) & 0xFu;
    L.bin_data_start = info;
    // late-bound gradient ramps, de-duplicated by (stops, interpolation space) as the ramp cache does
    for (uint32_t i = 0; i < e->n_ramp_patches; i++) {
        const vb_ramp_patch &p = e->ramp_patches[i];
        if (!p.n_stops || !p.stops || p.draw_data_offset >= e->n_draw_data) return VB_E_INVALID;
        uint32_t rid = (uint32_t)ramp_of.size();
        for (uint32_t k = 0; k < ramp_of.size(); k++) {
            const vb_ramp_patch &q = *ramp_of[k];
            if ((q.premul_interp != 0u) == (p.premul_interp != 0u) && q.n_stops == p.n_stops &&
                memcmp(q.stops, p.stops, sizeof(vb_ramp_stop) * p.n_stops) == 0) { rid = k; break; }
        }
        if (rid == ramp_of.size()) {
            ramp_of.push_back(&p);
            ramps.push_back(Ramp{(uint32_t)stops.size(), p.n_stops, p.premul_interp ? 1u : 0u, 0u});
            stops.insert(stops.end(), p.stops, p.stops + p.n_stops);
        }
        patches.push_back(Patch{L.draw_data_base + p.draw_data_offset, (rid << 2) | p.extend});
    }
    // late-bound images: shelf placement (ours; only the (x, y) written into the draw data matters to the pipeline)
    struct Placed { const uint8_t *key; uint32_t w, h, x, y; };
    std::vector<Placed> placed;
    uint32_t atlas_w = 1, x = 0, y = 0, shelf_h = 0;
    const uint32_t MAXW = 2048;
    for (uint32_t i = 0; i < e->n_image_patches; i++) {
        const vb_image_patch &im = e->image_patches[i];
        if (im.draw_data_offset >= e->n_draw_data) return VB_E_INVALID;
        const Placed *hit = nullptr;
        for (const Placed &q : placed)
            if (q.key == im.pixels && q.w == im.width && q.h == im.height) { hit = &q; break; }
        uint32_t px, py;
        if (!hit) {
            if (x + im.width > MAXW) { y += shelf_h; x = 0; shelf_h = 0; }
            placed.push_back(Placed{im.pixels, im.width, im.height, x, y});
            px = x; py = y;
            x += im.width;
            if (im.height > shelf_h) shelf_h = im.height;
            if (x > atlas_w) atlas_w = x;
        } else {
            px = hit->x; py = hit->y;
        }
        patches.push_back(Patch{L.draw_data_base + im.draw_data_offset, (px << 16) | py});
    }
    const uint32_t atlas_h = (y + shelf_h) > 1u ? (y + shelf_h) : 1u;

    // the six streams go straight to their places in the packed buffer
    if ((rc = ensure(r, sl.scene, total_words * 4 + 64))) return rc;
    char *base = (char *)sl.scene.p;
    if (e->n_path_tags) CK(r->err, cudaMemcpyAsync(base, e->path_tags, e->n_path_tags, cudaMemcpyHostToDevice, st));
    if (e->n_path_data) CK(r->err, cudaMemcpyAsync(base + (size_t)L.path_data_base * 4, e->path_data, (size_t)e->n_path_data * 4, cudaMemcpyHostToDevice, st));
    if (e->n_draw_tags) CK(r->err, cudaMemcpyAsync(base + (size_t)L.draw_tag_base * 4, e->draw_tags, (size_t)e->n_draw_tags * 4, cudaMemcpyHostToDevice, st));
    if (e->n_draw_data) CK(r->err, cudaMemcpyAsync(base + (size_t)L.draw_data_base * 4, e->draw_data, (size_t)e->n_draw_data * 4, cudaMemcpyHostToDevice, st));
    if (e->n_transforms) CK(r->err, cudaMemcpyAsync(base + (size_t)L.transform_base * 4, e->transforms, (size_t)e->n_transforms * 24, cudaMemcpyHostToDevice, st));
    if (e->n_styles) CK(r->err, cudaMemcpyAsync(base + (size_t)L.style_base * 4, e->styles, (size_t)e->n_styles * 8, cudaMemcpyHostToDevice, st));
    // patches, ramp descriptors and stops in one staging buffer
    const size_t pb = patches.size() * sizeof(Patch), rb = ramps.size() * sizeof(Ramp), sb = stops.size() * sizeof(vb_ramp_stop);
    const size_t o_r = (pb + 15) & ~(size_t)15, o_s = (o_r + rb + 15) & ~(size_t)15;
    if ((rc = ensure(r, r->resolve_tmp, o_s + sb + 16))) return rc;
    char *tmp = (char *)r->resolve_tmp.p;
    if (pb) CK(r->err, cudaMemcpyAsync(tmp, patches.data(), pb, cudaMemcpyHostToDevice, st));
    if (rb) CK(r->err, cudaMemcpyAsync(tmp + o_r, ramps.data(), rb, cudaMemcpyHostToDevice, st));
    if (sb) CK(r->err, cudaMemcpyAsync(tmp + o_s, stops.data(), sb, cudaMemcpyHostToDevice, st));
    vb_launch_resolve_finish((uint32_t *)sl.scene.p, e->n_path_tags, e->n_open_clips, padded, L.draw_tag_base + e->n_draw_tags, tmp,
                             (uint32_t)patches.size(), st);
    sl.n_ramps = (uint32_t)ramps.size();
    if ((rc = ensure(r, sl.ramps, (size_t)sl.n_ramps * 512 * 4))) return rc;
    vb_launch_make_ramps(tmp + o_r, tmp + o_s, sl.n_ramps, (uint32_t *)sl.ramps.p, st);
    sl.atlas_w = atlas_w;
    sl.atlas_h = atlas_h;
    if ((rc = ensure(r, sl.atlas, (size_t)atlas_w * atlas_h * 4))) return rc;
    CK(r->err, cudaMemsetAsync(sl.atlas.p, 0, (size_t)atlas_w * atlas_h * 4, st));
    for (const Placed &q : placed)
        if (q.key && q.w && q.h)
            CK(r->err, cudaMemcpy2DAsync((char *)sl.atlas.p + ((size_t)q.y * atlas_w + q.x) * 4, (size_t)atlas_w * 4, q.key, (size_t)q.w * 4, (size_t)q.w * 4, q.h,
                                 cudaMemcpyHostToDevice, st));
    CK(r->err, cudaGetLastError());
    // the host vectors above are read by the asynchronous copies: they must outlive them
    CK(r->err, cudaStreamSynchronize(st));
    sl.layout = L;
    sl.scene_words = total_words;
    sl.have_scene = true;
    if (layout_out) memcpy(layout_out, &L, sizeof(vb_layout));
    return VB_OK;
}


// ---- multi-GPU exchange set-up (k_exchange.cu) ----------------------------------------------------------------------------
// These entry points only manage the arena and the peer table; an overflowing exchanged frame is grown by render_attempts.
extern "C" int vb_exchange_configure(vb_renderer *r, uint32_t rank, uint32_t world, void **arena, size_t *arena_bytes) {
    if (!r || world < 1u || world > 8u || rank >= world) return VB_E_INVALID;
    const VbLayout &L = r->cur().layout;
    if (!r->cur().have_scene) return VB_E_NO_SCENE;
    CK(r->err, cudaSetDevice(r->device));
    CK(r->err, cudaStreamSynchronize(r->stream));
    vb_renderer::Exchange &x = r->xc;
    x.enabled = false;
    const uint32_t n_tags = (L.path_data_base - L.path_tag_base) * 4u;
    // my outbox holds my share of the lines (+ the ones needed by two stripes): generous and fixed, so that the arena -- which
    // the peers have mapped -- never moves
    const uint64_t cap = (uint64_t)n_tags * 4u / world * 2u + 262144u;
    x.lines_cap = cap > 0x7fffffffull ? 0x7fffffffu : (uint32_t)cap;
    x.n_paths = L.n_paths;
    x.half_bytes = vb_exchange_half_bytes(x.n_paths, x.lines_cap);
    const size_t bytes = 256 + 2 * x.half_bytes;
    int rc = ensure(r, x.arena, bytes);
    if (rc) return rc;
    CK(r->err, cudaMemset(x.arena.p, 0, 256)); // flags and epoch start at 0
    x.rank = rank;
    x.world = world;
    memset(x.peer, 0, sizeof x.peer);
    x.peer[rank] = x.arena.p;
    for (uint32_t i = 0; i <= world; i++) x.rows[i] = 0;
    x.configured = true;
    if (arena) *arena = x.arena.p;
    if (arena_bytes) *arena_bytes = bytes;
    return VB_OK;
}
extern "C" int vb_exchange_attach(vb_renderer *r, uint32_t peer_rank, void *peer_arena) {
    if (!r || !r->xc.configured || peer_rank >= r->xc.world || !peer_arena) return VB_E_INVALID;
    r->xc.peer[peer_rank] = peer_arena;
    return VB_OK;
}
extern "C" int vb_exchange_set_bounds(vb_renderer *r, const uint32_t *tile_rows) {
    if (!r || !r->xc.configured || !tile_rows) return VB_E_INVALID;
    for (uint32_t i = 0; i <= r->xc.world; i++) {
        if (i && tile_rows[i] < tile_rows[i - 1]) return VB_E_INVALID;
        r->xc.rows[i] = tile_rows[i];
    }
    return VB_OK;
}
extern "C" int vb_exchange_enable(vb_renderer *r, int on) {
    if (!r) return VB_E_INVALID;
    if (on) {
        if (!r->xc.configured) return VB_E_INVALID;
        for (uint32_t i = 0; i < r->xc.world; i++)
            if (!r->xc.peer[i]) return VB_E_INVALID;
    }
    r->xc.enabled = on != 0;
    return VB_OK;
}
