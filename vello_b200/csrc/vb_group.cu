// vb_group.cu -- vb_group: one frame on several devices of one box, one host thread. Stripes of tile rows per renderer,
// rebalanced from the device times of the last frame; optionally flatten sharded by tag range with the lines exchanged
// through peer memory (k_exchange.cu).
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "vb_internal.h"

struct vb_group {
    std::vector<vb_renderer *> subs;
    std::vector<int> devices;
    std::vector<uint32_t> bounds;   // tile-row boundaries, subs.size() + 1 entries
    std::vector<float> ms;          // device time of the last frame per renderer
    std::vector<char> peer_ok;      // renderer i can store into device 0's memory
    void *frame = nullptr;          // assembled frame on devices[0]
    size_t frame_cap = 0;
    uint32_t bounds_h = 0;          // height in tiles the boundaries were made for
    bool balancing = true;
    bool exchange = false;          // flatten sharded by tag range, lines exchanged through peer memory (k_exchange.cu)
    bool shared_device = false;     // two renderers on one GPU (tests)
    std::string err;
};

// Map device `to`'s memory into device `from` (NVLink / NVSwitch). Leaves `from` current.
static cudaError_t enable_peer(int from, int to) {
    int can = 0;
    cudaSetDevice(from);
    cudaError_t e = cudaDeviceCanAccessPeer(&can, from, to);
    if (e == cudaSuccess && !can) return cudaErrorPeerAccessUnsupported;
    if (e == cudaSuccess) e = cudaDeviceEnablePeerAccess(to, 0);
    cudaGetLastError();
    return e == cudaErrorPeerAccessAlreadyEnabled ? cudaSuccess : e;
}

extern "C" int vb_group_new(const int32_t *devices, uint32_t n, const vb_options *opt, vb_group **out) {
    if (!devices || !n || n > 64 || !out) return VB_E_INVALID;
    vb_group *g = new vb_group();
    for (uint32_t i = 0; i < n; i++) {
        vb_options o{};
        if (opt) o = *opt;
        o.device = devices[i];
        vb_renderer *r = nullptr;
        int rc = vb_renderer_new(&o, &r);
        if (rc) {
            vb_group_free(g);
            return rc;
        }
        g->subs.push_back(r);
        g->devices.push_back(devices[i]);
        // stores of `fine` on device i land in device 0's frame buffer through peer mapping
        g->peer_ok.push_back(devices[i] == devices[0] || enable_peer(devices[i], devices[0]) == cudaSuccess);
    }
    g->ms.assign(n, 0.0f);
    *out = g;
    return VB_OK;
}

extern "C" void vb_group_free(vb_group *g) {
    if (!g) return;
    for (vb_renderer *r : g->subs) vb_renderer_free(r);
    if (!g->devices.empty()) cudaSetDevice(g->devices[0]);
    if (g->frame) cudaFree(g->frame);
    delete g;
}
extern "C" uint32_t vb_group_size(const vb_group *g) { return g ? (uint32_t)g->subs.size() : 0u; }
extern "C" vb_renderer *vb_group_renderer(vb_group *g, uint32_t i) { return g && i < g->subs.size() ? g->subs[i] : nullptr; }
extern "C" const char *vb_group_last_error(vb_group *g) { return g ? g->err.c_str() : ""; }
extern "C" int vb_group_set_balancing(vb_group *g, int on) {
    if (!g) return VB_E_INVALID;
    g->balancing = on != 0;
    return VB_OK;
}
extern "C" void *vb_group_frame(vb_group *g, size_t *bytes) {
    if (!g) return nullptr;
    if (bytes) *bytes = g->frame_cap;
    return g->frame;
}
extern "C" int vb_group_stripes(vb_group *g, uint32_t *boundaries, float *device_ms) {
    if (!g) return VB_E_INVALID;
    if (boundaries)
        for (size_t i = 0; i < g->bounds.size(); i++) boundaries[i] = g->bounds[i];
    if (device_ms)
        for (size_t i = 0; i < g->ms.size(); i++) device_ms[i] = g->ms[i];
    return VB_OK;
}

// Move the stripe boundaries so that the device times of the last frame would have been equal, assuming the cost of a stripe is
// spread evenly over its tile rows (piecewise-linear cumulative cost); damped, every stripe keeps at least one tile row.
static void group_rebalance(vb_group *g, uint32_t ht) {
    const size_t n = g->subs.size();
    if (g->bounds.size() != n + 1 || g->bounds_h != ht) {
        g->bounds.assign(n + 1, 0u);
        for (size_t i = 0; i <= n; i++) g->bounds[i] = (uint32_t)((uint64_t)ht * i / n);
        g->bounds_h = ht;
        return;
    }
    if (!g->balancing || n < 2 || ht < n) return;
    double total = 0.0, lo = 1e30, hi = 0.0;
    for (size_t i = 0; i < n; i++) {
        if (!(g->ms[i] > 0.0f)) return; // no measurement yet
        total += g->ms[i];
        lo = std::min<double>(lo, g->ms[i]);
        hi = std::max<double>(hi, g->ms[i]);
    }
    if (hi - lo < 0.06 * (total / n)) return; // balanced within noise: keep the stripes (and the captured graphs)
    std::vector<uint32_t> nb(n + 1, 0u);
    nb[n] = ht;
    size_t seg = 0;
    double acc = 0.0; // cost of the stripes before `seg`
    for (size_t k = 1; k < n; k++) {
        const double want = total * k / n;
        while (seg + 1 < n && acc + g->ms[seg] < want) acc += g->ms[seg++];
        const double rows = (double)(g->bounds[seg + 1] - g->bounds[seg]);
        const double frac = g->ms[seg] > 0.0f ? (want - acc) / g->ms[seg] : 0.0;
        const double ideal = g->bounds[seg] + rows * frac;
        const double damped = 0.5 * g->bounds[k] + 0.5 * ideal;
        nb[k] = (uint32_t)(damped + 0.5);
    }
    for (size_t k = 1; k < n; k++) { // monotone, at least one row each
        if (nb[k] < nb[k - 1] + 1u) nb[k] = nb[k - 1] + 1u;
    }
    for (size_t k = n - 1; k >= 1; k--) {
        if (nb[k] > nb[k + 1] - 1u) nb[k] = nb[k + 1] - 1u;
    }
    g->bounds = nb;
}

// (re)build the exchange arenas for the uploaded scene and introduce the renderers to each other
static int group_setup_exchange(vb_group *g) {
    const uint32_t n = (uint32_t)g->subs.size();
    if (n > 8u) return VB_E_INVALID;
    std::vector<void *> arenas(n, nullptr);
    for (uint32_t i = 0; i < n; i++) {
        int rc = vb_exchange_configure(g->subs[i], i, n, &arenas[i], nullptr);
        if (rc) {
            g->err = g->subs[i]->err;
            return rc;
        }
    }
    for (uint32_t i = 0; i < n; i++) {
        for (uint32_t j = 0; j < n; j++) {
            if (i == j) continue;
            if (g->devices[i] != g->devices[j]) { // every GPU reads every other GPU's arena
                const cudaError_t e = enable_peer(g->devices[i], g->devices[j]);
                if (e != cudaSuccess) {
                    g->err = std::string("exchange needs peer access between all devices of the group: ") + cudaGetErrorString(e);
                    return VB_E_CUDA;
                }
            }
            int rc = vb_exchange_attach(g->subs[i], j, arenas[j]);
            if (rc) return rc;
        }
    }
    bool shared_device = false;
    for (uint32_t i = 0; i < n; i++)
        for (uint32_t j = i + 1; j < n; j++) shared_device = shared_device || g->devices[i] == g->devices[j];
    g->shared_device = shared_device;
    for (uint32_t i = 0; i < n; i++) {
        int rc = vb_exchange_enable(g->subs[i], 1);
        if (rc) return rc;
        // renderers that share a GPU (tests): no graph (re-)instantiation while a peer's wait kernel is resident on that GPU
        if (shared_device) g->subs[i]->use_graph = false;
    }
    return VB_OK;
}

extern "C" int vb_group_set_exchange(vb_group *g, int on) {
    if (!g) return VB_E_INVALID;
    g->exchange = on != 0;
    if (!g->exchange) {
        for (vb_renderer *r : g->subs) vb_exchange_enable(r, 0);
        return VB_OK;
    }
    for (vb_renderer *r : g->subs)
        if (!r->cur().have_scene) return VB_OK; // arenas are built by the next vb_group_scene_upload
    return group_setup_exchange(g);
}

extern "C" int vb_group_scene_upload(vb_group *g, const uint8_t *scene, size_t scene_len, const vb_layout *layout, const uint32_t *ramps,
                                     uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h) {
    if (!g) return VB_E_INVALID;
    // every device pulls the scene over its own PCIe link (asynchronous per renderer, so the copies run side by side)
    for (vb_renderer *r : g->subs) {
        int rc = vb_scene_upload(r, scene, scene_len, layout, ramps, ramp_w, ramp_h, atlas, atlas_w, atlas_h);
        if (rc) {
            g->err = r->err;
            return rc;
        }
    }
    return g->exchange ? group_setup_exchange(g) : VB_OK;
}

// out: nullptr (group frame), a device pointer on devices[0], or (host_out) a host pointer
static int group_render(vb_group *g, const vb_params *p, void *out_device, void *host_out, vb_frame_stats *stats) {
    if (!g || !p || p->bin_row1 > p->bin_row0 || p->tile_row1 > p->tile_row0) return VB_E_INVALID;
    const size_t n = g->subs.size();
    const uint32_t ht = (p->height + 15u) / 16u;
    if (g->exchange && ht < n) {
        g->err = "exchange needs at least one tile row per device";
        return VB_E_INVALID;
    }
    group_rebalance(g, ht);
    const size_t pitch = (size_t)p->width * 4u;
    void *frame = out_device;
    if (!host_out && !frame) {
        const size_t need = pitch * p->height;
        if (g->frame_cap < need) {
            CK(g->err, cudaSetDevice(g->devices[0]));
            if (g->frame) CK(g->err, cudaFree(g->frame));
            g->frame = nullptr;
            g->frame_cap = 0;
            CK(g->err, cudaMalloc(&g->frame, need));
            g->frame_cap = need;
        }
        frame = g->frame;
    }
    const bool halves = g->exchange && g->shared_device;
    const bool late_copy = host_out != nullptr && g->exchange; // without the exchange every frame queues its own read-back
    // Renderer i's destination. Device: straight into the frame on devices[0] when peer-mapped; otherwise (and for a host
    // destination) the renderer's own target. Host without late_copy: the frame copies its stripe itself, in one band.
    auto dest = [&](size_t i) {
        const size_t off = (size_t)g->bounds[i] * 16u * pitch;
        return FrameDest{(!host_out && g->peer_ok[i]) ? (char *)frame + off : nullptr, (host_out && !late_copy) ? (char *)host_out + off : nullptr,
                         1u, 0u, false};
    };
    // enqueue every device's stripe, then complete them (one host thread; the devices run side by side)
    std::vector<vb_params> ps(n, *p);
    int result = VB_OK;
    for (uint32_t attempt = 0;; attempt++) {
        if (g->exchange)
            for (vb_renderer *r : g->subs) vb_exchange_set_bounds(r, g->bounds.data());
        // phases: 0 = configs and arenas of every renderer, 1 (and 2) = the launches, last = the read-backs of a host
        // destination. A copy into pageable host memory blocks the host until it is done, so it must not be issued before
        // every renderer's frame has been launched (with the exchange on, a frame waits for its peers).
        const int n_launch = halves ? 2 : 1;
        for (int phase = 0; phase < 1 + n_launch + (late_copy ? 1 : 0); phase++) {
            for (size_t i = 0; i < n; i++) {
                vb_renderer *r = g->subs[i];
                ps[i].tile_row0 = g->bounds[i];
                ps[i].tile_row1 = g->bounds[i + 1];
                if (ps[i].tile_row1 <= ps[i].tile_row0) continue; // more devices than tile rows (never with the exchange on)
                const size_t row0 = (size_t)g->bounds[i] * 16u;
                int rc = VB_OK;
                if (phase == 0) rc = frame_prepare(r, &ps[i], dest(i));
                else if (phase <= n_launch) rc = halves ? frame_launch_half(r, phase - 1) : frame_launch(r);
                else {
                    const size_t h1 = std::min<size_t>((size_t)g->bounds[i + 1] * 16u, p->height);
                    cudaSetDevice(r->device);
                    if (h1 > row0 && cudaMemcpyAsync((char *)host_out + row0 * pitch, r->dest.out_dev, (h1 - row0) * pitch, cudaMemcpyDeviceToHost, r->stream) != cudaSuccess)
                        rc = VB_E_CUDA;
                }
                if (rc) {
                    g->err = r->err;
                    return rc;
                }
            }
        }
        result = VB_OK;
        bool redo = false;
        for (size_t i = 0; i < n; i++) {
            vb_renderer *r = g->subs[i];
            if (ps[i].tile_row1 <= ps[i].tile_row0) {
                if (stats) memset(&stats[i], 0, sizeof(vb_frame_stats));
                continue;
            }
            const size_t row0 = (size_t)g->bounds[i] * 16u;
            int rc = vb_frame_finish(r, stats ? &stats[i] : nullptr);
            if (rc == VB_E_BUMP_OVERFLOW) {
                if (g->exchange) { // an exchanged frame is re-issued on EVERY device (epochs advance together)
                    grow_arenas(r);
                    redo = true;
                    rc = VB_OK;
                } else {
                    // grow and re-run (first frames); with a host destination the re-run queues its read-back again
                    rc = render_attempts(r, &ps[i], dest(i), stats ? &stats[i] : nullptr);
                }
            }
            g->ms[i] = vb_last_frame_ms(r);
            if (rc == VB_OK && host_out && !late_copy) rc = wait_copies(r, rc);
            if (rc == VB_OK && !host_out && !g->peer_ok[i]) {
                // no peer mapping between these two devices: stage through the renderer's own target
                const size_t h0 = row0, h1 = std::min<size_t>((size_t)g->bounds[i + 1] * 16u, p->height);
                cudaSetDevice(r->device);
                if (h1 > h0 && (cudaMemcpyPeerAsync((char *)frame + row0 * pitch, g->devices[0], r->dest.out_dev, r->device, (h1 - h0) * pitch, r->stream) != cudaSuccess ||
                                cudaStreamSynchronize(r->stream) != cudaSuccess))
                    rc = VB_E_CUDA;
            }
            if (rc && result == VB_OK) {
                result = rc;
                g->err = r->err;
            }
        }
        if (!redo || result != VB_OK) break;
        if (attempt >= 8u) {
            g->err = "bump overflow persisted in an exchanged frame; failed bits per renderer:";
            for (vb_renderer *q : g->subs) g->err += " 0x" + std::to_string(q->cur().h_bump->failed);
            return VB_E_BUMP_OVERFLOW;
        }
    }
    return result;
}

extern "C" int vb_group_render_resident(vb_group *g, const vb_params *p, void *out_device, vb_frame_stats *stats) {
    return group_render(g, p, out_device, nullptr, stats);
}

extern "C" int vb_group_render(vb_group *g, const uint8_t *scene, size_t scene_len, const vb_layout *layout, const uint32_t *ramps,
                               uint32_t ramp_w, uint32_t ramp_h, const uint8_t *atlas, uint32_t atlas_w, uint32_t atlas_h, const vb_params *p,
                               void *out, uint32_t out_is_device, vb_frame_stats *stats) {
    if (!g || !p) return VB_E_INVALID;
    int rc = vb_group_scene_upload(g, scene, scene_len, layout, ramps, ramp_w, ramp_h, atlas, atlas_w, atlas_h);
    if (rc) return rc;
    if (out && !out_is_device) return group_render(g, p, nullptr, out, stats);
    return group_render(g, p, out, nullptr, stats);
}

