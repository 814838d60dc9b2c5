// group.cu — one process, several GPUs, behind the C ABI: the row-strip sharding of SURVEY §8(e) for hosts that are
// not Python (the reference's Rust process owns all its threads; a Rust `impl HeadlessRenderer` cannot call
// torch.distributed).  An aicb_group is one aicb_ctx per device; an aicb_group_scene is the scene replicated on each of
// them.  aicb_group_render_srgb8 cuts the frame into interleaved 16-row strips (strip s -> device s mod n), every
// device's encode_kernel stores its pixels straight into device 0's frame over NVLink (peer access), device 0's stream
// waits for the others' completion events and copies the frame to the caller: compute and delivery are one kernel
// chain per device, there is no collective and no host thread per GPU.
// Replaces the Rayon rows x pixels dispatch of trace_scene_to_image_impl (renderer.rs:516-556) across devices.
#include <cstring>
#include <vector>

#include "internal.h"

static const uint32_t GROUP_STRIP_ROWS = 16;

extern "C" {

void aicb_group_destroy(aicb_group *g) {
    if (!g) return;
    if (!g->ctx.empty()) {
        cudaSetDevice(g->ctx[0]->device);
        if (g->d_frame) cudaFree(g->d_frame);
        if (g->h_stage) cudaFreeHost(g->h_stage);
    }
    for (size_t i = 0; i < g->ctx.size(); i++) {
        cudaSetDevice(g->ctx[i]->device);
        if (g->done[i]) cudaEventDestroy(g->done[i]);
        if (i < g->light_barrier.size() && g->light_barrier[i]) cudaEventDestroy(g->light_barrier[i]);
        aicb_ctx_destroy(g->ctx[i]);
    }
    delete g;
}

aicb_status aicb_group_create(const int *device_ids, int n_devices, aicb_group **out) {
    if (!device_ids || n_devices < 1 || !out) return aicb_fail(AICB_ERR_INVALID, "NULL argument or no devices");
    *out = nullptr;
    aicb_group *g = new aicb_group();
    for (int i = 0; i < n_devices; i++) {
        aicb_ctx *c = nullptr;
        aicb_status st = aicb_ctx_create(device_ids[i], &c);
        if (st != AICB_OK) {
            aicb_group_destroy(g);
            return st;
        }
        g->ctx.push_back(c);
        g->done.push_back(nullptr);
        cudaError_t e = cudaEventCreateWithFlags(&g->done[i], cudaEventDisableTiming);
        if (e != cudaSuccess) {
            aicb_group_destroy(g);
            return aicb_cuda_fail(e, "cudaEventCreate");
        }
    }
    // every device stores into device 0's frame
    const int root = g->ctx[0]->device;
    for (int i = 1; i < n_devices; i++) {
        const int dev = g->ctx[i]->device;
        if (dev == root) continue;
        int can = 0;
        cudaDeviceCanAccessPeer(&can, dev, root);
        if (!can) {
            aicb_group_destroy(g);
            return aicb_fail(AICB_ERR_UNSUPPORTED, "device cannot access the root device's memory (no P2P / NVLink path)");
        }
        cudaSetDevice(dev);
        cudaError_t e = cudaDeviceEnablePeerAccess(root, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        if (e != cudaSuccess) {
            aicb_group_destroy(g);
            return aicb_cuda_fail(e, "cudaDeviceEnablePeerAccess");
        }
    }
    *out = g;
    return AICB_OK;
}

int aicb_group_size(const aicb_group *g) { return g ? (int)g->ctx.size() : 0; }

void aicb_group_scene_destroy(aicb_group_scene *gs) {
    if (!gs) return;
    for (aicb_scene *s : gs->scene) aicb_scene_destroy(s);
    delete gs;
}

aicb_status aicb_group_scene_create(aicb_group *g, const aicb_scene_desc *d, aicb_group_scene **out) {
    if (!g || !d || !out) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    *out = nullptr;
    aicb_group_scene *gs = new aicb_group_scene();
    gs->group = g;
    for (aicb_ctx *c : g->ctx) {   // the scene is replicated (<= ~0.3 GB at 256^3), SURVEY §8(e)
        aicb_scene *s = nullptr;
        aicb_status st = aicb_scene_create(c, d, &s);
        if (st != AICB_OK) {
            aicb_group_scene_destroy(gs);
            return st;
        }
        gs->scene.push_back(s);
    }
    *out = gs;
    return AICB_OK;
}

aicb_status aicb_group_scene_update_cubes(aicb_group_scene *gs, const int32_t (*cubes)[3], const uint16_t *ids,
                                          const uint8_t (*light)[4], size_t n) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    for (aicb_scene *s : gs->scene) {
        aicb_status st = aicb_scene_update_cubes(s, cubes, ids, light, n);
        if (st != AICB_OK) return st;
    }
    return AICB_OK;
}

// Both validate before they change anything, and every replica holds the same state: a call that fails on member 0
// fails there, before any replica changed.
aicb_status aicb_group_scene_update_blocks(aicb_group_scene *gs, const uint16_t *indices, const aicb_block_desc *descs, size_t n) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    for (aicb_scene *s : gs->scene) {
        aicb_status st = aicb_scene_update_blocks(s, indices, descs, n);
        if (st != AICB_OK) return st;
    }
    return AICB_OK;
}

aicb_status aicb_group_scene_upload_light(aicb_group_scene *gs, const uint8_t (*light)[4], size_t n_texels) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    for (aicb_scene *s : gs->scene) {
        aicb_status st = aicb_scene_upload_light(s, light, n_texels);
        if (st != AICB_OK) return st;
    }
    return AICB_OK;
}

aicb_status aicb_group_render_srgb8(aicb_group_scene *gs, const aicb_camera *cam, const aicb_options *opt,
                                    uint8_t (*out)[4], size_t out_len, aicb_render_info *info) {
    if (!gs || !cam || !opt) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    aicb_group *g = gs->group;
    const size_t pixels = (size_t)cam->fb_width * cam->fb_height;
    if (out_len != pixels) return aicb_fail(AICB_ERR_INVALID, "Viewport size does not match output buffer length");
    if (pixels && !out) return aicb_fail(AICB_ERR_INVALID, "out is NULL");
    const uint32_t n = (uint32_t)g->ctx.size();
    aicb_ctx *root = g->ctx[0];
    CU(cudaSetDevice(root->device));
    if (g->frame_pixels < pixels) {
        if (g->d_frame) cudaFree(g->d_frame);
        g->d_frame = nullptr;
        g->frame_pixels = 0;
        CU(cudaMalloc(&g->d_frame, pixels * 4 + 16));
        g->frame_pixels = pixels;
    }
    for (int attempt = 0;; attempt++) {
        // every device renders its strips into the root's frame; nothing here waits for a GPU
        for (uint32_t i = 0; i < n; i++) {
            aicb_shard sh;
            sh.strip_rows = GROUP_STRIP_ROWS;
            sh.index = i;
            sh.count = n;
            aicb_status st = aicb_render_srgb8_device_frame(gs->scene[i], cam, opt, &sh, g->d_frame, pixels, nullptr);
            if (st != AICB_OK) return st;
            CU(cudaSetDevice(g->ctx[i]->device));
            CU(cudaEventRecord(g->done[i], g->ctx[i]->stream));
        }
        CU(cudaSetDevice(root->device));
        for (uint32_t i = 1; i < n; i++) CU(cudaStreamWaitEvent(root->stream, g->done[i], 0));
        if (pixels) CU(cudaMemcpyAsync(out, g->d_frame, pixels * 4, cudaMemcpyDeviceToHost, root->stream));
        CU(cudaStreamSynchronize(root->stream));
        // RaytraceInfo: summed over the shards (renderer.rs:555); the frame took as long as its slowest device
        aicb_render_info total;
        std::memset(&total, 0, sizeof total);
        bool retry = false;
        for (uint32_t i = 0; i < n; i++) {
            aicb_render_info one;
            aicb_status st = aicb_render_finish(gs->scene[i], &one);
            if (st == AICB_ERR_RETRY) { retry = true; continue; }
            if (st != AICB_OK) return st;
            total.cubes_traced += one.cubes_traced;
            total.rays += one.rays;
            total.algorithmic_bytes += one.algorithmic_bytes;
            for (int k = 0; k < 6; k++) total.counters[k] += one.counters[k];
            total.kernel_ms = one.kernel_ms > total.kernel_ms ? one.kernel_ms : total.kernel_ms;
            for (int k = 0; k < 4; k++) total.stage_ms[k] = one.stage_ms[k] > total.stage_ms[k] ? one.stage_ms[k] : total.stage_ms[k];
            total.flaws |= one.flaws;
        }
        if (!retry) {
            if (info) *info = total;
            return AICB_OK;
        }
        if (attempt >= 5) return aicb_fail(AICB_ERR_OOM, "hit stream capacity exhausted");
    }
}

}  // extern "C"
