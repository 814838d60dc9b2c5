// internal.h — objects behind the opaque handles of include/aicb200.h (shared by aicb200.cu and light.cu).
#pragma once
#include <mutex>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "trace_kernel.cuh"

aicb_status aicb_fail(aicb_status st, const std::string &msg);
aicb_status aicb_cuda_fail(cudaError_t e, const char *what);
#define CU(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return aicb_cuda_fail(e__, #call); \
    } while (0)

struct LightNodePre;    // light_kernel.cuh
struct LightChain;      // light_kernel.cuh
struct LightBlockDev;   // light_kernel.cuh

struct aicb_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_k[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // AICB_PROFILE_KERNELS
    bool profile_kernels = false;
    bool dependent_launch = true; // programmatic dependent launch between the kernels of a frame (AICB_PDL=0 disables)
    bool stage_timing = true;    // record the per-kernel events of a frame (aicb_render_info::stage_ms)
    void *h_delta = nullptr, *d_delta = nullptr;  // staging of aicb_scene_update_cubes batches (pinned / device)
    size_t h_delta_bytes = 0;
    cudaEvent_t ev_delta = nullptr;
    void *d_debug = nullptr;
    uint32_t debug_warps = 0;
    unsigned int *d_tile_counter = nullptr;
    unsigned long long *d_counters = nullptr;
    float *d_lut = nullptr;
    // staging output buffers (grown on demand)
    void *d_out = nullptr;
    size_t d_out_bytes = 0;
    void *d_aux = nullptr;
    size_t d_aux_bytes = 0;
    // per-task streams between gen -> trace -> encode (trace_kernel.cuh)
    void *d_rays = nullptr;
    size_t d_rays_bytes = 0;
    void *d_task_cb = nullptr;   // TaskOut per task
    size_t d_task_cb_bytes = 0;
    void *d_hits = nullptr;      // HitRecord stream (march -> shade -> encode)
    size_t d_hits_bytes = 0;
    void *d_contrib = nullptr;   // ShadedHit per hit (shade -> encode)
    size_t d_contrib_bytes = 0;
    void *d_bin_list = nullptr;  // task ids of the rays that enter the space, per chord-length bin
    size_t d_bin_list_bytes = 0;
    // LightingOption::Bounce: the same streams for the secondary rays of a chunk, and the per-task bounce state
    void *d_rays2 = nullptr, *d_task_cb2 = nullptr, *d_hits2 = nullptr, *d_contrib2 = nullptr, *d_bin_list2 = nullptr;
    size_t d_rays2_bytes = 0, d_task_cb2_bytes = 0, d_hits2_bytes = 0, d_contrib2_bytes = 0, d_bin_list2_bytes = 0;
    void *d_bounce = nullptr;    // per task: secondary ray (48 B), RNG state (32 B), Rgb sum + steps (16 B), request (4 B)
    size_t d_bounce_bytes = 0;
    uint32_t hits_per_task = 8;  // capacity of the hit stream per ray; raised x4 when a frame overflows it,
    uint32_t shallow_frames = 0; //   lowered again after 16 frames in a row that needed a small fraction of it
    void *h_stage = nullptr;     // pinned staging of frames whose destination is pageable host memory
    size_t h_stage_bytes = 0;
    // the frame whose per-frame scratch (streams, counters, events) is in use
    bool frame_in_flight = false;
    cudaStream_t last_stream = nullptr;
    struct aicb_scene *last_scene = nullptr;
    void *d_task_aux = nullptr;
    size_t d_task_aux_bytes = 0;
    // light propagation: the static ray chart (space/light/chart), built and uploaded on first use
    LightNodePre *d_chart_pre = nullptr;   // the chart in depth-first preorder (the overflow walk)
    uint32_t chart_nodes = 0;
    LightChain *d_chains = nullptr;         // the chart as chains, the per-node cube offsets, the Euler tour of the chain tree
    uchar4 *d_node_rel = nullptr;
    uint16_t *d_euler = nullptr;
    uint32_t n_chains = 0, n_euler = 0;
    float4 *d_term_scratch = nullptr;       // term slots of the chain walk, one set per resident warp
    uint32_t chain_walk_blocks = 0;
    std::mutex mu;
};

struct aicb_scene {
    aicb_ctx *ctx = nullptr;
    aicb::DeviceScene ds{};
    std::vector<uint8_t> block_kind;   // host copy, for update_cubes
    size_t volume = 0;
    uint64_t device_bytes = 0;
    void *d_cells = nullptr;
    uint32_t *d_light = nullptr;
    aicb::BlockRec *d_blocks = nullptr;
    uint16_t *d_bricks = nullptr;
    float4 *d_palette = nullptr;
    float2 *d_pal_tab = nullptr;   // per palette entry: {alpha, log2(1 - alpha) bound} (marching kernel)
    float4 *d_blk_tab = nullptr;   // per block id: that pair and the palette entry of single-voxel blocks
    size_t n_bricks = 0, n_palette = 0;   // elements in d_bricks / d_palette (aicb_scene_update_blocks appends)
    // state of the last asynchronous render
    bool pending = false;
    uint64_t pending_rays = 0;
    uint64_t pending_pixels = 0;
    uint32_t pending_out_bytes_per_pixel = 0;
    // ---- light propagation state (light.cu) ----
    std::vector<uint16_t> h_ids;            // host mirror of Space::contents (edits are applied in order on the host)
    std::vector<uint32_t> h_block_light;    // per block: bits 0-5 opaque faces, 6 all-opaque, 7 visible, 8 has emission
    LightBlockDev *d_light_blocks = nullptr;
    uint8_t *d_pending = nullptr;           // per cube: queued priority (0 = not queued) — LightUpdateQueue
    uint32_t *d_list = nullptr;             // work list of one round (cube indices)
    uint32_t *d_new_light = nullptr;        // computed texels of one round
    uint8_t *d_diff = nullptr;              // difference_priority of one round
    uint32_t *d_scalars = nullptr;          // the propagation's counters (light_kernel.cuh: LightScalar)
    float4 *d_sky_term = nullptr;           // per chart node: the sky light its bundle collects (end_of_ray), for this scene's sky
    uint32_t *d_changed = nullptr;          // list positions whose cube changed by more than one unit this round
    uint32_t *d_tile_max = nullptr;         // per LIGHT_TILE cubes: upper bound of the queued priorities
    uint32_t *d_tile_count = nullptr;       // per LIGHT_TILE cubes: a count and its exclusive scan over the tiles (capped
    uint32_t *d_tile_off = nullptr;         //   rounds of aicb_light_step, aicb_light_take_changes)
    uint32_t light_max_distance = 0;
    uint64_t light_stats[4] = {0, 0, 0, 0};  // last propagation: cube updates, chart node visits, rounds queued, device microseconds
    double light_us_per_update = 0.1;       // running estimate of device microseconds per cube update (aicb_light_step)
    uint32_t *d_light_base = nullptr;       // change tracking: the light as of the last take (nullptr: not tracking)
    uint32_t *d_changes = nullptr;          // records of a take: changes_cap cubes (3 x int32), then changes_cap texels
    size_t changes_cap = 0;
};

// One process, several GPUs (group.cu renders, light.cu propagates light): one aicb_ctx per member, the scene
// replicated on each of them.
struct aicb_group {
    std::vector<aicb_ctx *> ctx;
    std::vector<cudaEvent_t> done;   // per device: its strips of the current frame are in device 0's frame
    void *d_frame = nullptr;         // on device 0
    size_t frame_pixels = 0;
    void *h_stage = nullptr;         // pinned staging for pageable destinations
    size_t h_stage_bytes = 0;
    // group light propagation (light.cu), set up on its first call
    bool light_peers_ready = false;          // peer access (with native atomics) between every pair of member devices
    std::vector<cudaEvent_t> light_barrier;  // per member: its arrival at a round's barrier (member 0's: the release)
};

struct aicb_group_scene {
    aicb_group *group = nullptr;
    std::vector<aicb_scene *> scene;
    uint64_t light_stats[4] = {0, 0, 0, 0};  // last group propagation: updates and visits summed, rounds, slowest member's time
};
