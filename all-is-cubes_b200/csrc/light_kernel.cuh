// light_kernel.cuh — device code of the secondary path: all-is-cubes' light propagation
// (all-is-cubes/src/space/light/updater.rs) as batched relaxation kernels.
//
// Design: the reference pops one cube at a time from a priority queue (32 at a time with threads,
// updater.rs:211-252) and recomputes its light by a depth-first walk over a static ray chart
// (walk_ray_tree, updater.rs:427-529).  Here the queue is a per-cube priority byte in HBM with a per-tile
// maximum beside it; one round = the cubes within a band of the highest queued priority:
// gather (tiles in index order, so the list is spatially sorted) -> compute -> apply (store, fill uninitialised
// neighbours) -> mark (re-queue the dependencies of the cubes that changed).
//
// compute / mark, the chain walk (compute_light_chains, below): ONE WARP PER CUBE, 32 CHAINS OF THE CHART AT A TIME.
// 99 % of the chart's nodes have exactly one child with bit-identical weights, so the tree is 1043 chains joined at 441
// branching nodes.  Lanes take ready chains from a per-warp queue and walk them node by node; the terms the reference
// adds up in depth-first order are written to per-chain slots and added afterwards in the Euler tour of the chain
// tree, which is that order — compute_light on a given field stays bit-identical to the reference.
//
// The overflow walk (compute_light_lockstep) computes the cubes whose walk needs more term slots than a chain holds:
// one warp steps through the chart in preorder for 32 cubes — node record, depth and weights are warp-uniform — and a
// lane takes part in a node iff its own walk would enter it; a subtree that no lane enters is skipped.  Every lane's
// f32 additions happen in place, in the reference's order, so it needs no term slots.
// The relaxation order differs from the reference's (batch = a priority band), which the reference leaves unspecified
// (queue.rs:226-246) — parity contract SURVEY §8(a) L4.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "trace_kernel.cuh"

// FlatNode (chart/shared.rs:13-25): 6 weights + 6 child indices (0 = none); root = 0.
struct LightChartNode {
    float w[6];
    uint32_t child[6];
};

// The same chart in depth-first preorder (children in Face6 order NX,NY,NZ,PX,PY,PZ, updater.rs:500), 32 bytes.
struct LightNodePre {
    float w[6];
    int8_t rel[3];        // the node's cube relative to the origin cube
    uint8_t depth;
    uint32_t end_dir;     // index one past the node's last descendant | direction (0..5) of the step from its parent << 29
};
static_assert(sizeof(LightNodePre) == 32, "LightNodePre must be 32 bytes");

// The EvaluatedBlock members light reads (evaluated.rs:189-272), 128 bytes.
struct LightBlockDev {
    float face_color[7][4];  // Within, NX..PZ (face7_color)
    float emission[3];
    uint32_t flags;          // bits 0-5 opaque[NX..PZ], 6 all opaque, 7 visible_or_animated, 8 emission != 0
};
static_assert(sizeof(LightBlockDev) == 128, "LightBlockDev must be 128 bytes");

// The chart as chains.  99 % of the chart's nodes have exactly one child, with bit-identical weights (they carry the
// same rays): the tree is 1043 chains (maximal single-child paths; 602 of them end in leaves) joined at 441 branching
// nodes, 8 chain levels deep.  A chain's nodes are consecutive in preorder.  One record per chain, numbered breadth
// first so that the children of a chain are consecutive; 48 bytes.
struct LightChain {
    float w[6];             // the weights of every node of the chain
    uint32_t first_node;    // preorder index of the chain's first node
    uint32_t first_child;   // first of its child chains
    uint16_t length;        // nodes
    uint8_t n_children;
    uint8_t _pad;
    uint16_t parent_branch; // branch slot of the chain it hangs off (0xffff: the root chain)
    uint16_t branch;        // its own branch slot if it has children, else 0xffff
    uint32_t _pad2[2];
};
static_assert(sizeof(LightChain) == 48, "LightChain must be 48 bytes");
constexpr int LIGHT_MAX_CHAINS = 1056;      // 1043, padded
constexpr int LIGHT_MAX_BRANCHES = 448;     // 441 chains have children
constexpr int LIGHT_CHAIN_K = 8;            // entry terms a chain can hold (more: the cube takes the overflow walk)
constexpr int LIGHT_CHAIN_SLOTS = LIGHT_CHAIN_K + 1;   // + the term of the pop at the chain's end
// per-warp scratch in global memory: the term slots, then one light_ahead_cache word per branch slot (rarely used)
constexpr int LIGHT_WARP_SCRATCH_F4 = LIGHT_MAX_CHAINS * LIGHT_CHAIN_SLOTS + LIGHT_MAX_BRANCHES / 4;

constexpr uint32_t LB_ALL_OPAQUE = 1u << 6, LB_VISIBLE = 1u << 7, LB_EMISSIVE = 1u << 8;
constexpr int LIGHT_MAX_DEPTH = 224;  // longest chart path is 219 (rays end at t = 127, generator.rs:101)

constexpr uint32_t TX_OPAQUE = 128u << 24, TX_NO_RAYS = 1u << 24, TX_UNINIT = 0u;
constexpr int PRIO_NEWLY_VISIBLE = 250, PRIO_ESTIMATED = 200;
constexpr uint32_t LIGHT_TILE = 1024;   // cubes per queue tile (256 words of pending bytes: one 256-thread block)

// The slots of LightParams::scalars, one propagation's counters in device memory.  A round's kernels read the round's
// list length and priority from there, so rounds are queued back to back without a host round trip; a round whose
// priority is already <= epsilon does nothing.  The per-round slots are reset before each round: [LIST_LEN, PRIORITY]
// and [CHANGED, OVERFLOW]; the others accumulate over the propagation.  [TAKEN, QUEUE_MAX] are used only by the
// capped rounds and the queue report of a step (aicb_light_step), SLOT_DIFFS only by aicb_light_take_changes.
enum LightScalar : uint32_t {
    SLOT_LIST_LEN = 0,    // cubes gathered this round
    SLOT_PRIORITY = 1,    // highest queued priority this round
    SLOT_MAX_DIFF = 2,    // largest difference applied
    SLOT_UPDATES = 3,     // cube updates
    SLOT_VISITS = 4,      // chart nodes visited, 64-bit (two slots)
    SLOT_CHANGED = 6,     // entries of the round's list whose cube changed by more than one unit
    SLOT_WALK_NEXT = 7,   // the next list entry the compute walk hands out this round
    SLOT_MARK_NEXT = 8,   // the next `changed` entry the mark walk hands out this round
    SLOT_OVERFLOW = 9,    // entries of the overflow list this round
    SLOT_TAKEN = 10,      // cubes the capped rounds of the step took so far, summed over the members (same in every member)
    SLOT_BAND = 11,       // cubes of the round's band in the member's own tiles (a capped round; peers read it)
    SLOT_QUEUED = 12,     // the step's queue report: queued cubes in the member's own tiles ...
    SLOT_QUEUE_MAX = 13,  // ... and their highest priority
    SLOT_DIFFS = 14,      // texels that differ from the change-tracking baseline
    LIGHT_SCALARS = 16    // slots allocated
};

struct LightParams {
    aicb::DeviceScene scene;        // cells, light, sky faces, tables (LUT)
    const LightBlockDev *blocks;
    const LightNodePre *chart_pre;  // the overflow walk's chart
    const LightChain *chains;       // the chart as chains (breadth-first numbering)
    const uchar4 *node_rel;         // per preorder node: cube relative to the origin (int8 x 3), direction of the step from its parent
    const uint16_t *euler;          // the Euler tour of the chain tree: chain | (0: its entry terms, 1: its pop term) << 15
    uint32_t n_chains, n_euler;
    float4 *term_scratch;           // per resident warp: LIGHT_MAX_CHAINS * LIGHT_CHAIN_SLOTS terms
    uint32_t *overflow;             // list entries whose walk needs more than LIGHT_CHAIN_K terms in one chain
    const float4 *sky_term;         // per preorder node: the sky light its bundle collects at the end of a ray (end_of_ray)
    uint32_t chart_nodes;
    uint32_t *tile_max;             // per LIGHT_TILE cubes: an upper bound of the tile's highest queued priority
    uint8_t *pending;
    uint32_t *list;
    uint32_t *new_light;
    uint8_t *diff;
    uint32_t *changed;              // positions in the round's list whose cube changed by more than one unit (the mark walk's work)
    uint32_t *scalars;              // LightScalar slots
    uint32_t volume;
    uint32_t max_distance;
    uint32_t priority;              // the round's priority level
    uint32_t epsilon_priority;
    uint32_t priority_band;     // cubes whose queued priority is within this many levels of the round's maximum are updated together
};

#ifdef __CUDACC__

namespace aicb_light {

using aicb::DeviceScene;

__device__ __forceinline__ float ps_clamped(float v) { return (v > 0.0f) ? v : 0.0f; }
__device__ __forceinline__ float ps_mul(float a, float b) {
    float v = a * b;
    return (v != v) ? 0.0f : v;
}
__device__ __forceinline__ float fm_sum(const float w[6]) { return (w[0] + w[3]) + (w[1] + w[4]) + (w[2] + w[5]); }

__device__ __forceinline__ uint32_t block_id_at(const DeviceScene &S, uint32_t idx) {
    return S.wide_cells ? (__ldg((const uint32_t *)S.cells + idx) & 0xffffu)
                        : ((uint32_t)__ldg((const uint16_t *)S.cells + idx) & 0x3fffu);
}
__device__ __forceinline__ bool cube_index(const DeviceScene &S, int x, int y, int z, uint32_t *idx) {
    uint32_t dx = (uint32_t)(x - S.lo[0]), dy = (uint32_t)(y - S.lo[1]), dz = (uint32_t)(z - S.lo[2]);
    if ((dx >= (uint32_t)S.size[0]) | (dy >= (uint32_t)S.size[1]) | (dz >= (uint32_t)S.size[2])) return false;
    *idx = (dx * (uint32_t)S.size[1] + dy) * (uint32_t)S.size[2] + dz;
    return true;
}
__device__ __forceinline__ void cube_of(const DeviceScene &S, uint32_t idx, int &x, int &y, int &z) {
    z = (int)(idx % (uint32_t)S.size[2]) + S.lo[2];
    y = (int)((idx / (uint32_t)S.size[2]) % (uint32_t)S.size[1]) + S.lo[1];
    x = (int)(idx / ((uint32_t)S.size[2] * (uint32_t)S.size[1])) + S.lo[0];
}
// UpdateCtx::get_evaluated flags (updater.rs:615-621): out of bounds = AIR (flags 0)
__device__ __forceinline__ uint32_t flags_at(const LightParams &P, int x, int y, int z) {
    uint32_t idx;
    if (!cube_index(P.scene, x, y, z, &idx)) return 0u;
    return __ldg(&P.blocks[block_id_at(P.scene, idx)].flags);
}
// LightStorage::get (updater.rs:585-595)
__device__ __forceinline__ uint32_t light_get(const LightParams &P, int x, int y, int z) {
    uint32_t idx;
    if (cube_index(P.scene, x, y, z, &idx)) return P.scene.light[idx];
    return aicb::light_outside(P.scene, x, y, z);
}
// PackedLight::scalar_in (data.rs:213-217) as a search: qthr[k] (k = 1..255) is the smallest f32 whose
// quantised value is >= k, computed on the host with the platform log2f (monotone) — bit-identical to
// the reference on that host.  `tables` = DeviceScene::tables; the thresholds live at [512, 768).
__device__ __forceinline__ uint32_t scalar_in_t(const float *tables, float v) {
    const float *thr = tables + 512;
    int lo = 0, hi = 255;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int mid = (lo + hi + 1) >> 1;
        if (v >= __ldg(thr + mid)) lo = mid; else hi = mid - 1;
    }
    return (uint32_t)lo;
}
__device__ __forceinline__ int difference_priority(uint32_t a, uint32_t b) {  // data.rs:193-211
    int d = 0;
#pragma unroll
    for (int s = 0; s < 24; s += 8) {
        int x = (a >> s) & 255, y = (b >> s) & 255;
        int e = x > y ? x - y : y - x;
        d = e > d ? e : d;
    }
    if ((a >> 24) != (b >> 24)) d = min(255, d + 63);
    return d;
}

// LightUpdateQueue::insert (queue.rs:107-133): raise the queued priority of a cube (never lowers it).
// The queue is one byte per cube; the byte is updated with a CAS on its containing word.
__device__ __forceinline__ void raise_pending(uint8_t *pending, uint32_t *tile_max, uint32_t idx, uint32_t prio) {
    if (tile_max[idx / LIGHT_TILE] < prio) atomicMax(tile_max + idx / LIGHT_TILE, prio);
    uint32_t *wp = (uint32_t *)(pending + (idx & ~3u));
    const uint32_t shift = (idx & 3u) * 8u;
    uint32_t old = *wp;
    while (((old >> shift) & 255u) < prio) {
        const uint32_t nv = (old & ~(255u << shift)) | (prio << shift);
        const uint32_t prev = atomicCAS(wp, old, nv);
        if (prev == old) break;
        old = prev;
    }
}
// light_needs_update (updater.rs:107-111)
__device__ __forceinline__ void mark_dependency(const LightParams &P, int x, int y, int z, uint32_t prio) {
    uint32_t idx;
    if (cube_index(P.scene, x, y, z, &idx)) raise_pending(P.pending, P.tile_max, idx, prio);
}

struct Accum {
    float in0, in1, in2, total;
};

// end_of_ray (updater.rs:889-924) + add_weighted_light (:926-929).  The sky light a chart node's bundle collects —
// sum over the six faces of sky_face * max(weight, 0), times 1 / sum(weights) — depends on the node and the sky
// only; it is tabulated per scene (`sky`, see light.cu) and a lane only applies its own alpha and bundle weight.
__device__ __forceinline__ void end_of_ray(Accum &a, float alpha, float bundle, const float4 sky) {
    if (bundle > 0.0f) {
        const float ka = ps_clamped(alpha), kb = ps_clamped(bundle);
        a.in0 = a.in0 + ps_mul(ps_mul(sky.x, ka), kb);
        a.in1 = a.in1 + ps_mul(ps_mul(sky.y, ka), kb);
        a.in2 = a.in2 + ps_mul(ps_mul(sky.z, ka), kb);
        a.total += bundle;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// compute_light (updater.rs:368-418) with walk_ray_tree (:427-529) and LightBuffer::traverse (:760-884) for the 32
// cubes of a warp in lockstep (see the header): the overflow walk.  Warp-collective: every lane calls it; `active` =
// this lane has a cube.  The warp visits the union of its cubes' node sets.  Per-lane state of the walk: `ld`, the
// depth of the lane's deepest live frame (-1: only the call of the root is pending; -2: the lane does not walk), and
// its frames (alpha after traverse(), ray_bundle_weight, the children's weight so far, light_ahead_cache) indexed by
// depth — the depth is warp-uniform, so these local-memory accesses are coalesced.
__device__ uint32_t compute_light_lockstep(const LightParams &P, const float *lut, bool active, int ox, int oy, int oz,
                                           uint32_t *visits_out) {
    const DeviceScene &S = P.scene;
    Accum acc = {0.f, 0.f, 0.f, 0.f};
    uint32_t oidx;
    uint32_t oflags = 0;
    const LightBlockDev *ob = nullptr;
    if (active && cube_index(S, ox, oy, oz, &oidx)) {
        ob = &P.blocks[block_id_at(S, oidx)];
        oflags = __ldg(&ob->flags);
    }
    const bool origin_opaque = (oflags & LB_ALL_OPAQUE) != 0;
    uint32_t visits = 0;
    float dw[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (active && origin_opaque) {
        if (oflags & LB_EMISSIVE) {  // !opaque_for_light_computation: add_weighted_light(emission, 1.0)
            acc.in0 = acc.in0 + ps_mul(__ldg(&ob->emission[0]), 1.0f);
            acc.in1 = acc.in1 + ps_mul(__ldg(&ob->emission[1]), 1.0f);
            acc.in2 = acc.in2 + ps_mul(__ldg(&ob->emission[2]), 1.0f);
            acc.total += 1.0f;
        }
    } else if (active) {
        if (oflags & LB_VISIBLE) {
#pragma unroll
            for (int f = 0; f < 6; f++) dw[f] = 1.0f;
        } else {  // directions_to_seek_light (updater.rs:669-690)
#pragma unroll
            for (int f = 0; f < 6; f++) {
                const int s = (f < 3) ? -1 : 1, a = f % 3;
                const uint32_t toward = flags_at(P, ox + (a == 0 ? s : 0), oy + (a == 1 ? s : 0), oz + (a == 2 ? s : 0));
                const uint32_t away = flags_at(P, ox - (a == 0 ? s : 0), oy - (a == 1 ? s : 0), oz - (a == 2 ? s : 0));
                dw[f] = ((away & LB_VISIBLE) || (toward & LB_EMISSIVE)) ? 1.0f : 0.0f;
            }
        }
    }
    int ld = (active && !origin_opaque) ? -1 : -2;
    if (__any_sync(0xffffffffu, ld == -1)) {
        float f_alpha[LIGHT_MAX_DEPTH], f_bundle[LIGHT_MAX_DEPTH], f_csum[LIGHT_MAX_DEPTH];
        float f_sky0[LIGHT_MAX_DEPTH], f_sky1[LIGHT_MAX_DEPTH], f_sky2[LIGHT_MAX_DEPTH];
        uint32_t f_ahead[LIGHT_MAX_DEPTH];
        uint8_t f_have[LIGHT_MAX_DEPTH];
        const int max_d2 = (int)(P.max_distance * P.max_distance);
        // all children of the frame at depth k are done (updater.rs:518-528): the rest of its bundle ends here
        auto pop_level = [&](int k) {
            if (ld == k) {
                end_of_ray(acc, f_alpha[k], fmaxf(f_bundle[k] - f_csum[k], 0.0f), make_float4(f_sky0[k], f_sky1[k], f_sky2[k], 0.f));
                ld = k - 1;
            }
        };
        // The walk is a chain of dependent loads per node (node record -> cube -> cell -> block flags).  Records are
        // read two nodes ahead and the lane's cell one node ahead of the node being processed — node n + 1 is the next
        // node whenever some lane descends, which is the common case in open air; a skip reloads.
        const bool walker = ld == -1;
        const uint32_t n_nodes = P.chart_nodes;
        auto load_rec = [&](uint32_t k, uint4 &a, uint4 &b, float4 &sk) {
            if (k < n_nodes) {
                const uint4 *np = reinterpret_cast<const uint4 *>(P.chart_pre + k);
                a = __ldg(np);
                b = __ldg(np + 1);
                sk = __ldg(P.sky_term + k);
            } else {
                a = make_uint4(0, 0, 0, 0);
                b = make_uint4(0, 0, 0, 0);
                sk = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        // the lane's cube at that node — only for lanes whose walk can still enter it: a lane enters a node of depth
        // e iff its deepest live frame is at e - 1 then, so now it is at e - 2 (and descends) or deeper (and pops)
        auto load_cell = [&](const uint4 &b, uint32_t &cidx, uint32_t &id) -> bool {
            id = 0;
            if (!walker || ld < (int)(b.z >> 24) - 2) return false;
            const int x = ox + (int)(int8_t)(b.z & 255u), y = oy + (int)(int8_t)((b.z >> 8) & 255u), z = oz + (int)(int8_t)((b.z >> 16) & 255u);
            if (!cube_index(S, x, y, z, &cidx)) return false;
            id = block_id_at(S, cidx);
            return true;
        };
        uint32_t n = 0;
        uint4 na, nb, pa, pb, qa, qb;
        float4 nsky, psky, qsky;
        load_rec(0, na, nb, nsky);
        load_rec(1, pa, pb, psky);
        uint32_t cidx = 0, cell_id = 0, cidx1 = 0, cell_id1 = 0;
        bool inb = load_cell(nb, cidx, cell_id), inb1 = false;
        int top = -1;   // deepest depth of the current path that holds a frame of some lane
        for (;;) {
            // requests for the next iteration
            inb1 = (n + 1 < n_nodes) ? load_cell(pb, cidx1, cell_id1) : false;
            load_rec(n + 2, qa, qb, qsky);
            const int d = (int)(nb.z >> 24);
            for (int k = top; k >= d; k--) pop_level(k);
            top = d - 1;
            const uint32_t end_dir = nb.w;
            const int relx = (int)(int8_t)(nb.z & 255u), rely = (int)(int8_t)((nb.z >> 8) & 255u), relz = (int)(int8_t)((nb.z >> 16) & 255u);
            const bool too_far = relx * relx + rely * rely + relz * relz > max_d2;   // updater.rs:452-455, exact in integers
            bool pushed = false;
            if (ld == d - 1) {   // this lane's walk enters the node
                visits++;
                const float cw[6] = {__uint_as_float(na.x), __uint_as_float(na.y), __uint_as_float(na.z),
                                     __uint_as_float(na.w), __uint_as_float(nb.x), __uint_as_float(nb.y)};
                float prod[6];
#pragma unroll
                for (int f = 0; f < 6; f++) prod[f] = cw[f] * dw[f];
                const float bundle = fm_sum(prod);
                const float e_alpha = d == 0 ? 1.0f : f_alpha[d - 1];
                if (bundle > 0.0f) {
                    const int e_x = ox + relx, e_y = oy + rely, e_z = oz + relz;
                    if (too_far || !inb) {
                        end_of_ray(acc, e_alpha, bundle, nsky);
                    } else {
                        // ---- LightBuffer::traverse ----
                        const int dir = (int)(end_dir >> 29);
                        const int e_face = d == 0 ? 0 : ((dir < 3) ? dir + 3 : dir - 3) + 1;
                        const LightBlockDev *ev = &P.blocks[cell_id];
                        const uint32_t fl = __ldg(&ev->flags);
                        float alpha = e_alpha;
                        bool have_ahead = false;
                        uint32_t ahead = 0;
                        if (fl & LB_VISIBLE) {
                            const bool hit_opaque_face = (e_face == 0) ? ((fl & LB_ALL_OPAQUE) != 0) : (((fl >> (e_face - 1)) & 1u) != 0);
                            if (hit_opaque_face && e_face == 0) {
                                alpha = 0.0f;  // (direction weights are zeroed too; nothing reads them afterwards)
                            } else {
                                float col[4];
#pragma unroll
                                for (int i = 0; i < 4; i++) col[i] = __ldg(&ev->face_color[e_face][i]);
#pragma unroll
                                for (int i = 0; i < 3; i++) col[i] = col[i] > 1.0f ? 1.0f : col[i];  // Rgba::clamp
                                const float hit_alpha = col[3];
                                const float kw = ps_clamped(fm_sum(prod));
                                if (hit_alpha > 0.0f && e_face != 0) {
                                    int lx = e_x, ly = e_y, lz = e_z;  // hit.adjacent(): the cube the ray came from
                                    const int ax = (e_face - 1) % 3, sgn = (e_face >= 4) ? 1 : -1;
                                    if (ax == 0) lx += sgn; else if (ax == 1) ly += sgn; else lz += sgn;
                                    const bool e_have_prev = d > 0 && f_have[d - 1] != 0;
                                    const uint32_t stored = e_have_prev ? f_ahead[d - 1] : light_get(P, lx, ly, lz);
                                    const float ka = ps_clamped(alpha);
                                    float lf[3];
                                    lf[0] = __ldg(&ev->emission[0]) + ps_mul(ps_mul(col[0], lut[stored & 255]), hit_alpha);
                                    lf[1] = __ldg(&ev->emission[1]) + ps_mul(ps_mul(col[1], lut[(stored >> 8) & 255]), hit_alpha);
                                    lf[2] = __ldg(&ev->emission[2]) + ps_mul(ps_mul(col[2], lut[(stored >> 16) & 255]), hit_alpha);
                                    acc.in0 = acc.in0 + ps_mul(ps_mul(lf[0], ka), kw);
                                    acc.in1 = acc.in1 + ps_mul(ps_mul(lf[1], ka), kw);
                                    acc.in2 = acc.in2 + ps_mul(ps_mul(lf[2], ka), kw);
                                    if (hit_opaque_face) alpha = 0.0f; else alpha *= 1.0f - hit_alpha;
                                }
                                if (hit_alpha < 1.0f) {
                                    float sv0 = 0.f, sv1 = 0.f, sv2 = 0.f;
                                    if (e_face != 0) {
                                        ahead = S.light[cidx];
                                        have_ahead = true;
                                        sv0 = lut[ahead & 255]; sv1 = lut[(ahead >> 8) & 255]; sv2 = lut[(ahead >> 16) & 255];
                                    }
                                    const float kh = ps_clamped(hit_alpha), ka = ps_clamped(alpha);
                                    const float l0 = __ldg(&ev->emission[0]) + ps_mul(sv0, kh);
                                    const float l1 = __ldg(&ev->emission[1]) + ps_mul(sv1, kh);
                                    const float l2 = __ldg(&ev->emission[2]) + ps_mul(sv2, kh);
                                    acc.in0 = acc.in0 + ps_mul(ps_mul(l0, ka), kw);
                                    acc.in1 = acc.in1 + ps_mul(ps_mul(l1, ka), kw);
                                    acc.in2 = acc.in2 + ps_mul(ps_mul(l2, ka), kw);
                                    alpha *= 1.0f - hit_alpha;
                                }
                            }
                        }
                        if (!(alpha > 0.0f)) {
                            end_of_ray(acc, alpha, bundle, nsky);
                        } else {
                            f_alpha[d] = alpha; f_bundle[d] = bundle; f_csum[d] = 0.0f;
                            f_ahead[d] = ahead; f_have[d] = have_ahead ? 1 : 0;
                            f_sky0[d] = nsky.x; f_sky1[d] = nsky.y; f_sky2[d] = nsky.z;
                            ld = d;
                            pushed = true;
                        }
                    }
                }
                if (d > 0) f_csum[d - 1] += bundle;   // the call returns its bundle weight (updater.rs:514, 528)
            }
            uint32_t next;
            if (__any_sync(0xffffffffu, pushed)) {
                top = d;
                next = n + 1;                    // a child if there is one, else the pops above end the frame
            } else {
                next = end_dir & 0x1fffffffu;    // nobody is inside: skip the subtree
            }
            if (next >= n_nodes) break;
            if (next == n + 1) {
                na = pa; nb = pb; nsky = psky; pa = qa; pb = qb; psky = qsky;
                cidx = cidx1; cell_id = cell_id1; inb = inb1;
            } else {
                load_rec(next, na, nb, nsky);
                load_rec(next + 1, pa, pb, psky);
                inb = load_cell(nb, cidx, cell_id);
            }
            n = next;
        }
        for (int k = top; k >= 0; k--) pop_level(k);
    }
    if (visits_out) *visits_out = visits;
    if (!active) return 0u;
    // LightBuffer::finish (updater.rs:932-944)
    const float scale = ps_clamped(1.0f / fmaxf(acc.total, 1.0f));
    if (acc.total > 0.0f)
        return scalar_in_t(S.tables, ps_mul(acc.in0, scale)) | (scalar_in_t(S.tables, ps_mul(acc.in1, scale)) << 8) |
               (scalar_in_t(S.tables, ps_mul(acc.in2, scale)) << 16) | (255u << 24);
    return origin_opaque ? TX_OPAQUE : TX_NO_RAYS;
}


// ---------------------------------------------------------------------------------------------------------------
// compute_light for ONE cube by the whole warp, chain by chain.
//
// Phase 1 — the walk.  Ready chains wait in a per-warp queue (shared memory); an idle lane takes one and walks its
// nodes in order (LightBuffer::traverse, updater.rs:760-884, per node exactly as the overflow walk does), 32 chains of
// the cube at a time.  A chain that is still alive at its end leaves (alpha, light_ahead_cache) in its branch slot and
// queues its children.  The walk of a cube visits ~3 K nodes on average; the lockstep walk stepped a warp through the
// union of 32 cubes' node sets with 5 lanes taking part per node, here every lane steps a node of its own.
//
// What the reference accumulates in depth-first order (incoming_light, total_rays: f32 additions, not associative) is
// not added during the walk: a lane writes each term (the three colour contributions and the weight) to its chain's
// slots.  Depth-first order over the tree = the Euler tour of the chain tree: a chain's entry terms in node order, its
// child chains, then the term of its pop (walk_ray_tree's `remaining bundle` end_of_ray, updater.rs:518-528 — non-zero
// only at branching nodes: inside a chain parent and child carry identical weights, so bundle - children is exactly 0).
// Phase 2 — the sum.  The warp goes through the static Euler tour 32 positions at a time, gathers the terms that
// exist, and adds them up in order (one lane per channel), bit-identical to the sequential walk.
// MARK: walk only, raising the queue priority of every cube whose light the walk reads (apply_light_update's
// dependency re-queue, updater.rs:355-360); no terms.
// ---------------------------------------------------------------------------------------------------------------
struct ChainShared {
    union {
        struct {   // phase 1
            uint16_t queue[LIGHT_MAX_CHAINS];
            float br_alpha[LIGHT_MAX_BRANCHES];   // alpha at the branching node (> 0); negated when it left a light_ahead_cache
        };
        struct {   // phase 2
            float4 stage[128];
            uint16_t list[128 * LIGHT_CHAIN_K];
        };
    };
    uint8_t cnt_entry[LIGHT_MAX_CHAINS];
    uint8_t cnt_pop[LIGHT_MAX_CHAINS];
};

// returns the new PackedLight texel (every lane); *overflowed: some chain had more terms than its slots hold
template <bool MARK>
__device__ uint32_t compute_light_chains(const LightParams &P, const float *lut, ChainShared &sh, float4 *terms,
                                         int ox, int oy, int oz, uint32_t mark_priority, uint32_t *visits_out,
                                         bool *overflowed) {
    const DeviceScene &S = P.scene;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    // ---- compute_light's prologue (updater.rs:368-418), warp-uniform: every lane evaluates the same cube
    uint32_t oidx;
    uint32_t oflags = 0;
    const LightBlockDev *ob = nullptr;
    if (cube_index(S, ox, oy, oz, &oidx)) {
        ob = &P.blocks[block_id_at(S, oidx)];
        oflags = __ldg(&ob->flags);
    }
    const bool origin_opaque = (oflags & LB_ALL_OPAQUE) != 0;
    __syncwarp();   // (the previous cube's phase 2 is through with the shared arrays)
    *overflowed = false;
    if (visits_out) *visits_out = 0;
    if (origin_opaque) {
        if (MARK) return 0u;
        Accum acc = {0.f, 0.f, 0.f, 0.f};
        if (oflags & LB_EMISSIVE) {
            acc.in0 = acc.in0 + ps_mul(__ldg(&ob->emission[0]), 1.0f);
            acc.in1 = acc.in1 + ps_mul(__ldg(&ob->emission[1]), 1.0f);
            acc.in2 = acc.in2 + ps_mul(__ldg(&ob->emission[2]), 1.0f);
            acc.total += 1.0f;
        }
        const float scale = ps_clamped(1.0f / fmaxf(acc.total, 1.0f));
        if (acc.total > 0.0f)
            return scalar_in_t(S.tables, ps_mul(acc.in0, scale)) | (scalar_in_t(S.tables, ps_mul(acc.in1, scale)) << 8) |
                   (scalar_in_t(S.tables, ps_mul(acc.in2, scale)) << 16) | (255u << 24);
        return TX_OPAQUE;
    }
    float dw[6];
    if (oflags & LB_VISIBLE) {
#pragma unroll
        for (int f = 0; f < 6; f++) dw[f] = 1.0f;
    } else {  // directions_to_seek_light (updater.rs:669-690)
#pragma unroll
        for (int f = 0; f < 6; f++) {
            const int s = (f < 3) ? -1 : 1, a = f % 3;
            const uint32_t toward = flags_at(P, ox + (a == 0 ? s : 0), oy + (a == 1 ? s : 0), oz + (a == 2 ? s : 0));
            const uint32_t away = flags_at(P, ox - (a == 0 ? s : 0), oy - (a == 1 ? s : 0), oz - (a == 2 ? s : 0));
            dw[f] = ((away & LB_VISIBLE) || (toward & LB_EMISSIVE)) ? 1.0f : 0.0f;
        }
    }
    const int max_d2 = (int)(P.max_distance * P.max_distance);
    uint32_t *br_ahead = reinterpret_cast<uint32_t *>(terms + LIGHT_MAX_CHAINS * LIGHT_CHAIN_SLOTS);
    if (!MARK) {   // no chain has a term yet
        uint32_t *z0 = reinterpret_cast<uint32_t *>(sh.cnt_entry), *z1 = reinterpret_cast<uint32_t *>(sh.cnt_pop);
        for (unsigned k = lane; k < LIGHT_MAX_CHAINS / 4; k += 32) { z0[k] = 0u; z1[k] = 0u; }
    }
    if (lane == 0) sh.queue[0] = 0;
    __syncwarp();

    // ---- phase 1 ----
    constexpr uint32_t NONE = 0xffffffffu;
    uint32_t head = 0, tail = 1;          // (warp-uniform)
    uint32_t cur = NONE;                  // the lane's chain
    uint32_t node = 0, remaining = 0, tcount = 0, visits = 0;
    uint32_t push_n = 0, push_first = 0;
    float alpha = 0.f, bundle = 0.f;
    bool have = false, over = false;
    uint32_t ahead = 0;
    uint32_t c_first_child = 0, c_meta = 0;   // n_children | branch << 16
    // the lane's node pipeline: the current node's cube offset, index and block id are in registers when its step
    // begins (requested one step earlier), the next node's offset too (requested two steps earlier)
    uchar4 r4c = make_uchar4(0, 0, 0, 0), r4n = make_uchar4(0, 0, 0, 0);
    bool inb_c = false;
    uint32_t cidx_c = 0, id_c = 0;
    auto locate = [&](const uchar4 r4, uint32_t &cidx, uint32_t &id) -> bool {
        const int x = ox + (int)(int8_t)r4.x, y = oy + (int)(int8_t)r4.y, z = oz + (int)(int8_t)r4.z;
        id = 0;
        if (!cube_index(S, x, y, z, &cidx)) return false;
        id = block_id_at(S, cidx);
        return true;
    };
    for (;;) {
        // children of the chains that ended alive in the last iteration
        {
            uint32_t inc = push_n;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
                if ((int)lane >= off) inc += t;
            }
            const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
            if (total) {
                const uint32_t at = tail + inc - push_n;
                for (uint32_t j = 0; j < push_n; j++) sh.queue[at + j] = (uint16_t)(push_first + j);
                tail += total;
                push_n = 0;
                __syncwarp();
            }
        }
        // idle lanes take chains
        {
            const bool idle = cur == NONE;
            const unsigned m = __ballot_sync(0xffffffffu, idle);
            const uint32_t avail = tail - head;
            const uint32_t rank = __popc(m & lt_mask);
            if (idle && rank < avail) {
                cur = sh.queue[head + rank];
                const uint4 *cp = reinterpret_cast<const uint4 *>(P.chains + cur);
                const uint4 c0 = __ldg(cp), c1 = __ldg(cp + 1), c2 = __ldg(cp + 2);
                const float cw[6] = {__uint_as_float(c0.x), __uint_as_float(c0.y), __uint_as_float(c0.z),
                                     __uint_as_float(c0.w), __uint_as_float(c1.x), __uint_as_float(c1.y)};
                float prod[6];
#pragma unroll
                for (int f = 0; f < 6; f++) prod[f] = cw[f] * dw[f];
                bundle = fm_sum(prod);
                node = c1.z;
                c_first_child = c1.w;
                remaining = c2.x & 0xffffu;
                const uint32_t n_children = (c2.x >> 16) & 0xffu;
                const uint32_t pb = c2.y & 0xffffu, br = c2.y >> 16;
                c_meta = n_children | (br << 16);
                tcount = 0;
                if (pb == 0xffffu) { alpha = 1.0f; have = false; ahead = 0; }
                else {
                    alpha = sh.br_alpha[pb];
                    have = alpha < 0.0f;
                    ahead = 0;
                    if (have) { alpha = -alpha; ahead = br_ahead[pb]; }
                }
                if (!(bundle > 0.0f)) {   // the walk enters the chain's first node and leaves at once (updater.rs:447-450)
                    visits++;
                    cur = NONE;
                } else {
                    r4c = __ldg(P.node_rel + node);
                    r4n = remaining > 1u ? __ldg(P.node_rel + node + 1) : r4c;
                    inb_c = locate(r4c, cidx_c, id_c);
                }
            }
            const uint32_t takers = __popc(m);
            head += takers < avail ? takers : avail;
        }
        if (__ballot_sync(0xffffffffu, cur != NONE) == 0u) break;
        if (cur != NONE) {
            visits++;
            // requests for the steps to come
            bool inb_n = false;
            uint32_t cidx_n = 0, id_n = 0;
            if (remaining > 1u) inb_n = locate(r4n, cidx_n, id_n);
            const uchar4 r4nn = remaining > 2u ? __ldg(P.node_rel + node + 2) : r4n;
            const uchar4 r4 = r4c;
            const int relx = (int)(int8_t)r4.x, rely = (int)(int8_t)r4.y, relz = (int)(int8_t)r4.z;
            const bool too_far = relx * relx + rely * rely + relz * relz > max_d2;   // updater.rs:452-455
            const int e_x = ox + relx, e_y = oy + rely, e_z = oz + relz;
            const uint32_t cidx = cidx_c;
            const bool inb = inb_c;
            bool ended = false;      // the ray bundle ends here: end_of_ray with the whole bundle
            if (too_far || !inb) {
                ended = true;
            } else {
                // ---- LightBuffer::traverse ----
                const int dir = (int)r4.w;
                const int e_face = node == 0u ? 0 : ((dir < 3) ? dir + 3 : dir - 3) + 1;
                const LightBlockDev *ev = &P.blocks[id_c];
                const uint32_t fl = __ldg(&ev->flags);
                const float e_alpha = alpha;
                const bool e_have_prev = have;
                const uint32_t e_ahead_prev = ahead;
                have = false;
                ahead = 0;
                if (fl & LB_VISIBLE) {
                    const bool hit_opaque_face = (e_face == 0) ? ((fl & LB_ALL_OPAQUE) != 0) : (((fl >> (e_face - 1)) & 1u) != 0);
                    if (hit_opaque_face && e_face == 0) {
                        alpha = 0.0f;
                    } else {
                        float col[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) col[i] = __ldg(&ev->face_color[e_face][i]);
#pragma unroll
                        for (int i = 0; i < 3; i++) col[i] = col[i] > 1.0f ? 1.0f : col[i];  // Rgba::clamp
                        const float hit_alpha = col[3];
                        const float kw = ps_clamped(bundle);
                        if (hit_alpha > 0.0f && e_face != 0) {
                            int lx = e_x, ly = e_y, lz = e_z;  // hit.adjacent(): the cube the ray came from
                            const int ax = (e_face - 1) % 3, sgn = (e_face >= 4) ? 1 : -1;
                            if (ax == 0) lx += sgn; else if (ax == 1) ly += sgn; else lz += sgn;
                            if (MARK) mark_dependency(P, lx, ly, lz, mark_priority);
                            if (!MARK) {
                                const uint32_t stored = e_have_prev ? e_ahead_prev : light_get(P, lx, ly, lz);
                                const float ka = ps_clamped(e_alpha);
                                float lf[3];
                                lf[0] = __ldg(&ev->emission[0]) + ps_mul(ps_mul(col[0], lut[stored & 255]), hit_alpha);
                                lf[1] = __ldg(&ev->emission[1]) + ps_mul(ps_mul(col[1], lut[(stored >> 8) & 255]), hit_alpha);
                                lf[2] = __ldg(&ev->emission[2]) + ps_mul(ps_mul(col[2], lut[(stored >> 16) & 255]), hit_alpha);
                                if (tcount < (uint32_t)LIGHT_CHAIN_K)
                                    terms[cur * LIGHT_CHAIN_SLOTS + tcount] = make_float4(ps_mul(ps_mul(lf[0], ka), kw), ps_mul(ps_mul(lf[1], ka), kw), ps_mul(ps_mul(lf[2], ka), kw), 0.0f);
                                else over = true;
                                tcount++;
                            }
                            if (hit_opaque_face) alpha = 0.0f; else alpha *= 1.0f - hit_alpha;
                        }
                        if (hit_alpha < 1.0f) {
                            if (MARK) mark_dependency(P, e_x, e_y, e_z, mark_priority);
                            if (!MARK) {
                                float sv0 = 0.f, sv1 = 0.f, sv2 = 0.f;
                                if (e_face != 0) {
                                    ahead = S.light[cidx];
                                    have = true;
                                    sv0 = lut[ahead & 255]; sv1 = lut[(ahead >> 8) & 255]; sv2 = lut[(ahead >> 16) & 255];
                                }
                                const float kh = ps_clamped(hit_alpha), ka = ps_clamped(alpha);
                                const float l0 = __ldg(&ev->emission[0]) + ps_mul(sv0, kh);
                                const float l1 = __ldg(&ev->emission[1]) + ps_mul(sv1, kh);
                                const float l2 = __ldg(&ev->emission[2]) + ps_mul(sv2, kh);
                                if (tcount < (uint32_t)LIGHT_CHAIN_K)
                                    terms[cur * LIGHT_CHAIN_SLOTS + tcount] = make_float4(ps_mul(ps_mul(l0, ka), kw), ps_mul(ps_mul(l1, ka), kw), ps_mul(ps_mul(l2, ka), kw), 0.0f);
                                else over = true;
                                tcount++;
                            }
                            alpha *= 1.0f - hit_alpha;
                        }
                    }
                }
                if (!(alpha > 0.0f)) ended = true;
            }
            if (ended) {
                if (!MARK) {   // end_of_ray (bundle > 0 here)
                    const float4 sky = __ldg(P.sky_term + node);
                    const float ka = ps_clamped(alpha), kb = ps_clamped(bundle);
                    if (tcount < (uint32_t)LIGHT_CHAIN_K)
                        terms[cur * LIGHT_CHAIN_SLOTS + tcount] = make_float4(ps_mul(ps_mul(sky.x, ka), kb), ps_mul(ps_mul(sky.y, ka), kb), ps_mul(ps_mul(sky.z, ka), kb), bundle);
                    else over = true;
                    tcount++;
                    sh.cnt_entry[cur] = (uint8_t)(tcount < (uint32_t)LIGHT_CHAIN_K ? tcount : (uint32_t)LIGHT_CHAIN_K);
                }
                cur = NONE;
            } else if (--remaining == 0u) {
                // alive at the chain's last node: its children are walked, then the rest of its bundle ends here
                const uint32_t n_children = c_meta & 0xffffu, br = c_meta >> 16;
                if (!MARK) {
                    float csum = 0.0f;
                    for (uint32_t j = 0; j < n_children; j++) {
                        const uint4 *cp = reinterpret_cast<const uint4 *>(P.chains + c_first_child + j);
                        const uint4 c0 = __ldg(cp);
                        const uint2 c1 = __ldg(reinterpret_cast<const uint2 *>(cp + 1));
                        const float cw[6] = {__uint_as_float(c0.x), __uint_as_float(c0.y), __uint_as_float(c0.z),
                                             __uint_as_float(c0.w), __uint_as_float(c1.x), __uint_as_float(c1.y)};
                        float prod[6];
#pragma unroll
                        for (int f = 0; f < 6; f++) prod[f] = cw[f] * dw[f];
                        csum += fm_sum(prod);
                    }
                    const float rem = fmaxf(bundle - csum, 0.0f);
                    if (rem > 0.0f) {
                        const float4 sky = __ldg(P.sky_term + node);
                        const float ka = ps_clamped(alpha), kb = ps_clamped(rem);
                        terms[cur * LIGHT_CHAIN_SLOTS + LIGHT_CHAIN_K] = make_float4(ps_mul(ps_mul(sky.x, ka), kb), ps_mul(ps_mul(sky.y, ka), kb), ps_mul(ps_mul(sky.z, ka), kb), rem);
                        sh.cnt_pop[cur] = 1;
                    }
                    sh.cnt_entry[cur] = (uint8_t)(tcount < (uint32_t)LIGHT_CHAIN_K ? tcount : (uint32_t)LIGHT_CHAIN_K);
                }
                if (n_children) {
                    sh.br_alpha[br] = have ? -alpha : alpha;
                    if (have) br_ahead[br] = ahead;
                    push_n = n_children;
                    push_first = c_first_child;
                }
                cur = NONE;
            } else {
                node++;
                r4c = r4n; r4n = r4nn;
                inb_c = inb_n; cidx_c = cidx_n; id_c = id_n;
            }
        }
        __syncwarp();
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) visits += __shfl_xor_sync(0xffffffffu, visits, off);
    if (visits_out) *visits_out = visits;
    if (MARK) return 0u;
    if (__any_sync(0xffffffffu, over)) { *overflowed = true; return 0u; }
    __syncwarp();

    // ---- phase 2: the terms in depth-first order; lane (k & 3) of every quad carries channel k ----
    // 128 positions of the Euler tour at a time: their terms' slots are listed in order, then fetched 128 at a time
    // (four independent loads per lane) into shared memory and added one after the other.
    float acc = 0.0f;
    const unsigned ch = lane & 3u;
    for (uint32_t p0 = 0; p0 < P.n_euler; p0 += 128) {
        uint32_t c[4], kind[4], cnt[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint32_t p = p0 + 32u * q + lane;
            c[q] = 0; kind[q] = 0; cnt[q] = 0;
            if (p < P.n_euler) {
                const uint32_t e = __ldg(P.euler + p);
                c[q] = e & 0x7fffu; kind[q] = e >> 15;
                cnt[q] = kind[q] ? sh.cnt_pop[c[q]] : sh.cnt_entry[c[q]];
            }
        }
        if (__ballot_sync(0xffffffffu, (cnt[0] | cnt[1] | cnt[2] | cnt[3]) != 0u) == 0u) continue;
        uint32_t total = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t inc = cnt[q];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
                if ((int)lane >= off) inc += t;
            }
            const uint32_t at = total + inc - cnt[q];
            for (uint32_t k = 0; k < cnt[q]; k++)
                sh.list[at + k] = (uint16_t)(c[q] * LIGHT_CHAIN_SLOTS + (kind[q] ? (uint32_t)LIGHT_CHAIN_K : k));
            total += __shfl_sync(0xffffffffu, inc, 31);
        }
        __syncwarp();
        for (uint32_t base = 0; base < total; base += 128) {
            const uint32_t m = total - base < 128u ? total - base : 128u;
            float4 t[4];
#pragma unroll
            for (int r = 0; r < 4; r++) {
                const uint32_t j = 32u * r + lane;
                if (j < m) t[r] = terms[sh.list[base + j]];
            }
#pragma unroll
            for (int r = 0; r < 4; r++) {
                const uint32_t j = 32u * r + lane;
                if (j < m) sh.stage[j] = t[r];
            }
            __syncwarp();
            const float *st = reinterpret_cast<const float *>(sh.stage);
            for (uint32_t j = 0; j < m; j++) acc = acc + st[j * 4 + ch];
            __syncwarp();
        }
    }
    Accum a;
    a.in0 = __shfl_sync(0xffffffffu, acc, 0);
    a.in1 = __shfl_sync(0xffffffffu, acc, 1);
    a.in2 = __shfl_sync(0xffffffffu, acc, 2);
    a.total = __shfl_sync(0xffffffffu, acc, 3);
    // LightBuffer::finish (updater.rs:932-944)
    const float scale = ps_clamped(1.0f / fmaxf(a.total, 1.0f));
    if (a.total > 0.0f)
        return scalar_in_t(S.tables, ps_mul(a.in0, scale)) | (scalar_in_t(S.tables, ps_mul(a.in1, scale)) << 8) |
               (scalar_in_t(S.tables, ps_mul(a.in2, scale)) << 16) | (255u << 24);
    return TX_NO_RAYS;
}

}  // namespace aicb_light
#endif
