// light.cu — host side of the secondary path (SURVEY §8(a) L1-L4): the static light-ray chart
// (space/light/chart/generator.rs), the per-block derived table, and the batched relaxation driver
// replacing LightStorage::update_light_from_queue / apply_light_update / fast_evaluate_light /
// modified_cube_needs_update (space/light/updater.rs) and Mutation::evaluate_light (space.rs:1496-1527).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <unordered_map>

#include "internal.h"
#include "light_kernel.cuh"

using namespace aicb;
using namespace aicb_light;

// ---------------------------------------------------------------------------------------------
// chart generation (generator.rs:49-215) — host, once per context
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int CHAIN_WALK_BLOCKS_PER_SM = 6;   // 4 warps, 80 registers, 26 KB of shared memory each (8 blocks of 64 registers: -15 %)

struct TreeNode {
    int8_t cube[3];
    int children[6];
    float weight[6];
};

// scale_to_integer_step (raycast.rs:797-819) for s = 0.5
double stis_half(double ds) {
    if (ds == 0.0) return INFINITY;
    return (1.0 - 0.5) / std::fabs(ds);  // rem_euclid(+-0.5, 1) == 0.5 either way
}

std::vector<LightChartNode> build_chart() {
    std::vector<TreeNode> pool;
    pool.push_back(TreeNode{{0, 0, 0}, {-1, -1, -1, -1, -1, -1}, {0, 0, 0, 0, 0, 0}});
    const int R = 5;  // RAY_DIRECTION_STEP
    for (int x = -R; x <= R; x++)
        for (int y = -R; y <= R; y++)
            for (int z = -R; z <= R; z++) {
                if (!(std::abs(x) == R || std::abs(y) == R || std::abs(z) == R)) continue;
                const float fx = (float)x, fy = (float)y, fz = (float)z;
                const float len = std::sqrt(fx * fx + fy * fy + fz * fz);
                const float d[3] = {fx / len, fy / len, fz / len};  // Vector3D::normalize
                float cos6[6];
                for (int f = 0; f < 6; f++) {
                    float u[3] = {0, 0, 0};
                    u[f % 3] = (f < 3) ? -1.0f : 1.0f;
                    const float dot = u[0] * d[0] + u[1] * d[1] + u[2] * d[2];
                    cos6[f] = std::fmax(dot, 0.0f);
                }
                // ray_to_steps (generator.rs:100-113): Ray::new([0.5;3], direction).cast(), t <= 127.
                // Unbounded Raycaster (raycast.rs:577-626) from the cube (0,0,0).
                const double dd[3] = {(double)d[0], (double)d[1], (double)d[2]};
                int step[3];
                double t_delta[3], t_max[3];
                for (int a = 0; a < 3; a++) {
                    step[a] = dd[a] == 0.0 ? 0 : (dd[a] < 0.0 ? -1 : 1);
                    t_delta[a] = 1.0 / std::fabs(dd[a]);
                    t_max[a] = stis_half(dd[a]);
                }
                int cube[3] = {0, 0, 0};
                for (int f = 0; f < 6; f++) pool[0].weight[f] += cos6[f];  // the root is on every path
                int cur = 0;
                for (;;) {
                    int axis;
                    if (t_max[0] < t_max[1]) axis = (t_max[0] < t_max[2]) ? 0 : 2;
                    else axis = (t_max[1] < t_max[2]) ? 1 : 2;
                    const double t = t_max[axis];
                    cube[axis] += step[axis];
                    t_max[axis] += t_delta[axis];
                    if (!(t <= 127.0)) break;
                    const int dir = step[axis] > 0 ? 3 + axis : axis;  // Face::from_adjacency(previous, this)
                    int child = pool[cur].children[dir];
                    if (child < 0) {
                        child = (int)pool.size();
                        pool[cur].children[dir] = child;
                        pool.push_back(TreeNode{{(int8_t)cube[0], (int8_t)cube[1], (int8_t)cube[2]}, {-1, -1, -1, -1, -1, -1}, {0, 0, 0, 0, 0, 0}});
                    }
                    cur = child;
                    for (int f = 0; f < 6; f++) pool[cur].weight[f] += cos6[f];
                }
            }
    std::vector<LightChartNode> flat(pool.size());
    for (size_t i = 0; i < pool.size(); i++)
        for (int f = 0; f < 6; f++) {
            flat[i].w[f] = pool[i].weight[f];
            flat[i].child[f] = pool[i].children[f] < 0 ? 0u : (uint32_t)pool[i].children[f];
        }
    return flat;
}

// The chart in depth-first preorder, as the overflow walk (light_kernel.cuh) steps through it: children in Face6
// order (the order walk_ray_tree recurses in, updater.rs:500), each node with its depth, its cube relative to the
// origin, the direction of the step from its parent and the index one past its last descendant.
std::vector<LightNodePre> build_chart_preorder(const std::vector<LightChartNode> &flat, std::vector<uint32_t> *flat_index = nullptr) {
    std::vector<LightNodePre> pre;
    pre.reserve(flat.size());
    struct Item { uint32_t node; int8_t rel[3]; uint8_t depth; uint8_t dir; uint32_t slot; uint8_t next_child; };
    std::vector<Item> stack;
    stack.push_back(Item{0, {0, 0, 0}, 0, 0, 0, 0});
    while (!stack.empty()) {
        Item &it = stack.back();
        if (it.next_child == 0) {   // first visit: emit the node
            it.slot = (uint32_t)pre.size();
            LightNodePre n;
            std::memcpy(n.w, flat[it.node].w, sizeof n.w);
            n.rel[0] = it.rel[0]; n.rel[1] = it.rel[1]; n.rel[2] = it.rel[2];
            n.depth = it.depth;
            n.end_dir = (uint32_t)it.dir << 29;
            pre.push_back(n);
            if (flat_index) flat_index->push_back(it.node);
        }
        int f = it.next_child;
        while (f < 6 && flat[it.node].child[f] == 0) f++;
        if (f < 6) {
            it.next_child = (uint8_t)(f + 1);
            Item c;
            c.node = flat[it.node].child[f];
            c.rel[0] = it.rel[0]; c.rel[1] = it.rel[1]; c.rel[2] = it.rel[2];
            c.rel[f % 3] = (int8_t)(c.rel[f % 3] + ((f < 3) ? -1 : 1));
            c.depth = (uint8_t)(it.depth + 1);
            c.dir = (uint8_t)f;
            c.slot = 0;
            c.next_child = 0;
            stack.push_back(c);   // (invalidates `it`)
        } else {
            pre[it.slot].end_dir |= (uint32_t)pre.size();
            stack.pop_back();
        }
    }
    return pre;
}

const std::vector<LightNodePre> &chart_preorder_host() {
    static const std::vector<LightNodePre> pre = build_chart_preorder(build_chart());
    return pre;
}

// The chart as chains (light_kernel.cuh: LightChain): maximal single-child paths of the preorder chart, numbered
// breadth first; the Euler tour of the chain tree is the depth-first order the terms of a walk are added in.
struct ChainTables {
    std::vector<LightChain> chains;
    std::vector<uchar4> node_rel;
    std::vector<uint16_t> euler;
};
const ChainTables &chain_tables_host() {
    static const ChainTables tables = [] {
        const std::vector<LightNodePre> &pre = chart_preorder_host();
        const uint32_t n = (uint32_t)pre.size();
        auto end_of = [&](uint32_t i) { return pre[i].end_dir & 0x1fffffffu; };
        auto children_of = [&](uint32_t i) {
            std::vector<uint32_t> c;
            for (uint32_t k = i + 1; k < end_of(i); k = end_of(k)) c.push_back(k);
            return c;
        };
        ChainTables t;
        t.node_rel.resize(n);
        for (uint32_t i = 0; i < n; i++)
            t.node_rel[i] = make_uchar4((uint8_t)pre[i].rel[0], (uint8_t)pre[i].rel[1], (uint8_t)pre[i].rel[2], (uint8_t)(pre[i].end_dir >> 29));
        std::vector<uint32_t> start;           // chain -> first node
        std::vector<uint16_t> parent_branch;
        start.push_back(0);
        parent_branch.push_back(0xffff);
        uint16_t n_branches = 0;
        for (size_t c = 0; c < start.size(); c++) {
            LightChain ch;
            std::memset(&ch, 0, sizeof ch);
            std::memcpy(ch.w, pre[start[c]].w, sizeof ch.w);
            ch.first_node = start[c];
            uint32_t e = start[c];
            std::vector<uint32_t> kids = children_of(e);
            while (kids.size() == 1) { e = kids[0]; kids = children_of(e); }
            ch.length = (uint16_t)(e - start[c] + 1);
            ch.n_children = (uint8_t)kids.size();
            ch.parent_branch = parent_branch[c];
            ch.branch = kids.empty() ? (uint16_t)0xffff : n_branches++;
            ch.first_child = (uint32_t)start.size();
            for (uint32_t k : kids) { start.push_back(k); parent_branch.push_back(ch.branch); }
            t.chains.push_back(ch);
        }
        // Euler tour (iterative): enter(c), children in order, exit(c)
        struct It { uint32_t c; uint32_t next; };
        std::vector<It> stack;
        stack.push_back(It{0, 0});
        t.euler.push_back(0);
        while (!stack.empty()) {
            It &it = stack.back();
            const LightChain &ch = t.chains[it.c];
            if (it.next < ch.n_children) {
                const uint32_t k = ch.first_child + it.next++;
                t.euler.push_back((uint16_t)k);
                stack.push_back(It{k, 0});
            } else {
                t.euler.push_back((uint16_t)(it.c | 0x8000u));
                stack.pop_back();
            }
        }
        return t;
    }();
    return tables;
}

void free_chart(aicb_ctx *c) {
    void **ptrs[] = {(void **)&c->d_chart_pre, (void **)&c->d_chains, (void **)&c->d_node_rel, (void **)&c->d_euler,
                     (void **)&c->d_term_scratch};
    for (void **p : ptrs) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
}

aicb_status upload_chart(aicb_ctx *ctx) {
    {
        const ChainTables &t = chain_tables_host();
        if (t.chains.size() > (size_t)LIGHT_MAX_CHAINS || t.chains.size() >= 0x8000u)
            return aicb_fail(AICB_ERR_INVALID, "light chart has more chains than the walk's shared arrays hold");
        size_t branches = 0;
        for (const LightChain &c : t.chains) branches += c.n_children ? 1 : 0;
        if (branches > (size_t)LIGHT_MAX_BRANCHES) return aicb_fail(AICB_ERR_INVALID, "light chart has more branching chains than expected");
        CU(cudaMalloc(&ctx->d_chains, t.chains.size() * sizeof(LightChain)));
        CU(cudaMemcpy(ctx->d_chains, t.chains.data(), t.chains.size() * sizeof(LightChain), cudaMemcpyHostToDevice));
        CU(cudaMalloc(&ctx->d_node_rel, t.node_rel.size() * sizeof(uchar4)));
        CU(cudaMemcpy(ctx->d_node_rel, t.node_rel.data(), t.node_rel.size() * sizeof(uchar4), cudaMemcpyHostToDevice));
        CU(cudaMalloc(&ctx->d_euler, t.euler.size() * sizeof(uint16_t)));
        CU(cudaMemcpy(ctx->d_euler, t.euler.data(), t.euler.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
        ctx->n_chains = (uint32_t)t.chains.size();
        ctx->n_euler = (uint32_t)t.euler.size();
        // one set of term slots per resident warp of the chain walk
        int per_sm = CHAIN_WALK_BLOCKS_PER_SM;
        if (const char *e = getenv("AICB_LIGHT_CTAS")) {   // experiments: fewer resident blocks
            const int v = atoi(e);
            if (v >= 1 && v < per_sm) per_sm = v;
        }
        ctx->chain_walk_blocks = (uint32_t)ctx->num_sms * (uint32_t)per_sm;
        CU(cudaMalloc(&ctx->d_term_scratch, (size_t)ctx->num_sms * CHAIN_WALK_BLOCKS_PER_SM * 4 * LIGHT_WARP_SCRATCH_F4 * sizeof(float4)));
    }
    const std::vector<LightNodePre> &pre = chart_preorder_host();
    CU(cudaMalloc(&ctx->d_chart_pre, pre.size() * sizeof(LightNodePre)));
    CU(cudaMemcpy(ctx->d_chart_pre, pre.data(), pre.size() * sizeof(LightNodePre), cudaMemcpyHostToDevice));
    ctx->chart_nodes = (uint32_t)pre.size();
    return AICB_OK;
}

aicb_status ensure_chart(aicb_ctx *ctx) {
    if (ctx->d_chart_pre) return AICB_OK;   // (d_chart_pre is the last allocation of upload_chart)
    const aicb_status st = upload_chart(ctx);
    if (st != AICB_OK) free_chart(ctx);   // a later call starts over instead of leaking the tables that did fit
    return st;
}

// ---------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------
// The queue: one priority byte per cube (0 = not queued) and, per LIGHT_TILE cubes, an upper bound of the tile's
// highest byte (raised with every insert, recomputed by whoever scans the tile).  Finding the round's priority reads
// the tile bounds only; gathering reads only the tiles that can hold a cube of the round.
__global__ void __launch_bounds__(256) k_tile_rebuild(const LightParams P, uint32_t n_tiles) {
    __shared__ uint32_t s_max[8];
    const uint32_t n_words = (P.volume + 3) / 4;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t w = tile * (LIGHT_TILE / 4) + threadIdx.x;
        const uint32_t v = w < n_words ? ((const uint32_t *)P.pending)[w] : 0u;
        uint32_t m = max(max(v & 255u, (v >> 8) & 255u), max((v >> 16) & 255u, v >> 24));
        for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, off));
        if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0;
            for (int i = 0; i < 8; i++) t = max(t, s_max[i]);
            P.tile_max[tile] = t;
        }
        __syncthreads();
    }
}

__global__ void k_find_max(const LightParams P, uint32_t n_tiles) {
    uint32_t m = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_tiles; i += gridDim.x * blockDim.x) m = max(m, P.tile_max[i]);
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(P.scalars + SLOT_PRIORITY, m);
}

// Thread -> word of the tile in k_gather (which writes it out) and in the capped rounds' kernels.  With a power-of-two
// z extent the tile is a few whole z-rows, and the threads are laid out so that 8 consecutive threads (32 cubes) cover a
// 4 x 8 patch of (y, z) instead of 32 cubes in a line.  The layout was chosen for a walk that shared node records between
// neighbouring cubes.  It stays because it fixes the list order, the order in which cubes are handed out to the walks
// and applied: another layout changes the relaxation's behaviour and its speed.
__device__ __forceinline__ uint32_t gather_word_of_thread(const LightParams &P) {
    uint32_t wl = threadIdx.x;
    const uint32_t nz = (uint32_t)P.scene.size[2];
    if (nz >= 8 && nz <= 256 && (nz & (nz - 1)) == 0) {
        const uint32_t wpr = nz / 4, q = threadIdx.x >> 3, within = threadIdx.x & 7;
        const uint32_t row_group = q / (wpr / 2), pz = q % (wpr / 2);
        wl = (row_group * 4 + (within >> 1)) * wpr + pz * 2 + (within & 1);
    }
    return wl;
}

// The bytes of queue word w (value v) in the round's band, as k_gather selects them: bit k set for byte k; *cnt = how
// many.
__device__ __forceinline__ uint32_t band_select(const LightParams &P, uint32_t v, uint32_t w, uint32_t prio, uint32_t *cnt) {
    uint32_t sel = 0, c = 0;
#pragma unroll
    for (uint32_t k = 0; k < 4; k++) {
        const uint32_t p = (v >> (8 * k)) & 255u;
        if (p > P.epsilon_priority && p + P.priority_band >= prio && w * 4 + k < P.volume) { sel |= 1u << k; c++; }
    }
    *cnt = c;
    return sel;
}

// One block per tile: the cubes of a tile reach the list in index order (block-wide scan), so consecutive list entries
// are neighbours.
__global__ void __launch_bounds__(256) k_gather(const LightParams P, uint32_t n_tiles) {
    __shared__ uint32_t s_part[8], s_max[8], s_base;
    const uint32_t prio = P.scalars[SLOT_PRIORITY];
    if (prio <= P.epsilon_priority) return;
    const uint32_t n_words = (P.volume + 3) / 4;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // thread -> word of the tile: gather_word_of_thread, written out here (the inlined helper schedules differently)
    uint32_t wl = threadIdx.x;
    {
        const uint32_t nz = (uint32_t)P.scene.size[2];
        if (nz >= 8 && nz <= 256 && (nz & (nz - 1)) == 0) {
            const uint32_t wpr = nz / 4, q = threadIdx.x >> 3, within = threadIdx.x & 7;
            const uint32_t row_group = q / (wpr / 2), pz = q % (wpr / 2);
            wl = (row_group * 4 + (within >> 1)) * wpr + pz * 2 + (within & 1);
        }
    }
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t tm = P.tile_max[tile];
        if (tm <= P.epsilon_priority || tm + P.priority_band < prio) continue;   // (block-uniform)
        const uint32_t w = tile * (LIGHT_TILE / 4) + wl;
        uint32_t v = w < n_words ? ((uint32_t *)P.pending)[w] : 0u;
        uint32_t sel = 0, cnt = 0;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) {
            const uint32_t p = (v >> (8 * k)) & 255u;
            if (p > P.epsilon_priority && p + P.priority_band >= prio && w * 4 + k < P.volume) { sel |= 1u << k; cnt++; }
        }
        // exclusive scan of cnt over the block
        uint32_t inc = cnt;
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
            if ((int)lane >= off) inc += t;
        }
        if (lane == 31) s_part[wid] = inc;
        // what stays queued in this tile
        uint32_t rest = 0;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) if (!(sel & (1u << k))) rest = max(rest, (v >> (8 * k)) & 255u);
        for (int off = 16; off > 0; off >>= 1) rest = max(rest, __shfl_down_sync(0xffffffffu, rest, off));
        if (lane == 0) s_max[wid] = rest;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t total = 0, m = 0;
            for (int i = 0; i < 8; i++) { const uint32_t c = s_part[i]; s_part[i] = total; total += c; m = max(m, s_max[i]); }
            s_base = total ? atomicAdd(P.scalars + SLOT_LIST_LEN, total) : 0u;
            P.tile_max[tile] = m;
        }
        __syncthreads();
        if (cnt) {
            uint32_t at = s_base + s_part[wid] + inc - cnt;
#pragma unroll
            for (uint32_t k = 0; k < 4; k++)
                if (sel & (1u << k)) { P.list[at++] = w * 4 + k; v &= ~(255u << (8 * k)); }
            ((uint32_t *)P.pending)[w] = v;
        }
        __syncthreads();
    }
}

// k_compute_overflow: 8 CTAs of 4 warps per SM (64 registers; the records requested ahead spill to L1-resident local
// memory): the walk is latency bound, and 32 resident warps measured +14 % over the 20 that 94 registers allow (6 / 10
// CTAs: +2 % / -30 %).
#ifndef AICB_LIGHT_MIN_BLOCKS
#define AICB_LIGHT_MIN_BLOCKS 8
#endif

// compute_light / the dependency re-queue with the chain walk (light_kernel.cuh: compute_light_chains): one warp per
// cube, cubes handed out by a counter.  k_walk_chains<false> writes new_light for the round's list (or explicit
// cubes); a cube one of whose chains needs more than LIGHT_CHAIN_K terms goes to the overflow list and is computed by
// the overflow walk (k_compute_overflow).  k_walk_chains<true> is the mark walk: the dependency re-queue of
// apply_light_update (updater.rs:355-360) for the entries of `changed`.
template <bool MARK>
__global__ void __launch_bounds__(128, CHAIN_WALK_BLOCKS_PER_SM) k_walk_chains(const LightParams P, uint32_t n, const int32_t *explicit_cubes) {
    __shared__ float s_lut[256];
    __shared__ ChainShared s_sh[4];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = P.scene.tables[i];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    ChainShared &sh = s_sh[wib];
    float4 *terms = P.term_scratch + (size_t)(blockIdx.x * 4 + wib) * LIGHT_WARP_SCRATCH_F4;
    if (!explicit_cubes) n = MARK ? P.scalars[SLOT_CHANGED] : P.scalars[SLOT_LIST_LEN];
    unsigned long long total_visits = 0;
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(P.scalars + (MARK ? SLOT_MARK_NEXT : SLOT_WALK_NEXT), 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n) break;
        const uint32_t i = MARK ? P.changed[item] : item;   // position in the round's list
        int x, y, z;
        if (explicit_cubes) { x = explicit_cubes[3 * i]; y = explicit_cubes[3 * i + 1]; z = explicit_cubes[3 * i + 2]; }
        else cube_of(P.scene, P.list[i], x, y, z);
        const uint32_t prio = MARK ? (uint32_t)P.diff[i] / 2u + 1u : 0u;
        uint32_t visits = 0;
        bool overflowed = false;
        const uint32_t nv = compute_light_chains<MARK>(P, s_lut, sh, terms, x, y, z, prio, &visits, &overflowed);
        if (!MARK && lane == 0) {
            if (overflowed) P.overflow[atomicAdd(P.scalars + SLOT_OVERFLOW, 1u)] = i;
            else P.new_light[i] = nv;
        }
        total_visits += visits;
    }
    if (!MARK && lane == 0 && total_visits) atomicAdd(reinterpret_cast<unsigned long long *>(P.scalars + SLOT_VISITS), total_visits);
}

// the overflow walk: the cubes the chain walk could not hold (the SLOT_OVERFLOW entries of `overflow`)
__global__ void __launch_bounds__(128, AICB_LIGHT_MIN_BLOCKS) k_compute_overflow(const LightParams P, const int32_t *explicit_cubes) {
    __shared__ float s_lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = P.scene.tables[i];
    __syncthreads();
    const uint32_t n = P.scalars[SLOT_OVERFLOW];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    unsigned long long total_visits = 0;
    for (uint32_t base = warp * 32u; base < n; base += n_warps * 32u) {
        const bool active = base + lane < n;
        const uint32_t i = active ? P.overflow[base + lane] : 0u;
        int x = 0, y = 0, z = 0;
        if (active) {
            if (explicit_cubes) { x = explicit_cubes[3 * i]; y = explicit_cubes[3 * i + 1]; z = explicit_cubes[3 * i + 2]; }
            else cube_of(P.scene, P.list[i], x, y, z);
        }
        uint32_t visits = 0;
        const uint32_t nv = compute_light_lockstep(P, s_lut, active, x, y, z, &visits);
        if (active) P.new_light[i] = nv;
        total_visits += visits;
    }
    for (int off = 16; off > 0; off >>= 1) total_visits += __shfl_down_sync(0xffffffffu, total_visits, off);
    if (lane == 0 && total_visits) atomicAdd(reinterpret_cast<unsigned long long *>(P.scalars + SLOT_VISITS), total_visits);
}

// apply_light_update (updater.rs:295-363) minus the dependency re-queue (k_walk_chains<true>)
__global__ void k_apply(const LightParams P) {
    const uint32_t n = P.scalars[SLOT_LIST_LEN];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t idx = P.list[i];
    uint32_t *light = const_cast<uint32_t *>(P.scene.light);
    const uint32_t old = light[idx], nv = P.new_light[i];
    const int d = difference_priority(nv, old);
    P.diff[i] = (uint8_t)d;
    atomicAdd(P.scalars + SLOT_UPDATES, 1u);
    if (d > 0) {
        light[idx] = nv;
        atomicMax(P.scalars + SLOT_MAX_DIFF, (uint32_t)d);
        int x, y, z;
        cube_of(P.scene, idx, x, y, z);
        const float *lut = P.scene.tables;
#pragma unroll
        for (int f = 0; f < 6; f++) {
            const int s = (f < 3) ? -1 : 1, a = f % 3;
            uint32_t nidx;
            if (!cube_index(P.scene, x + (a == 0 ? s : 0), y + (a == 1 ? s : 0), z + (a == 2 ? s : 0), &nidx)) continue;
            const uint32_t nl = light[nidx];
            if ((nl >> 24) != 0) continue;            // only LightStatus::Uninitialized neighbours
            if (nl == nv) continue;
            if (__ldg(&P.blocks[block_id_at(P.scene, nidx)].flags) & LB_ALL_OPAQUE) continue;
            // PackedLight::guess(new.value()): re-quantise the decoded value, status Uninitialized
            const uint32_t g = scalar_in_t(lut, lut[nv & 255]) | (scalar_in_t(lut, lut[(nv >> 8) & 255]) << 8) | (scalar_in_t(lut, lut[(nv >> 16) & 255]) << 16);
            atomicCAS(&light[nidx], nl, g);
        }
    }
    }
}

// apply_light_update re-queues a cube's dependencies only when its packed difference exceeds 1 (updater.rs:355-360).
// The entries of the round's list that did are compacted (in list order within a block of 256) so that the mark walk
// is handed only cubes that need it.
__global__ void __launch_bounds__(256) k_compact_changed(const LightParams P) {
    __shared__ uint32_t s_part[8], s_base;
    const uint32_t n = P.scalars[SLOT_LIST_LEN];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t base = blockIdx.x * 256u; base < n; base += gridDim.x * 256u) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t keep = (i < n && P.diff[i] > 1) ? 1u : 0u;
        uint32_t inc = keep;
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
            if ((int)lane >= off) inc += t;
        }
        if (lane == 31) s_part[wid] = inc;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t total = 0;
            for (int k = 0; k < 8; k++) { const uint32_t c = s_part[k]; s_part[k] = total; total += c; }
            s_base = total ? atomicAdd(P.scalars + SLOT_CHANGED, total) : 0u;
        }
        __syncthreads();
        if (keep) P.changed[s_base + s_part[wid] + inc - 1] = i;
        __syncthreads();
    }
}

// fast_evaluate_light (updater.rs:537-582): one thread per (x, z) column, top down
__global__ void k_fast_evaluate(const LightParams P) {
    const DeviceScene &S = P.scene;
    const uint32_t col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= (uint32_t)S.size[0] * (uint32_t)S.size[2]) return;
    const int x = (int)(col / (uint32_t)S.size[2]) + S.lo[0], z = (int)(col % (uint32_t)S.size[2]) + S.lo[2];
    uint32_t *light = const_cast<uint32_t *>(S.light);
    bool covered = false;
    for (int y = S.lo[1] + S.size[1] - 1; y >= S.lo[1]; y--) {
        uint32_t idx;
        cube_index(S, x, y, z, &idx);
        const uint32_t fl = __ldg(&P.blocks[block_id_at(S, idx)].flags);
        uint32_t value;
        uint8_t pend = 0;
        if ((fl & LB_ALL_OPAQUE) && !(fl & LB_EMISSIVE)) {
            covered = true;
            value = TX_OPAQUE;
        } else {
            bool any = (fl & LB_VISIBLE) != 0;
            if (!any) {
                any = (flags_at(P, x - 1, y, z) | flags_at(P, x + 1, y, z) | flags_at(P, x, y - 1, z) | flags_at(P, x, y + 1, z) |
                       flags_at(P, x, y, z - 1) | flags_at(P, x, y, z + 1)) & LB_VISIBLE;
            }
            if (any) {
                pend = PRIO_ESTIMATED;
                value = covered ? TX_UNINIT : S.sky_faces[4];  // block_sky.in_direction(PY)
            } else {
                value = TX_NO_RAYS;
            }
        }
        light[idx] = value;
        P.pending[idx] = pend;
    }
}

struct EditOp {
    uint32_t idx;
    uint32_t cell;        // new cell word, or 0xffffffff = leave
    uint8_t set_opaque;   // light := OPAQUE
    uint8_t pending_op;   // 0 none, 1 remove, 2 raise to NEWLY_VISIBLE
    uint8_t _pad[2];
};

__global__ void k_edits(const LightParams P, const EditOp *ops, uint32_t n, uint32_t wide) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const EditOp op = ops[i];
    if (op.cell != 0xffffffffu) {
        if (wide) ((uint32_t *)P.scene.cells)[op.idx] = op.cell;
        else ((uint16_t *)P.scene.cells)[op.idx] = (uint16_t)op.cell;
    }
    if (op.set_opaque) const_cast<uint32_t *>(P.scene.light)[op.idx] = TX_OPAQUE;
    if (op.pending_op == 1) P.pending[op.idx] = 0;
    else if (op.pending_op == 2) P.pending[op.idx] = PRIO_NEWLY_VISIBLE;
}

LightParams make_params(aicb_scene *s) {
    LightParams P;
    std::memset(&P, 0, sizeof P);
    P.scene = s->ds;
    P.blocks = s->d_light_blocks;
    P.chart_pre = s->ctx->d_chart_pre;
    P.sky_term = s->d_sky_term;
    P.chains = s->ctx->d_chains;
    P.node_rel = s->ctx->d_node_rel;
    P.euler = s->ctx->d_euler;
    P.n_chains = s->ctx->n_chains;
    P.n_euler = s->ctx->n_euler;
    P.term_scratch = s->ctx->d_term_scratch;
    P.overflow = s->d_changed;   // (a round's overflow list is consumed before k_compact_changed lists its changed cubes)
    P.chart_nodes = s->ctx->chart_nodes;
    P.tile_max = s->d_tile_max;
    P.changed = s->d_changed;
    P.pending = s->d_pending;
    P.list = s->d_list;
    P.new_light = s->d_new_light;
    P.diff = s->d_diff;
    P.scalars = s->d_scalars;
    P.volume = (uint32_t)s->volume;
    P.max_distance = s->light_max_distance;
    return P;
}

aicb_status ensure_light_state(aicb_scene *s) {
    if (s->light_max_distance == 0) return aicb_fail(AICB_ERR_INVALID, "scene has LightPhysics::None (light_max_distance == 0)");
    aicb_status st = ensure_chart(s->ctx);
    if (st != AICB_OK) return st;
    if (!s->d_light) {  // a scene created without a light volume starts all NO_RAYS (initialize_light, updater.rs:628-656)
        std::vector<uint32_t> init(s->volume, TX_NO_RAYS);
        CU(cudaMalloc(&s->d_light, s->volume * 4 + 16));
        CU(cudaMemcpy(s->d_light, init.data(), s->volume * 4, cudaMemcpyHostToDevice));
        s->ds.light = s->d_light;
        s->device_bytes += s->volume * 4;
    }
    if (!s->d_sky_term) {
        // end_of_ray (updater.rs:889-924) without the lane's alpha and bundle weight: per chart node, the sky light
        // its bundle collects — the same f32 operations, in the same order, as the reference evaluates per ray end
        const std::vector<LightNodePre> &pre = chart_preorder_host();
        float lut[256];
        lut[0] = 0.0f;
        for (int i = 1; i < 256; i++) lut[i] = (float)std::exp2((double)(((float)i - 144.0f) / 10.0f));
        auto psc = [](float v) { return v > 0.0f ? v : 0.0f; };
        auto psm = [](float a, float b) { float v = a * b; return (v != v) ? 0.0f : v; };
        std::vector<float4> sky(pre.size());
        for (size_t k = 0; k < pre.size(); k++) {
            const float *cw = pre[k].w;
            float t[6][3];
            for (int f = 0; f < 6; f++) {
                const uint32_t tx = s->ds.sky_faces[f];
                const float kk = psc(cw[f]);
                t[f][0] = psm(lut[tx & 255], kk);
                t[f][1] = psm(lut[(tx >> 8) & 255], kk);
                t[f][2] = psm(lut[(tx >> 16) & 255], kk);
            }
            const float kr = psc(1.0f / ((cw[0] + cw[3]) + (cw[1] + cw[4]) + (cw[2] + cw[5])));
            float c[3];
            for (int i = 0; i < 3; i++) c[i] = psm((t[0][i] + t[3][i]) + (t[1][i] + t[4][i]) + (t[2][i] + t[5][i]), kr);
            sky[k] = make_float4(c[0], c[1], c[2], 0.0f);
        }
        CU(cudaMalloc(&s->d_sky_term, sky.size() * sizeof(float4)));
        CU(cudaMemcpy(s->d_sky_term, sky.data(), sky.size() * sizeof(float4), cudaMemcpyHostToDevice));
        s->device_bytes += sky.size() * sizeof(float4);
    }
    if (!s->d_pending) {
        CU(cudaMalloc(&s->d_pending, s->volume + 16));
        CU(cudaMemset(s->d_pending, 0, s->volume + 16));
        CU(cudaMalloc(&s->d_list, s->volume * 4 + 16));
        CU(cudaMalloc(&s->d_new_light, s->volume * 4 + 16));
        CU(cudaMalloc(&s->d_diff, s->volume + 16));
        CU(cudaMalloc(&s->d_scalars, LIGHT_SCALARS * 4));
        CU(cudaMalloc(&s->d_tile_max, ((s->volume + LIGHT_TILE - 1) / LIGHT_TILE + 1) * 4));
        CU(cudaMalloc(&s->d_changed, s->volume * 4 + 16));
        s->device_bytes += s->volume * 4;
        s->device_bytes += s->volume * 10;
    }
    if (!s->d_tile_off) {
        const size_t tiles = (s->volume + LIGHT_TILE - 1) / LIGHT_TILE + 1;
        CU(cudaMalloc(&s->d_tile_count, tiles * 4));
        CU(cudaMalloc(&s->d_tile_off, tiles * 4));
        s->device_bytes += tiles * 8;
    }
    return AICB_OK;
}

// the parameters of a propagation's rounds
LightParams propagate_params(aicb_scene *s, uint8_t epsilon) {
    LightParams P = make_params(s);
    P.epsilon_priority = (uint32_t)epsilon / 2 + 1;
    // Cubes within 16 priority levels of the round's maximum are relaxed together: 3.5x the throughput of strict
    // level-by-level rounds (few cubes per round leave the GPU idle) for 8 % more updates; the parity contract
    // (tests/test_gpu_light.py) holds for every band, 0 = one level per round, 255 = all pending cubes.
    const char *e = getenv("AICB_LIGHT_BAND");
    P.priority_band = e ? (uint32_t)atoi(e) : 16u;
    return P;
}

// Mutation::set x n (space.rs:1346-1352 -> side_effects_of_set -> modified_cube_needs_update, updater.rs:135-173):
// validates every edit, then applies them in order to the host mirror of every member (the members are replicas) and
// returns what each member's device has to change.  Nothing changes when an edit is invalid.
aicb_status edit_ops(const std::vector<aicb_scene *> &members, const int32_t (*cubes)[3], const uint16_t *new_ids,
                     size_t n_edits, std::vector<EditOp> *out) {
    const aicb_scene *s = members[0];
    const DeviceScene &ds = s->ds;
    auto index_of = [&](int x, int y, int z, uint32_t *idx) {
        uint32_t dx = (uint32_t)(x - ds.lo[0]), dy = (uint32_t)(y - ds.lo[1]), dz = (uint32_t)(z - ds.lo[2]);
        if (dx >= (uint32_t)ds.size[0] || dy >= (uint32_t)ds.size[1] || dz >= (uint32_t)ds.size[2]) return false;
        *idx = (dx * (uint32_t)ds.size[1] + dy) * (uint32_t)ds.size[2] + dz;
        return true;
    };
    std::unordered_map<uint32_t, EditOp> ops;
    auto op_of = [&](uint32_t idx) -> EditOp & {
        auto it = ops.find(idx);
        if (it == ops.end()) {
            EditOp o;
            std::memset(&o, 0, sizeof o);
            o.idx = idx;
            o.cell = 0xffffffffu;
            it = ops.emplace(idx, o).first;
        }
        return it->second;
    };
    // validate everything before the host mirror (or anything else) changes
    for (size_t i = 0; i < n_edits; i++) {
        uint32_t idx;
        if (!index_of(cubes[i][0], cubes[i][1], cubes[i][2], &idx)) return aicb_fail(AICB_ERR_INVALID, "cube out of bounds");
        if (new_ids[i] >= s->h_block_light.size()) return aicb_fail(AICB_ERR_INVALID, "block id out of range");
    }
    for (size_t i = 0; i < n_edits; i++) {
        uint32_t idx;
        index_of(cubes[i][0], cubes[i][1], cubes[i][2], &idx);
        if (s->h_ids[idx] == new_ids[i]) continue;  // Mutation::set of the same block changes nothing
        for (aicb_scene *m : members) m->h_ids[idx] = new_ids[i];
        EditOp &o = op_of(idx);
        o.cell = ds.wide_cells ? (new_ids[i] | ((uint32_t)s->block_kind[new_ids[i]] << 16))
                               : (new_ids[i] | ((uint32_t)s->block_kind[new_ids[i]] << 14));
        const uint32_t fl = s->h_block_light[new_ids[i]];
        if ((fl & LB_ALL_OPAQUE) && !(fl & LB_EMISSIVE)) {  // opaque_for_light_computation
            o.set_opaque = 1;
            o.pending_op = 1;
        } else {
            o.pending_op = 2;
        }
        for (int f = 0; f < 6; f++) {
            const int sgn = (f < 3) ? -1 : 1, a = f % 3;
            uint32_t nidx;
            if (!index_of(cubes[i][0] + (a == 0 ? sgn : 0), cubes[i][1] + (a == 1 ? sgn : 0), cubes[i][2] + (a == 2 ? sgn : 0), &nidx))
                continue;
            const int opp = (f < 3) ? f + 3 : f - 3;
            if (!((s->h_block_light[s->h_ids[nidx]] >> opp) & 1u)) op_of(nidx).pending_op = 2;
        }
    }
    out->clear();
    out->reserve(ops.size());
    for (auto &kv : ops) out->push_back(kv.second);
    return AICB_OK;
}

// the device side of edit_ops: cells, light and queue bytes of the edited cubes and their neighbours
aicb_status apply_edit_ops(aicb_scene *s, const std::vector<EditOp> &flat) {
    if (flat.empty()) return AICB_OK;
    EditOp *d_ops = nullptr;
    CU(cudaMalloc(&d_ops, flat.size() * sizeof(EditOp)));
    cudaError_t e = cudaMemcpyAsync(d_ops, flat.data(), flat.size() * sizeof(EditOp), cudaMemcpyHostToDevice, s->ctx->stream);
    if (e == cudaSuccess) {
        LightParams P = make_params(s);
        k_edits<<<(unsigned)((flat.size() + 127) / 128), 128, 0, s->ctx->stream>>>(P, d_ops, (uint32_t)flat.size(), s->ds.wide_cells);
        e = cudaStreamSynchronize(s->ctx->stream);
    }
    cudaFree(d_ops);
    if (e != cudaSuccess) return aicb_cuda_fail(e, "light edits");
    return AICB_OK;
}

// the light-side record of a block definition; its flags are also kept on the host (aicb_scene::h_block_light)
LightBlockDev light_block_of(const aicb_block_desc &b) {
    LightBlockDev o;
    std::memset(&o, 0, sizeof o);
    std::memcpy(o.face_color[0], b.light_color, 16);
    for (int f = 0; f < 6; f++) std::memcpy(o.face_color[f + 1], b.light_face_colors[f], 16);
    std::memcpy(o.emission, b.light_emission, 12);
    uint32_t fl = b.light_opaque_faces & 0x3f;
    if (fl == 0x3f) fl |= LB_ALL_OPAQUE;
    if (b.light_visible) fl |= LB_VISIBLE;
    if (!(b.light_emission[0] == 0.0f && b.light_emission[1] == 0.0f && b.light_emission[2] == 0.0f)) fl |= LB_EMISSIVE;
    o.flags = fl;
    return o;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// called from aicb200.cu
// ---------------------------------------------------------------------------------------------
aicb_status aicb_light_scene_upload(aicb_scene *s, const aicb_scene_desc *d) {
    s->light_max_distance = d->light_max_distance;
    if (s->volume) s->h_ids.assign(d->block_ids, d->block_ids + s->volume);
    std::vector<LightBlockDev> lb(d->n_blocks);
    s->h_block_light.resize(d->n_blocks);
    for (size_t i = 0; i < d->n_blocks; i++) {
        lb[i] = light_block_of(d->blocks[i]);
        s->h_block_light[i] = lb[i].flags;
    }
    if (!lb.empty()) {
        CU(cudaMalloc(&s->d_light_blocks, lb.size() * sizeof(LightBlockDev)));
        CU(cudaMemcpy(s->d_light_blocks, lb.data(), lb.size() * sizeof(LightBlockDev), cudaMemcpyHostToDevice));
        s->device_bytes += lb.size() * sizeof(LightBlockDev);
    }
    return AICB_OK;
}

// the light-side records of replaced block definitions (aicb_scene_update_blocks)
aicb_status aicb_light_blocks_update(aicb_scene *s, const uint16_t *indices, const aicb_block_desc *descs, size_t n) {
    for (size_t i = 0; i < n; i++) {
        const LightBlockDev o = light_block_of(descs[i]);
        if (indices[i] < s->h_block_light.size()) s->h_block_light[indices[i]] = o.flags;
        if (s->d_light_blocks) CU(cudaMemcpy(s->d_light_blocks + indices[i], &o, sizeof o, cudaMemcpyHostToDevice));
    }
    return AICB_OK;
}

void aicb_light_scene_free(aicb_scene *s) {
    if (s->d_light_blocks) cudaFree(s->d_light_blocks);
    if (s->d_pending) cudaFree(s->d_pending);
    if (s->d_list) cudaFree(s->d_list);
    if (s->d_new_light) cudaFree(s->d_new_light);
    if (s->d_diff) cudaFree(s->d_diff);
    if (s->d_scalars) cudaFree(s->d_scalars);
    if (s->d_tile_max) cudaFree(s->d_tile_max);
    if (s->d_changed) cudaFree(s->d_changed);
    if (s->d_sky_term) cudaFree(s->d_sky_term);
    if (s->d_tile_count) cudaFree(s->d_tile_count);
    if (s->d_tile_off) cudaFree(s->d_tile_off);
    if (s->d_light_base) cudaFree(s->d_light_base);
    if (s->d_changes) cudaFree(s->d_changes);
}

void aicb_light_ctx_free(aicb_ctx *c) { free_chart(c); }

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

uint32_t aicb_light_chart_chains(uint32_t *preorder, uint32_t (*chains)[6], uint16_t *euler) {
    const ChainTables &t = chain_tables_host();
    if (preorder) {
        std::vector<uint32_t> order;
        build_chart_preorder(build_chart(), &order);
        std::memcpy(preorder, order.data(), order.size() * sizeof(uint32_t));
    }
    if (chains)
        for (size_t c = 0; c < t.chains.size(); c++) {
            const LightChain &ch = t.chains[c];
            chains[c][0] = ch.first_node; chains[c][1] = ch.length; chains[c][2] = ch.n_children;
            chains[c][3] = ch.first_child; chains[c][4] = ch.parent_branch; chains[c][5] = ch.branch;
        }
    if (euler) std::memcpy(euler, t.euler.data(), t.euler.size() * sizeof(uint16_t));
    return (uint32_t)t.chains.size();
}

uint32_t aicb_light_chart(float *weights, uint32_t *children) {
    static const std::vector<LightChartNode> chart = build_chart();
    for (size_t i = 0; i < chart.size(); i++) {
        if (weights) std::memcpy(weights + 6 * i, chart[i].w, 24);
        if (children) std::memcpy(children + 6 * i, chart[i].child, 24);
    }
    return (uint32_t)chart.size();
}

aicb_status aicb_light_fast_evaluate(aicb_scene *s) {
    if (!s) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lock(s->ctx->mu);
    CU(cudaSetDevice(s->ctx->device));
    aicb_status st = ensure_light_state(s);
    if (st != AICB_OK) return st;
    LightParams P = make_params(s);
    const uint32_t cols = (uint32_t)s->ds.size[0] * (uint32_t)s->ds.size[2];
    if (cols) k_fast_evaluate<<<(cols + 127) / 128, 128, 0, s->ctx->stream>>>(P);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s->ctx->stream));
    return AICB_OK;
}

aicb_status aicb_light_compute(aicb_scene *s, const int32_t (*cubes)[3], size_t n, uint8_t (*out)[4]) {
    if (!s || (n && (!cubes || !out))) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    if (n > s->volume) return aicb_fail(AICB_ERR_INVALID, "more cubes than the Space holds");
    std::lock_guard<std::mutex> lock(s->ctx->mu);
    CU(cudaSetDevice(s->ctx->device));
    aicb_status st = ensure_light_state(s);
    if (st != AICB_OK) return st;
    if (!n) return AICB_OK;
    LightParams P = make_params(s);
    int32_t *d_cubes = nullptr;
    CU(cudaMalloc(&d_cubes, n * 12));
    CU(cudaMemcpy(d_cubes, cubes, n * 12, cudaMemcpyHostToDevice));
    cudaMemsetAsync(s->d_scalars, 0, LIGHT_SCALARS * 4, s->ctx->stream);
    k_walk_chains<false><<<s->ctx->chain_walk_blocks, 128, 0, s->ctx->stream>>>(P, (uint32_t)n, d_cubes);
    k_compute_overflow<<<s->ctx->num_sms * 8, 128, 0, s->ctx->stream>>>(P, d_cubes);
    uint32_t h[LIGHT_SCALARS];
    cudaError_t e = cudaMemcpyAsync(out, s->d_new_light, n * 4, cudaMemcpyDeviceToHost, s->ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, s->d_scalars, sizeof h, cudaMemcpyDeviceToHost, s->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->ctx->stream);
    if (e == cudaSuccess) {
        s->light_stats[0] = n;
        s->light_stats[1] = (uint64_t)h[SLOT_VISITS] | ((uint64_t)h[SLOT_VISITS + 1] << 32);
        s->light_stats[2] = h[SLOT_OVERFLOW];   // cubes that took the overflow walk (a chain with more terms than its slots)
        s->light_stats[3] = 0;
    }
    cudaFree(d_cubes);
    if (e != cudaSuccess) return aicb_cuda_fail(e, "light compute");
    return AICB_OK;
}

aicb_status aicb_light_download(aicb_scene *s, uint8_t (*out)[4], size_t n_texels) {
    if (!s || !out) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    if (n_texels != s->volume) return aicb_fail(AICB_ERR_INVALID, "light volume size mismatch");
    if (!s->d_light) return aicb_fail(AICB_ERR_INVALID, "scene has no light volume (LightPhysics::None)");
    std::lock_guard<std::mutex> lock(s->ctx->mu);
    CU(cudaSetDevice(s->ctx->device));
    // ordered behind everything queued on the context's stream (cube deltas, propagation)
    CU(cudaMemcpyAsync(out, s->d_light, s->volume * 4, cudaMemcpyDeviceToHost, s->ctx->stream));
    CU(cudaStreamSynchronize(s->ctx->stream));
    return AICB_OK;
}

aicb_status aicb_light_stats(const aicb_scene *s, uint64_t out[4]) {
    if (!s || !out) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    for (int i = 0; i < 4; i++) out[i] = s->light_stats[i];
    return AICB_OK;
}
}

// ---------------------------------------------------------------------------------------------
// light propagation on a device group (aicb_group_light_*): the relaxation sharded by slabs
// ---------------------------------------------------------------------------------------------
// Every member holds a full replica of the scene, its light and its queue.  Member i owns the queue tiles
// [tile_lo[i], tile_lo[i + 1]) (an even split of whole LIGHT_TILE tiles: a slab along x in the Z-major layout, possibly
// empty); only the owner gathers, computes and applies its cubes.  A round keeps the single-scene round's meaning
// (relax() with one member) with barriers (B) between its steps, all stream-ordered through member 0 (no device-side
// waits):
//   find_max over the member's queue            B1
//   clear the queue outside the member's tiles, round priority := the members' maximum, gather, compute (the member's
//   full replica is read)                       B2  (no replica is written while a peer may still read it)
//   apply: the owner stores each changed texel into every replica     B3
//   guess the Uninitialized neighbours (PackedLight::guess): a CAS on the replica of the neighbour's owner   B4
//   copy guessed texels from their owner into the other replicas; mark (the dependency re-queue) into the member's
//   full-size queue                             B5
//   merge: each owner takes the byte-wise maximum of its peers' queue bytes in its own tiles.
// Between the members' queues: outside its tiles a member's queue only ever holds marks already merged into their
// owners (so its find_max still yields the global maximum) and is cleared after B1, before that member gathers.
namespace {

constexpr uint32_t GROUP_LIGHT_MAX = 16;   // members of a propagating group

struct GroupPeers {
    uint32_t *light[GROUP_LIGHT_MAX];       // every member's replica (device pointers, peer-mapped)
    uint8_t *pending[GROUP_LIGHT_MAX];
    uint32_t *tile_max[GROUP_LIGHT_MAX];
    uint32_t *scalars[GROUP_LIGHT_MAX];
    uint32_t tile_lo[GROUP_LIGHT_MAX + 1];  // member i owns the tiles [tile_lo[i], tile_lo[i + 1])
    uint32_t n, self;
};

__device__ __forceinline__ uint32_t owner_of(const GroupPeers &G, uint32_t idx) {
    const uint32_t tile = idx / LIGHT_TILE;
    uint32_t o = G.n - 1;
    while (o > 0 && tile < G.tile_lo[o]) o--;
    return o;
}

// after B1: the queue outside the member's own tiles (already merged into their owners) is cleared
__global__ void __launch_bounds__(256) k_group_clear_foreign(const LightParams P, const GroupPeers G, uint32_t n_tiles) {
    const uint32_t lo = G.tile_lo[G.self], hi = G.tile_lo[G.self + 1];
    const uint32_t n_words = (P.volume + 3) / 4;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if ((tile >= lo && tile < hi) || P.tile_max[tile] == 0) continue;   // (block-uniform)
        const uint32_t w = tile * (LIGHT_TILE / 4) + threadIdx.x;
        if (w < n_words) ((uint32_t *)P.pending)[w] = 0u;
        __syncthreads();   // every thread has read the tile's bound
        if (threadIdx.x == 0) P.tile_max[tile] = 0u;
    }
}

// after B1: the round's priority is the highest over the members.  A peer may raise its own [1] to the same maximum
// while it is read here; either value yields the same maximum.
__global__ void k_group_max(const LightParams P, const GroupPeers G) {
    if (threadIdx.x >= G.n) return;
    const uint32_t m = *(volatile const uint32_t *)(G.scalars[threadIdx.x] + SLOT_PRIORITY);
    if (m) atomicMax(P.scalars + SLOT_PRIORITY, m);
}

// after B2: apply_light_update (updater.rs:295-363) for the member's own cubes, stored into every replica; the
// guesses of k_apply are k_group_guess, the dependency re-queue is k_walk_chains<true>
__global__ void k_group_apply(const LightParams P, const GroupPeers G) {
    const uint32_t n = P.scalars[SLOT_LIST_LEN];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t idx = P.list[i];
        const uint32_t old = P.scene.light[idx], nv = P.new_light[i];
        const int d = difference_priority(nv, old);
        P.diff[i] = (uint8_t)d;
        atomicAdd(P.scalars + SLOT_UPDATES, 1u);
        if (d > 0) {
            for (uint32_t m = 0; m < G.n; m++) G.light[m][idx] = nv;
            atomicMax(P.scalars + SLOT_MAX_DIFF, (uint32_t)d);
        }
    }
}

// after B3: PackedLight::guess for the Uninitialized neighbours of the member's changed cubes, as in k_apply, with
// the CAS on the neighbour's owner's replica (one winner per texel whichever member guesses)
__global__ void k_group_guess(const LightParams P, const GroupPeers G) {
    const uint32_t n = P.scalars[SLOT_LIST_LEN];
    const float *lut = P.scene.tables;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (P.diff[i] == 0) continue;
        const uint32_t nv = P.new_light[i];
        int x, y, z;
        cube_of(P.scene, P.list[i], x, y, z);
#pragma unroll
        for (int f = 0; f < 6; f++) {
            const int s = (f < 3) ? -1 : 1, a = f % 3;
            uint32_t nidx;
            if (!cube_index(P.scene, x + (a == 0 ? s : 0), y + (a == 1 ? s : 0), z + (a == 2 ? s : 0), &nidx)) continue;
            uint32_t *owner = G.light[owner_of(G, nidx)];
            const uint32_t nl = owner[nidx];
            if ((nl >> 24) != 0) continue;            // only LightStatus::Uninitialized neighbours
            if (nl == nv) continue;
            if (__ldg(&P.blocks[block_id_at(P.scene, nidx)].flags) & LB_ALL_OPAQUE) continue;
            const uint32_t g = scalar_in_t(lut, lut[nv & 255]) | (scalar_in_t(lut, lut[(nv >> 8) & 255]) << 8) | (scalar_in_t(lut, lut[(nv >> 16) & 255]) << 16);
            atomicCAS(owner + nidx, nl, g);
        }
    }
}

// after B4: the Uninitialized neighbours of the member's changed cubes (every texel a guess may have changed) are
// copied from their owner's replica into the others.  Several members may store one texel: all store the same value.
__global__ void k_group_broadcast(const LightParams P, const GroupPeers G) {
    const uint32_t n = P.scalars[SLOT_LIST_LEN];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (P.diff[i] == 0) continue;
        int x, y, z;
        cube_of(P.scene, P.list[i], x, y, z);
        for (int f = 0; f < 6; f++) {
            const int s = (f < 3) ? -1 : 1, a = f % 3;
            uint32_t nidx;
            if (!cube_index(P.scene, x + (a == 0 ? s : 0), y + (a == 1 ? s : 0), z + (a == 2 ? s : 0), &nidx)) continue;
            const uint32_t o = owner_of(G, nidx);
            const uint32_t v = G.light[o][nidx];
            if ((v >> 24) != 0) continue;
            for (uint32_t m = 0; m < G.n; m++)
                if (m != o) G.light[m][nidx] = v;
        }
    }
}

// after B5: the owner takes the byte-wise maximum of its peers' queue bytes in its own tiles (only the tiles a peer's
// bound says hold something)
__global__ void __launch_bounds__(256) k_group_merge(const LightParams P, const GroupPeers G) {
    const uint32_t lo = G.tile_lo[G.self], hi = G.tile_lo[G.self + 1];
    const uint32_t n_words = (P.volume + 3) / 4;
    for (uint32_t tile = lo + blockIdx.x; tile < hi; tile += gridDim.x) {
        const uint32_t w = tile * (LIGHT_TILE / 4) + threadIdx.x;
        uint32_t v = w < n_words ? ((const uint32_t *)P.pending)[w] : 0u;
        uint32_t tm = 0;
        for (uint32_t p = 0; p < G.n; p++) {
            if (p == G.self) continue;
            const uint32_t ptm = G.tile_max[p][tile];   // (block-uniform)
            if (ptm == 0) continue;
            tm = max(tm, ptm);
            if (w < n_words) v = __vmaxu4(v, ((const uint32_t *)G.pending[p])[w]);
        }
        if (tm) {
            if (w < n_words) ((uint32_t *)P.pending)[w] = v;
            if (threadIdx.x == 0 && P.tile_max[tile] < tm) P.tile_max[tile] = tm;
        }
    }
}

// ---- capped rounds and the queue report of a step (aicb_light_step) ----
// A capped round relaxes the same band as an uncapped one but takes only its first `rem` cubes (rem = what is left of
// the step's cap) in a fixed order: tiles in increasing order, within a tile k_gather's thread -> word and byte order.
// The members' tiles are consecutive ranges in member order, so that order is global in a group too.
//   k_band_count   the band's cubes per tile
//   k_tile_scan    each tile's first rank within the member, and the member's total (SLOT_BAND)
//   (a group: one more barrier, after which every member's SLOT_BAND is final)
//   k_band_take    the member's share: clamp(rem - (the band cubes of the members before it), 0, its own); every member
//                  adds the same total to SLOT_TAKEN
//   k_gather_capped  the cubes of rank < take, each at its rank in the list; tiles past the cap are left untouched,
//                  the tile that straddles it keeps its other cubes queued and gets its bound recomputed
// Compute, apply and mark are the uncapped round's kernels.
__global__ void __launch_bounds__(256) k_band_count(const LightParams P, uint32_t n_tiles, uint32_t *tile_count) {
    __shared__ uint32_t s_cnt[8];
    const uint32_t prio = P.scalars[SLOT_PRIORITY];
    const uint32_t n_words = (P.volume + 3) / 4;
    const uint32_t wl = gather_word_of_thread(P);
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t tm = P.tile_max[tile];
        if (prio <= P.epsilon_priority || tm <= P.epsilon_priority || tm + P.priority_band < prio) {   // (block-uniform)
            if (threadIdx.x == 0) tile_count[tile] = 0;
            continue;
        }
        const uint32_t w = tile * (LIGHT_TILE / 4) + wl;
        uint32_t cnt;
        band_select(P, w < n_words ? ((const uint32_t *)P.pending)[w] : 0u, w, prio, &cnt);
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = cnt;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0;
            for (int i = 0; i < 8; i++) t += s_cnt[i];
            tile_count[tile] = t;
        }
        __syncthreads();
    }
}

// One block of 1024 threads: off[i] = count[0] + ... + count[i - 1]; *total = the sum of all.
__global__ void __launch_bounds__(1024) k_tile_scan(const uint32_t *count, uint32_t *off, uint32_t n, uint32_t *total) {
    __shared__ uint32_t s_warp[32];
    const uint32_t per = (n + blockDim.x - 1) / blockDim.x;
    const uint32_t lo = min(threadIdx.x * per, n), hi = min(lo + per, n);
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += count[i];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = sum;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if ((int)lane >= o) inc += t;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const uint32_t v = lane < (blockDim.x >> 5) ? s_warp[lane] : 0u;
        uint32_t vi = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, vi, o);
            if ((int)lane >= o) vi += t;
        }
        s_warp[lane] = vi - v;
        if (lane == 31) *total = vi;
    }
    __syncthreads();
    uint32_t run = s_warp[wid] + inc - sum;
    for (uint32_t i = lo; i < hi; i++) {
        off[i] = run;
        run += count[i];
    }
}

// One thread.  Peers' SLOT_BAND are final: they were written before the barrier this kernel follows, and are written
// again only after the round's later barriers.
__global__ void k_band_take(const LightParams P, const GroupPeers G, uint32_t cap) {
    uint32_t before = 0, total = 0;
    for (uint32_t m = 0; m < G.n; m++) {
        const uint32_t c = *(volatile const uint32_t *)(G.scalars[m] + SLOT_BAND);
        if (m < G.self) before += c;
        total += c;
    }
    const uint32_t taken = P.scalars[SLOT_TAKEN];
    const uint32_t rem = cap > taken ? cap - taken : 0u;
    P.scalars[SLOT_LIST_LEN] = rem > before ? min(rem - before, P.scalars[SLOT_BAND]) : 0u;
    P.scalars[SLOT_TAKEN] = taken + min(rem, total);
}

__global__ void __launch_bounds__(256) k_gather_capped(const LightParams P, uint32_t n_tiles, const uint32_t *tile_off) {
    __shared__ uint32_t s_part[8], s_max[8];
    const uint32_t prio = P.scalars[SLOT_PRIORITY];
    if (prio <= P.epsilon_priority) return;
    const uint32_t take = P.scalars[SLOT_LIST_LEN];
    const uint32_t n_words = (P.volume + 3) / 4;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t wl = gather_word_of_thread(P);
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t tm = P.tile_max[tile];
        if (tm <= P.epsilon_priority || tm + P.priority_band < prio) continue;   // (block-uniform)
        const uint32_t first = tile_off[tile];
        if (first >= take) continue;   // past the cap (block-uniform)
        const uint32_t w = tile * (LIGHT_TILE / 4) + wl;
        uint32_t v = w < n_words ? ((uint32_t *)P.pending)[w] : 0u;
        uint32_t cnt;
        const uint32_t sel = band_select(P, v, w, prio, &cnt);
        uint32_t inc = cnt;
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
            if ((int)lane >= off) inc += t;
        }
        if (lane == 31) s_part[wid] = inc;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t total = 0;
            for (int i = 0; i < 8; i++) { const uint32_t c = s_part[i]; s_part[i] = total; total += c; }
        }
        __syncthreads();
        uint32_t at = first + s_part[wid] + inc - cnt;   // rank of the thread's first band cube
        uint32_t rest = 0;
        bool took = false;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) {
            const uint32_t p = (v >> (8 * k)) & 255u;
            if ((sel & (1u << k)) && at < take) {
                P.list[at++] = w * 4 + k;
                v &= ~(255u << (8 * k));
                took = true;
            } else {
                rest = max(rest, p);
            }
        }
        if (took) ((uint32_t *)P.pending)[w] = v;
        rest = __reduce_max_sync(0xffffffffu, rest);
        if (lane == 0) s_max[wid] = rest;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t m = 0;
            for (int i = 0; i < 8; i++) m = max(m, s_max[i]);
            P.tile_max[tile] = m;
        }
        __syncthreads();
    }
}

// The queue report of a step: queued cubes and their highest priority in the member's own tiles (after the merge, they
// hold the member's share of the queue), reading only the tiles whose bound is above 0.
__global__ void __launch_bounds__(256) k_queue_report(const LightParams P, const GroupPeers G) {
    const uint32_t lo = G.tile_lo[G.self], hi = G.tile_lo[G.self + 1];
    const uint32_t n_words = (P.volume + 3) / 4;
    for (uint32_t tile = lo + blockIdx.x; tile < hi; tile += gridDim.x) {
        if (P.tile_max[tile] == 0) continue;   // (block-uniform)
        const uint32_t w = tile * (LIGHT_TILE / 4) + threadIdx.x;
        const uint32_t v = w < n_words ? ((const uint32_t *)P.pending)[w] : 0u;
        uint32_t cnt = 0, m = 0;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) {
            const uint32_t p = (v >> (8 * k)) & 255u;
            cnt += p ? 1u : 0u;
            m = max(m, p);
        }
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        m = __reduce_max_sync(0xffffffffu, m);
        if ((threadIdx.x & 31) == 0 && cnt) {
            atomicAdd(P.scalars + SLOT_QUEUED, cnt);
            atomicMax(P.scalars + SLOT_QUEUE_MAX, m);
        }
    }
}

// ---- change tracking (aicb_light_take_changes): texels that differ from the baseline, per tile of LIGHT_TILE cubes
// (one block of 256 threads, 4 consecutive cubes per thread, so a tile's cubes are in index order) ----
__device__ __forceinline__ uint32_t diff_mask(const uint32_t *light, const uint32_t *base, uint32_t volume, uint32_t i0) {
    uint32_t mask = 0;
#pragma unroll
    for (uint32_t k = 0; k < 4; k++)
        if (i0 + k < volume && light[i0 + k] != base[i0 + k]) mask |= 1u << k;
    return mask;
}

__global__ void __launch_bounds__(256) k_diff_count(const uint32_t *light, const uint32_t *base, uint32_t volume,
                                                    uint32_t n_tiles, uint32_t *tile_count) {
    __shared__ uint32_t s_cnt[8];
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        uint32_t cnt = __popc(diff_mask(light, base, volume, tile * LIGHT_TILE + 4 * threadIdx.x));
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = cnt;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0;
            for (int i = 0; i < 8; i++) t += s_cnt[i];
            tile_count[tile] = t;
        }
        __syncthreads();
    }
}

// the records of the changed texels at their rank (tile_off = the scan of k_diff_count's counts), and the baseline of
// those cubes moved to the current light
__global__ void __launch_bounds__(256) k_diff_take(const DeviceScene S, uint32_t *base, uint32_t n_tiles,
                                                   const uint32_t *tile_count, const uint32_t *tile_off,
                                                   int32_t *cubes, uint32_t *texels) {
    __shared__ uint32_t s_part[8];
    const uint32_t volume = (uint32_t)S.size[0] * (uint32_t)S.size[1] * (uint32_t)S.size[2];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (tile_count[tile] == 0) continue;   // (block-uniform)
        const uint32_t i0 = tile * LIGHT_TILE + 4 * threadIdx.x;
        const uint32_t mask = diff_mask(S.light, base, volume, i0);
        const uint32_t cnt = __popc(mask);
        uint32_t inc = cnt;
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
            if ((int)lane >= off) inc += t;
        }
        if (lane == 31) s_part[wid] = inc;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t total = 0;
            for (int i = 0; i < 8; i++) { const uint32_t c = s_part[i]; s_part[i] = total; total += c; }
        }
        __syncthreads();
        uint32_t at = tile_off[tile] + s_part[wid] + inc - cnt;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) {
            if (!(mask & (1u << k))) continue;
            const uint32_t idx = i0 + k, t = S.light[idx];
            int x, y, z;
            cube_of(S, idx, x, y, z);
            cubes[3 * at] = x;
            cubes[3 * at + 1] = y;
            cubes[3 * at + 2] = z;
            texels[at] = t;
            base[idx] = t;
            at++;
        }
        __syncthreads();
    }
}

// Peer access between every pair of distinct member devices, with native atomics (k_group_guess); members on one
// device need neither.  Once per group.
aicb_status group_light_setup(aicb_group *g) {
    if (g->light_peers_ready) return AICB_OK;
    const size_t n = g->ctx.size();
    if (n > GROUP_LIGHT_MAX) return aicb_fail(AICB_ERR_UNSUPPORTED, "light propagation on a group of more than 16 members");
    for (size_t a = 0; a < n; a++)
        for (size_t b = 0; b < n; b++) {
            const int da = g->ctx[a]->device, db = g->ctx[b]->device;
            if (da == db) continue;
            int can = 0, atomics = 0;
            CU(cudaDeviceCanAccessPeer(&can, da, db));
            CU(cudaDeviceGetP2PAttribute(&atomics, cudaDevP2PAttrNativeAtomicSupported, da, db));
            if (!can || !atomics)
                return aicb_fail(AICB_ERR_UNSUPPORTED, "group light propagation needs peer access with native atomics between every pair of devices");
            CU(cudaSetDevice(da));
            cudaError_t e = cudaDeviceEnablePeerAccess(db, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
            if (e != cudaSuccess) return aicb_cuda_fail(e, "cudaDeviceEnablePeerAccess");
        }
    if (g->light_barrier.size() != n) {
        g->light_barrier.assign(n, nullptr);
        for (size_t i = 0; i < n; i++) {
            CU(cudaSetDevice(g->ctx[i]->device));
            CU(cudaEventCreateWithFlags(&g->light_barrier[i], cudaEventDisableTiming));
        }
    }
    g->light_peers_ready = true;
    return AICB_OK;
}

// evaluate_light (space.rs:1496-1527) over the members of a propagation: rounds until the highest queued priority is
// <= from_difference(epsilon).  One member runs the single-scene round; two or more members (the replicas of a device
// group `g`) run the sharded round above.  The caller holds every member's lock and has set up every member's light
// state.  Each member's light_stats are its own counters; `group_stats` (may be null) gets the updates and visits
// summed over the members, the rounds and the slowest member's device time.
// `step` (aicb_light_step; null for evaluate_light) adds the queue report and, with a cap below UINT64_MAX, runs capped
// rounds that stop once the step has taken `cap` cubes; a cap of 0 runs no round.
struct StepArgs {
    uint64_t cap;
    aicb_light_updates *out;   // filled on success (not null)
};
aicb_status relax(const std::vector<aicb_scene *> &members, aicb_group *g, uint8_t epsilon, uint64_t *group_stats,
                  uint64_t *updates_done, uint8_t *max_diff, uint64_t *node_visits, const StepArgs *step = nullptr) {
    const uint32_t n = (uint32_t)members.size();
    const bool sharded = n > 1;
    if (sharded) {
        const aicb_status st = group_light_setup(g);
        if (st != AICB_OK) return st;
    }
    const uint32_t n_tiles = (uint32_t)((members[0]->volume + LIGHT_TILE - 1) / LIGHT_TILE);
    std::vector<LightParams> P(n);
    std::vector<GroupPeers> G(n);   // (a single member's: its own tiles, for the step's kernels)
    {
        GroupPeers base;
        std::memset(&base, 0, sizeof base);
        base.n = n;
        for (uint32_t i = 0; i < n; i++) {
            aicb_scene *s = members[i];
            base.light[i] = s->d_light;
            base.pending[i] = s->d_pending;
            base.tile_max[i] = s->d_tile_max;
            base.scalars[i] = s->d_scalars;
            base.tile_lo[i] = (uint32_t)((uint64_t)n_tiles * i / n);
        }
        base.tile_lo[n] = n_tiles;
        for (uint32_t i = 0; i < n; i++) {
            G[i] = base;
            G[i].self = i;
        }
    }
    for (uint32_t i = 0; i < n; i++) P[i] = propagate_params(members[i], epsilon);
    const bool capped = step && step->cap != UINT64_MAX;
    const uint32_t cap = capped ? (uint32_t)(step->cap < 0xffffffffull ? step->cap : 0xffffffffull) : 0u;
    auto ctx = [&](uint32_t i) { return members[i]->ctx; };
    auto barrier = [&]() -> aicb_status {
        for (uint32_t i = 1; i < n; i++) {
            CU(cudaSetDevice(ctx(i)->device));
            CU(cudaEventRecord(g->light_barrier[i], ctx(i)->stream));
        }
        CU(cudaSetDevice(ctx(0)->device));
        for (uint32_t i = 1; i < n; i++) CU(cudaStreamWaitEvent(ctx(0)->stream, g->light_barrier[i], 0));
        CU(cudaEventRecord(g->light_barrier[0], ctx(0)->stream));
        for (uint32_t i = 1; i < n; i++) {
            CU(cudaSetDevice(ctx(i)->device));
            CU(cudaStreamWaitEvent(ctx(i)->stream, g->light_barrier[0], 0));
        }
        return AICB_OK;
    };
    // one step of every member, in member order, on the member's device and stream
    auto each = [&](auto &&step) -> aicb_status {
        for (uint32_t i = 0; i < n; i++) {
            aicb_ctx *c = ctx(i);
            CU(cudaSetDevice(c->device));
            const aicb_status r = step(i, c, c->stream, c->num_sms * 8);
            if (r != AICB_OK) return r;
        }
        return AICB_OK;
    };
#define RELAX_TRY(call)                          \
    do {                                         \
        const aicb_status r__ = (call);          \
        if (r__ != AICB_OK) return r__;          \
    } while (0)
    RELAX_TRY(each([&](uint32_t i, aicb_ctx *c, cudaStream_t cs, int blocks) -> aicb_status {
        CU(cudaEventRecord(c->ev0, cs));
        CU(cudaMemsetAsync(members[i]->d_scalars, 0, LIGHT_SCALARS * 4, cs));
        k_tile_rebuild<<<blocks, 256, 0, cs>>>(P[i], n_tiles);   // (fast_evaluate / edits write the priority bytes directly)
        return AICB_OK;
    }));
    const int ROUNDS_PER_SYNC = 8;
    uint64_t rounds = 0;
    std::vector<uint32_t> h(LIGHT_SCALARS * n);
    for (int batch = 0; batch < 100000 && !(capped && cap == 0); batch++) {
        for (int round = 0; round < ROUNDS_PER_SYNC; round++) {
            RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int) -> aicb_status {
                uint32_t *sc = members[i]->d_scalars;
                CU(cudaMemsetAsync(sc + SLOT_LIST_LEN, 0, (SLOT_PRIORITY - SLOT_LIST_LEN + 1) * 4, cs));
                CU(cudaMemsetAsync(sc + SLOT_CHANGED, 0, (SLOT_OVERFLOW - SLOT_CHANGED + 1) * 4, cs));
                k_find_max<<<16, 256, 0, cs>>>(P[i], n_tiles);
                return AICB_OK;
            }));
            if (sharded) RELAX_TRY(barrier());   // B1
            if (capped) {
                RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int blocks) -> aicb_status {
                    if (sharded) {
                        k_group_clear_foreign<<<blocks, 256, 0, cs>>>(P[i], G[i], n_tiles);
                        k_group_max<<<1, 32, 0, cs>>>(P[i], G[i]);
                    }
                    aicb_scene *s = members[i];
                    k_band_count<<<blocks, 256, 0, cs>>>(P[i], n_tiles, s->d_tile_count);
                    k_tile_scan<<<1, 1024, 0, cs>>>(s->d_tile_count, s->d_tile_off, n_tiles, s->d_scalars + SLOT_BAND);
                    return AICB_OK;
                }));
                if (sharded) RELAX_TRY(barrier());   // every member's SLOT_BAND is final
            }
            RELAX_TRY(each([&](uint32_t i, aicb_ctx *c, cudaStream_t cs, int blocks) -> aicb_status {
                if (capped) {
                    k_band_take<<<1, 1, 0, cs>>>(P[i], G[i], cap);
                    k_gather_capped<<<blocks, 256, 0, cs>>>(P[i], n_tiles, members[i]->d_tile_off);
                } else {
                    if (sharded) {
                        k_group_clear_foreign<<<blocks, 256, 0, cs>>>(P[i], G[i], n_tiles);
                        k_group_max<<<1, 32, 0, cs>>>(P[i], G[i]);
                    }
                    k_gather<<<blocks, 256, 0, cs>>>(P[i], n_tiles);
                }
                k_walk_chains<false><<<c->chain_walk_blocks, 128, 0, cs>>>(P[i], 0, nullptr);
                k_compute_overflow<<<blocks, 128, 0, cs>>>(P[i], nullptr);
                if (!sharded) k_apply<<<blocks, 128, 0, cs>>>(P[i]);   // apply and guess in one kernel
                return AICB_OK;
            }));
            if (sharded) {
                RELAX_TRY(barrier());   // B2
                RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int blocks) -> aicb_status {
                    k_group_apply<<<blocks, 128, 0, cs>>>(P[i], G[i]);
                    return AICB_OK;
                }));
                RELAX_TRY(barrier());   // B3
                RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int blocks) -> aicb_status {
                    k_group_guess<<<blocks, 128, 0, cs>>>(P[i], G[i]);
                    return AICB_OK;
                }));
                RELAX_TRY(barrier());   // B4
            }
            RELAX_TRY(each([&](uint32_t i, aicb_ctx *c, cudaStream_t cs, int blocks) -> aicb_status {
                if (sharded) k_group_broadcast<<<blocks, 128, 0, cs>>>(P[i], G[i]);
                k_compact_changed<<<blocks, 256, 0, cs>>>(P[i]);
                k_walk_chains<true><<<c->chain_walk_blocks, 128, 0, cs>>>(P[i], 0, nullptr);
                return AICB_OK;
            }));
            if (sharded) {
                RELAX_TRY(barrier());   // B5
                RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int blocks) -> aicb_status {
                    k_group_merge<<<blocks, 256, 0, cs>>>(P[i], G[i]);
                    return AICB_OK;
                }));
            }
        }
        RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int) -> aicb_status {
            CU(cudaMemcpyAsync(&h[LIGHT_SCALARS * i], members[i]->d_scalars, LIGHT_SCALARS * 4, cudaMemcpyDeviceToHost, cs));
            return AICB_OK;
        }));
        RELAX_TRY(each([&](uint32_t, aicb_ctx *, cudaStream_t cs, int) -> aicb_status {
            CU(cudaStreamSynchronize(cs));
            CU(cudaGetLastError());
            return AICB_OK;
        }));
        rounds += ROUNDS_PER_SYNC;
        // every member's round priority is the members' maximum
        const uint32_t prio = h[SLOT_PRIORITY];
        if (getenv("AICB_LIGHT_TRACE")) {
            uint64_t cubes = 0, updates = 0;
            for (uint32_t i = 0; i < n; i++) {
                cubes += h[LIGHT_SCALARS * i + SLOT_LIST_LEN];
                updates += h[LIGHT_SCALARS * i + SLOT_UPDATES];
            }
            fprintf(stderr, "[aicb200 light] batch %d: last round %llu cubes at priority %u; %llu updates so far\n", batch,
                    (unsigned long long)cubes, prio, (unsigned long long)updates);
        }
        if (prio <= P[0].epsilon_priority) break;   // the batch's last round found nothing above epsilon
        if (capped && h[SLOT_TAKEN] >= cap) break;   // the step's cap is used up
    }
    if (step) {
        RELAX_TRY(each([&](uint32_t i, aicb_ctx *, cudaStream_t cs, int blocks) -> aicb_status {
            k_queue_report<<<blocks, 256, 0, cs>>>(P[i], G[i]);
            CU(cudaMemcpyAsync(&h[LIGHT_SCALARS * i], members[i]->d_scalars, LIGHT_SCALARS * 4, cudaMemcpyDeviceToHost, cs));
            return AICB_OK;
        }));
    }
    uint64_t total = 0, visits = 0, slowest = 0, queued = 0;
    uint32_t maxd = 0, queue_max = 0;
    float slowest_ms = 0.0f;
    RELAX_TRY(each([&](uint32_t, aicb_ctx *c, cudaStream_t cs, int) -> aicb_status {
        CU(cudaEventRecord(c->ev1, cs));
        return AICB_OK;
    }));
    RELAX_TRY(each([&](uint32_t i, aicb_ctx *c, cudaStream_t, int) -> aicb_status {
        CU(cudaEventSynchronize(c->ev1));
        CU(cudaGetLastError());
        float ms = 0.0f;
        CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        slowest_ms = ms > slowest_ms ? ms : slowest_ms;
        aicb_scene *s = members[i];
        const uint32_t *hi = &h[LIGHT_SCALARS * i];
        s->light_stats[0] = hi[SLOT_UPDATES];
        s->light_stats[1] = (uint64_t)hi[SLOT_VISITS] | ((uint64_t)hi[SLOT_VISITS + 1] << 32);
        s->light_stats[2] = rounds;
        s->light_stats[3] = (uint64_t)(ms * 1000.0f);   // device time of the propagation in microseconds
        total += s->light_stats[0];
        visits += s->light_stats[1];
        slowest = s->light_stats[3] > slowest ? s->light_stats[3] : slowest;
        maxd = hi[SLOT_MAX_DIFF] > maxd ? hi[SLOT_MAX_DIFF] : maxd;
        queued += hi[SLOT_QUEUED];
        queue_max = hi[SLOT_QUEUE_MAX] > queue_max ? hi[SLOT_QUEUE_MAX] : queue_max;
        return AICB_OK;
    }));
#undef RELAX_TRY
    if (group_stats) {
        group_stats[0] = total;
        group_stats[1] = visits;
        group_stats[2] = rounds;
        group_stats[3] = slowest;
    }
    if (updates_done) *updates_done = total;
    if (max_diff) *max_diff = (uint8_t)maxd;
    if (node_visits) *node_visits = visits;
    if (step) {
        aicb_light_updates &o = *step->out;
        std::memset(&o, 0, sizeof o);
        o.update_count = total;
        o.queue_count = queued;
        o.chart_node_visits = visits;
        o.rounds = (uint32_t)rounds;
        o.max_update_difference = (uint8_t)maxd;
        o.max_queue_priority = (uint8_t)queue_max;
        o.device_ms = slowest_ms;
    }
    return AICB_OK;
}

// every member's lock, in member order, for the duration of a call
struct MemberLock {
    std::vector<std::unique_lock<std::mutex>> locks;
    explicit MemberLock(const std::vector<aicb_scene *> &members) {
        for (aicb_scene *s : members) locks.emplace_back(s->ctx->mu);
    }
};

// Mutation::set x n_edits (none for evaluate_light alone) on every member, then evaluate_light(epsilon): a single scene
// is a propagation of one member.  LightPhysics::None and invalid edits fail before any member changed.
// A step (max_updates not null: aicb_light_step) turns its time budget into an update cap with members[0]'s estimate of
// device microseconds per update, as update_light_from_queue turns the time left into a cost budget
// (updater.rs:197-203, 270-278), and refines the estimate afterwards.
aicb_status edit_and_relax(const std::vector<aicb_scene *> &members, aicb_group *g, const int32_t (*cubes)[3],
                           const uint16_t *new_ids, size_t n_edits, uint8_t epsilon, uint64_t *group_stats,
                           uint64_t *updates_done, uint8_t *max_diff, uint64_t *node_visits,
                           const uint64_t *max_updates = nullptr, double budget_us = -1.0, aicb_light_updates *out = nullptr) {
    if (budget_us != budget_us) return aicb_fail(AICB_ERR_INVALID, "budget_us is NaN");
    MemberLock lock(members);
    for (aicb_scene *s : members) {
        CU(cudaSetDevice(s->ctx->device));
        const aicb_status st = ensure_light_state(s);
        if (st != AICB_OK) return st;
    }
    std::vector<EditOp> ops;
    aicb_status st = edit_ops(members, cubes, new_ids, n_edits, &ops);
    if (st != AICB_OK) return st;
    for (aicb_scene *s : members) {
        CU(cudaSetDevice(s->ctx->device));
        st = apply_edit_ops(s, ops);
        if (st != AICB_OK) return st;
    }
    if (!max_updates) return relax(members, g, epsilon, group_stats, updates_done, max_diff, node_visits);
    aicb_scene *lead = members[0];
    uint64_t cap = *max_updates;
    if (budget_us >= 0.0) {
        const double c = std::floor(budget_us / lead->light_us_per_update);
        uint64_t by_time = c >= 1.8e19 ? UINT64_MAX - 1 : (uint64_t)c;
        if (budget_us > 0.0 && by_time == 0) by_time = 1;
        cap = by_time < cap ? by_time : cap;
    }
    aicb_light_updates info;
    const StepArgs step{cap, out ? out : &info};
    st = relax(members, g, epsilon, group_stats, updates_done, max_diff, node_visits, &step);
    if (st != AICB_OK) return st;
    // device microseconds per cube update, a running average with weight 1/8 per step
    const aicb_light_updates &r = *step.out;
    if (r.update_count > 0) {
        const double us = (double)r.device_ms * 1000.0 / (double)r.update_count;
        lead->light_us_per_update += (us - lead->light_us_per_update) / 8.0;
    }
    return AICB_OK;
}

// change tracking on one scene (a group: member 0); the caller holds the scene's lock
aicb_status track_changes(aicb_scene *s, int enable) {
    CU(cudaSetDevice(s->ctx->device));
    if (!enable) {
        if (s->d_light_base) {
            CU(cudaStreamSynchronize(s->ctx->stream));
            cudaFree(s->d_light_base);
            s->d_light_base = nullptr;
            s->device_bytes -= s->volume * 4;
        }
        if (s->d_changes) {
            cudaFree(s->d_changes);
            s->d_changes = nullptr;
            s->device_bytes -= s->changes_cap * 16;
            s->changes_cap = 0;
        }
        return AICB_OK;
    }
    const aicb_status st = ensure_light_state(s);
    if (st != AICB_OK) return st;
    if (!s->d_light_base) {
        CU(cudaMalloc(&s->d_light_base, s->volume * 4 + 16));
        s->device_bytes += s->volume * 4;
    }
    // ordered behind everything queued on the context's stream (cube deltas with light)
    CU(cudaMemcpyAsync(s->d_light_base, s->d_light, s->volume * 4, cudaMemcpyDeviceToDevice, s->ctx->stream));
    CU(cudaStreamSynchronize(s->ctx->stream));
    return AICB_OK;
}

aicb_status take_changes(aicb_scene *s, int32_t (*cubes)[3], uint8_t (*texels)[4], size_t cap, size_t *n_changed) {
    if (!s->d_light_base) return aicb_fail(AICB_ERR_INVALID, "light change tracking is not enabled");
    CU(cudaSetDevice(s->ctx->device));
    aicb_ctx *c = s->ctx;
    const uint32_t n_tiles = (uint32_t)((s->volume + LIGHT_TILE - 1) / LIGHT_TILE);
    const int blocks = c->num_sms * 8;
    k_diff_count<<<blocks, 256, 0, c->stream>>>(s->d_light, s->d_light_base, (uint32_t)s->volume, n_tiles, s->d_tile_count);
    k_tile_scan<<<1, 1024, 0, c->stream>>>(s->d_tile_count, s->d_tile_off, n_tiles, s->d_scalars + SLOT_DIFFS);
    uint32_t total = 0;
    CU(cudaMemcpyAsync(&total, s->d_scalars + SLOT_DIFFS, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaGetLastError());
    *n_changed = total;
    if (total == 0 || total > cap) return AICB_OK;
    if (s->changes_cap < total) {
        if (s->d_changes) {
            cudaFree(s->d_changes);
            s->device_bytes -= s->changes_cap * 16;
        }
        s->d_changes = nullptr;
        s->changes_cap = 0;
        const size_t want = total < 4096 ? 4096 : (size_t)total + total / 2;
        CU(cudaMalloc(&s->d_changes, want * 16));
        s->changes_cap = want;
        s->device_bytes += want * 16;
    }
    int32_t *d_cubes = (int32_t *)s->d_changes;
    uint32_t *d_texels = s->d_changes + 3 * s->changes_cap;
    k_diff_take<<<blocks, 256, 0, c->stream>>>(s->ds, s->d_light_base, n_tiles, s->d_tile_count, s->d_tile_off, d_cubes, d_texels);
    CU(cudaMemcpyAsync(cubes, d_cubes, (size_t)total * 12, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(texels, d_texels, (size_t)total * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaGetLastError());
    return AICB_OK;
}

}  // namespace

extern "C" {

aicb_status aicb_light_evaluate(aicb_scene *s, uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff,
                                uint64_t *node_visits) {
    if (!s) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return edit_and_relax({s}, nullptr, nullptr, nullptr, 0, epsilon, nullptr, updates_done, max_diff, node_visits);
}

// Mutation::set x n (space.rs:1346-1352 -> side_effects_of_set -> modified_cube_needs_update,
// updater.rs:135-173) applied in order on the host mirror, then evaluate_light(epsilon).
aicb_status aicb_light_edit_and_propagate(aicb_scene *s, const int32_t (*cubes)[3], const uint16_t *new_ids, size_t n_edits,
                                          uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff) {
    if (!s || (n_edits && (!cubes || !new_ids))) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return edit_and_relax({s}, nullptr, cubes, new_ids, n_edits, epsilon, nullptr, updates_done, max_diff, nullptr);
}

aicb_status aicb_group_light_fast_evaluate(aicb_group_scene *gs) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    for (aicb_scene *s : gs->scene) {   // every column is computed the same way on every replica
        aicb_status st = aicb_light_fast_evaluate(s);
        if (st != AICB_OK) return st;
    }
    return AICB_OK;
}

aicb_status aicb_group_light_evaluate(aicb_group_scene *gs, uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff,
                                      uint64_t *node_visits) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return edit_and_relax(gs->scene, gs->group, nullptr, nullptr, 0, epsilon, gs->light_stats, updates_done, max_diff,
                          node_visits);
}

aicb_status aicb_group_light_edit_and_propagate(aicb_group_scene *gs, const int32_t (*cubes)[3], const uint16_t *new_ids,
                                                size_t n_edits, uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff) {
    if (!gs || (n_edits && (!cubes || !new_ids))) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return edit_and_relax(gs->scene, gs->group, cubes, new_ids, n_edits, epsilon, gs->light_stats, updates_done, max_diff,
                          nullptr);
}

aicb_status aicb_light_step(aicb_scene *s, const int32_t (*cubes)[3], const uint16_t *new_ids, size_t n_edits,
                            uint8_t epsilon, uint64_t max_updates, double budget_us, aicb_light_updates *out) {
    if (!s || (n_edits && (!cubes || !new_ids))) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return edit_and_relax({s}, nullptr, cubes, new_ids, n_edits, epsilon, nullptr, nullptr, nullptr, nullptr, &max_updates,
                          budget_us, out);
}

aicb_status aicb_group_light_step(aicb_group_scene *gs, const int32_t (*cubes)[3], const uint16_t *new_ids,
                                  size_t n_edits, uint8_t epsilon, uint64_t max_updates, double budget_us,
                                  aicb_light_updates *out) {
    if (!gs || (n_edits && (!cubes || !new_ids))) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return edit_and_relax(gs->scene, gs->group, cubes, new_ids, n_edits, epsilon, gs->light_stats, nullptr, nullptr,
                          nullptr, &max_updates, budget_us, out);
}

aicb_status aicb_light_track_changes(aicb_scene *s, int enable) {
    if (!s) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lock(s->ctx->mu);
    return track_changes(s, enable);
}

aicb_status aicb_light_take_changes(aicb_scene *s, int32_t (*cubes)[3], uint8_t (*texels)[4], size_t cap,
                                    size_t *n_changed) {
    if (!s || !n_changed || (cap && (!cubes || !texels))) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lock(s->ctx->mu);
    return take_changes(s, cubes, texels, cap, n_changed);
}

aicb_status aicb_group_light_track_changes(aicb_group_scene *gs, int enable) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return aicb_light_track_changes(gs->scene[0], enable);
}

aicb_status aicb_group_light_take_changes(aicb_group_scene *gs, int32_t (*cubes)[3], uint8_t (*texels)[4], size_t cap,
                                          size_t *n_changed) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    return aicb_light_take_changes(gs->scene[0], cubes, texels, cap, n_changed);
}

aicb_status aicb_group_light_download(aicb_group_scene *gs, int member, uint8_t (*out)[4], size_t n_texels) {
    if (!gs) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    if (member < 0 || (size_t)member >= gs->scene.size()) return aicb_fail(AICB_ERR_INVALID, "member out of range");
    return aicb_light_download(gs->scene[member], out, n_texels);
}

aicb_status aicb_group_light_stats(const aicb_group_scene *gs, int member, uint64_t out[4]) {
    if (!gs || !out) return aicb_fail(AICB_ERR_INVALID, "NULL argument");
    if (member < -1 || member >= (int)gs->scene.size()) return aicb_fail(AICB_ERR_INVALID, "member out of range");
    const uint64_t *src = member < 0 ? gs->light_stats : gs->scene[member]->light_stats;
    for (int i = 0; i < 4; i++) out[i] = src[i];
    return AICB_OK;
}

}  // extern "C"
