// s4_tree.cu — S4: resolve the python renderer's tile quadtree on the device, then build every leaf's depth-ordered list.
//
// Reference semantics restated (not copied): gauss_render.py:290-344
//   BFS over tiles; a tile is skipped if w <= 1 or h <= 1 (:301), background-filled if no Gaussian overlaps it
//   (:313-315), split into TL, BL, TR, BR children if it holds more than max_gaussians_per_tile Gaussians or is wider /
//   taller than max_tile_size (:319-335), else rendered with its Gaussians ordered nearest-first (:340-344).
// Role of rasterizer_impl.cu:69-137,285-326 (duplicateWithKeys + 64-bit radix sort + identifyTileRanges) in the CUDA
// back-end of the reference; none of its structure is kept.
//
// Pipeline per camera (all sizes stay on the device; the host never waits for a count):
//   1. g2pc_depth_sort      one radix sort of N (depth key, value) pairs, value = (packed node range << 32 | Gaussian id)
//                           written by the preprocess kernel (cub::DeviceRadixSort, library call).
//   2. g2pc_build_tree      one CTA walks the levels top-down on the per-node overlap counts of the preprocess kernel,
//                           numbers the leaves in the reference's BFS order (level-major, then child-rank path order),
//                           lays out instance / pixel offsets, sorts the leaves heaviest-first for the blend and writes
//                           the frame header.  A frame that does not fit the caller's buffers (or needs a deeper table)
//                           sets the sticky POISON word: every later kernel of this and the following frames becomes a
//                           no-op until the host has read the header, fixed the sizes and replayed.
//   3. g2pc_multisplit      stable one-pass-per-chunk multisplit of the depth-ordered stream into the leaves' lists:
//        count    CTA c takes 256 consecutive sorted entries and counts its instances per leaf (shared-memory histogram)
//        scan     per leaf, exclusive prefix over the chunks (+ the leaf's list offset)          -> matrix[c][leaf]
//        scatter  CTA c marks bit (leaf, k) for every instance in a shared-memory bit matrix (order-free atomicOr); an
//                 instance's place is matrix[c][leaf] + the set bits of its leaf before bit k (popc): the lists come out
//                 depth-ordered without any sort of the ~7 N instances (the round-1 path emitted (leaf, id) pairs and
//                 ran a 2-pass 20 M-pair radix sort per camera).  Splats that cover many tiles are walked by the whole
//                 warp (colour_common.cuh warp_for_each_node).
#include <cub/cub.cuh>
#include "colour_common.cuh"

namespace {

constexpr int TB = 1024;
constexpr int SORT_CAP = 4096;  // leaves sorted heaviest-first in shared memory (more leaves: launch order = BFS order)

struct TreeParams {
    QtMeta meta;
    QtTables tab;
    int32_t n1;
    uint32_t* node_cnt;      // read, then cleared for the next frame
    uint8_t* node_state;
    int32_t* node_leaf;      // per node: leaf id, -1 (no leaf: empty / absent / dropped) or -2 (split)
    g2pc_leaf_t* leaves;
    int32_t* leaf_order;     // leaves sorted by descending work (longest-processing-time-first launch order)
    int32_t max_leaves;
    int64_t inst_capacity, pix_capacity, matrix_capacity;
    int32_t ms_chunks;
    int32_t frame;
    int32_t* header;         // G2PC_HDR_WORDS
    uint32_t* fail;          // shared failure word (colour_common.cuh)
    int32_t* work_counters;  // G2PC_WORK_COUNTERS ints, cleared here for the blend of this frame
    int32_t nodes_2d;
};

// key (BFS rank within a level: child rank = 2*xbit + ybit per level, most significant first) -> (ix, iy)
__device__ __forceinline__ void deinterleave(int key, int level, int& ix, int& iy) {
    ix = 0; iy = 0;
    for (int b = 0; b < level; ++b) {
        iy |= ((key >> (2 * b)) & 1) << b;
        ix |= ((key >> (2 * b + 1)) & 1) << b;
    }
}

__global__ void __launch_bounds__(TB) tree_kernel(const TreeParams p) {
    __shared__ int s_warp[33];
    __shared__ int s_flags[2];
    __shared__ unsigned long long s_sort[SORT_CAP];
    if (g2pc_frame_skipped(p.fail, p.frame)) {  // this or an earlier frame failed: report and do nothing
        report_skipped_frame(p.fail, p.frame, p.header);
        return;
    }
    const int L = p.meta.num_levels;
    if (threadIdx.x == 0) { s_flags[0] = 0; s_flags[1] = 0; }
    __syncthreads();
    int leaf_base = 0;
    long long inst_total = 0;
    for (int l = 0; l < L; ++l) {
        const int nn = 1 << (2 * l);
        const int o1 = (1 << l) - 1, o2 = off2(l);
        for (int k0 = 0; k0 < nn; k0 += TB) {
            const int key = k0 + threadIdx.x;
            int is_leaf = 0, node = -1, ix = 0, iy = 0;
            uint32_t cnt = 0;
            if (key < nn) {
                deinterleave(key, l, ix, iy);
                node = o2 + (iy << l) + ix;
                bool exists = (l == 0);
                if (l > 0) {
                    const int pnode = off2(l - 1) + ((iy >> 1) << (l - 1)) + (ix >> 1);
                    exists = p.node_state[pnode] == NODE_SPLIT;
                }
                uint8_t st = NODE_NONE;
                int32_t nl = -1;
                if (exists) {
                    const int fx = p.tab.xf[o1 + ix], fy = p.tab.yf[o1 + iy];
                    if (!((fx | fy) & QT_FLAG_DROPPED)) {
                        cnt = p.node_cnt[node];
                        // cnt: exact on the leaf-candidate levels, a non-empty flag above them (a node larger than
                        // max_tile_size splits whatever it holds — unless it is empty: then it is background and has
                        // no children, gauss_render.py:313-335)
                        const bool big = ((fx | fy) & QT_FLAG_BIG) != 0;
                        if (cnt == 0) st = NODE_EMPTY;
                        else if (big || cnt > (uint32_t)p.meta.max_gaussians_per_tile) {
                            st = NODE_SPLIT;
                            nl = -2;
                            if (l == L - 1) { st = NODE_NONE; nl = -1; s_flags[0] = 1; }  // deeper than the tabulated levels
                        } else {
                            st = NODE_LEAF;
                            is_leaf = 1;
                        }
                    }
                }
                p.node_state[node] = st;
                p.node_leaf[node] = nl;
            }
            int tot;
            const int pre = block_scan(is_leaf, s_warp, tot);
            if (is_leaf) {
                const int li = leaf_base + pre;
                if (li < p.max_leaves) {
                    g2pc_leaf_t lf;
                    lf.r0 = p.tab.ys[o1 + iy];
                    lf.c0 = p.tab.xs[o1 + ix];
                    lf.w = p.tab.xe[o1 + ix] - lf.c0 + 1;
                    lf.h = p.tab.ye[o1 + iy] - lf.r0 + 1;
                    lf.inst_begin = 0;
                    lf.inst_count = (int32_t)cnt;
                    lf.pix_offset = 0;
                    lf.node = node;
                    p.leaves[li] = lf;
                    p.node_leaf[node] = li;
                } else {
                    s_flags[1] = 1;
                }
            }
            leaf_base += tot;
        }
        __syncthreads();  // node_state of level l visible to level l+1
    }
    const int nl = leaf_base < p.max_leaves ? leaf_base : p.max_leaves;
    // exclusive scans of the instance counts and pixel counts over the leaves, in order
    int pix_base = 0;
    for (int k0 = 0; k0 < nl; k0 += TB) {
        const int i = k0 + threadIdx.x;
        int c = 0, a = 0;
        // every list starts on a 16-byte boundary (the blend stages id chunks with TMA bulk copies): pad to 4 ids
        if (i < nl) { c = (p.leaves[i].inst_count + 3) & ~3; a = p.leaves[i].w * p.leaves[i].h; }
        int tc, ta;
        const int pc = block_scan(c, s_warp, tc);
        const int pa = block_scan(a, s_warp, ta);
        if (i < nl) {
            // 32-bit list offsets: a frame with more than 2^31 instances is reported through the capacity check below
            p.leaves[i].inst_begin = (int32_t)(inst_total + pc);
            p.leaves[i].pix_offset = pix_base + pa;
        }
        inst_total += tc;
        pix_base += ta;
    }
    __syncthreads();
    // launch order for the blend: heaviest leaves first (instances x pixels, ties by index) — bitonic sort in smem
    if (nl <= SORT_CAP) {
        int m = 1;
        while (m < nl) m <<= 1;
        for (int i = threadIdx.x; i < m; i += TB) {
            unsigned long long key = ~0ull;
            if (i < nl) {
                unsigned long long w = (unsigned long long)p.leaves[i].inst_count *
                                       (unsigned long long)(p.leaves[i].w * p.leaves[i].h);
                w = w < (1ull << 44) - 1ull ? w : (1ull << 44) - 1ull;
                key = (((1ull << 44) - 1ull - w) << 16) | (unsigned long long)i;  // ascending key = descending work
            }
            s_sort[i] = key;
        }
        __syncthreads();
        bitonic_sort<TB>(s_sort, m);
        for (int i = threadIdx.x; i < nl; i += TB) p.leaf_order[i] = (int)(s_sort[i] & 0xFFFFull);
    } else {
        for (int i = threadIdx.x; i < nl; i += TB) p.leaf_order[i] = i;
    }
    // the counts are consumed: clear them for the next frame's preprocess
    for (int k = threadIdx.x; k < p.nodes_2d; k += TB) p.node_cnt[k] = 0u;
    if (threadIdx.x < G2PC_WORK_COUNTERS) p.work_counters[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        const int cap_over = (inst_total > p.inst_capacity || (long long)pix_base > p.pix_capacity ||
                              (long long)p.ms_chunks * (long long)nl > p.matrix_capacity || inst_total > 0x7FFFFFFFll)
                             // (ms_chunks = rows the multisplit needs: chunks + segments, g2pc_multisplit_rows)
                                 ? 1 : 0;
        write_frame_header(p.header, p.fail, p.frame, leaf_base, inst_total, pix_base, s_flags[0], s_flags[1], cap_over);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Multisplit.  An entry of the sorted stream is (range << 32 | gid); its leaves are enumerated from the packed node range
// at the base level; Gaussians that touch a split node re-derive their rect from the projection record and query the
// deeper candidate levels (count-driven splits only — rare).
struct MsParams {
    const unsigned long long* val_sorted;
    int64_t n;
    const float4* proj;
    int32_t width, height;
    QtMeta meta;
    QtTables tab;
    int32_t n1;
    uint32_t level_mask;
    int32_t base_level;
    const int32_t* node_leaf;
    const int32_t* header;
    const uint32_t* fail;
    int32_t frame;
    const g2pc_leaf_t* leaves;
    uint32_t* matrix;      // [chunk][num_leaves]: counts, then absolute list offsets (in place)
    uint32_t* inst_gid;
    int32_t leaf_cap;      // leaves the shared-memory tables are sized for (<= max_leaves of the tree)
    int32_t base_clean;    // the base level has no dropped / degenerate node: membership = the packed range, no table look-ups
    uint32_t clean_mask;   // the same, per level
    int32_t grid_w;        // > 0: flat tile grid (s7_tiles.cu): leaf = iy * grid_w + ix, the packed range is the tile rect
};

// f(leaf, owner_lane, owner_gid) for every leaf the lane's entry overlaps; warp-cooperative (all 32 lanes must call).
template <typename F>
__device__ __forceinline__ void for_each_leaf(const MsParams& p, const QtTables& T, const int32_t* __restrict__ s_leaf,
                                              uint32_t range, uint32_t gid, F f) {
    if (p.grid_w > 0) {
        warp_for_each_node(range, gid, [&](int ix, int iy, int owner, uint32_t og) { f(iy * p.grid_w + ix, owner, og); });
        return;
    }
    const int lb = p.base_level;
    const int o1 = (1 << lb) - 1;
    unsigned deeper = 0;
    if (p.base_clean) {
        warp_for_each_node(range, gid, [&](int ix, int iy, int owner, uint32_t og) {
            const int32_t v = s_leaf[(iy << lb) + ix];
            if (v >= 0) f(v, owner, og);
            else if (v == -2) deeper |= 1u << owner;
        });
    } else {
        warp_for_each_node(range, gid, [&](int ix, int iy, int owner, uint32_t og) {
            if (!axis_member(T.ys + o1, T.ye + o1, T.yf + o1, iy) || !axis_member(T.xs + o1, T.xe + o1, T.xf + o1, ix)) return;
            const int32_t v = s_leaf[(iy << lb) + ix];
            if (v >= 0) f(v, owner, og);
            else if (v == -2) deeper |= 1u << owner;
        });
    }
    if (p.meta.num_levels <= lb + 1) return;
    int xlo, xhi, ylo, yhi;
    g2pc_unpack_range(range, xlo, xhi, ylo, yhi);
    // ---- count-driven splits below the base level ----
    // Rare at 1280 px; at 1920 px with 6 M Gaussians most of the sphere's base nodes split two levels down (C5: 150 M
    // instances per camera, almost all from here), so the deeper levels get the same warp-cooperative walk as the base
    // level (per-lane loops with per-node table checks ran at 5 of 32 threads: 69 + 13 ms per camera, ncu r02g).
    // combine the flags raised on behalf of each owner
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) deeper |= __shfl_xor_sync(0xffffffffu, deeper, o);
    const int lane = threadIdx.x & 31;
    bool mine = (deeper >> lane) & 1u;
    if (!mine && xlo <= xhi) {
        // a child tile may overhang its parent by a pixel to the right / below (children are ceil(size / 2) wide): a
        // Gaussian can sit in a deeper leaf of the base node just left of / above its own base range
        const int ex = max(xlo - 1, 0), ey = max(ylo - 1, 0);
        for (int iy = ey; iy <= yhi; ++iy)
            for (int ix = ex; ix <= xhi; ++ix)
                if ((iy < ylo || ix < xlo) && s_leaf[(iy << lb) + ix] == -2) mine = true;
    }
    if (!__any_sync(0xffffffffu, mine)) return;
    float x0 = 0.f, x1 = 0.f, y0 = 0.f, y1 = 0.f;
    if (mine) {
        const float4 q0 = __ldg(p.proj + 3 * (int64_t)gid);
        const float4 q2 = __ldg(p.proj + 3 * (int64_t)gid + 2);
        gaussian_rect(q0.x, q0.y, q2.z, p.width, p.height, x0, x1, y0, y1);
    }
    const float isx0 = 1.0f / (float)p.width, isy0 = 1.0f / (float)p.height;
    for (int l = lb + 1; l < p.meta.num_levels; ++l) {  // (uniform)
        if (!((p.level_mask >> l) & 1u)) continue;
        const int ol = (1 << l) - 1;
        int axlo = 1, axhi = 0, aylo = 1, ayhi = 0;
        if (mine) {
            axis_range(T.xs + ol, T.xe + ol, l, x0, x1, isx0 * (float)(1 << l), axlo, axhi);
            if (axlo <= axhi) axis_range(T.ys + ol, T.ye + ol, l, y0, y1, isy0 * (float)(1 << l), aylo, ayhi);
        }
        const bool some = axlo <= axhi && aylo <= ayhi;
        const int32_t* nl = p.node_leaf + off2(l);
        if (((p.clean_mask >> l) & 1u) && l <= G2PC_RANGE_MAX_LEVEL) {
            // no dropped / degenerate node at this level: membership = the range; cooperative walk
            const uint32_t rl = some ? g2pc_pack_range(axlo, axhi, aylo, ayhi) : (uint32_t)G2PC_RANGE_EMPTY;
            warp_for_each_node(rl, gid, [&](int ix, int iy, int owner, uint32_t og) {
                const int32_t v = __ldg(nl + (iy << l) + ix);
                if (v >= 0) f(v, owner, og);
            });
            continue;
        }
        if (!some) continue;
        for (int iy = aylo; iy <= ayhi; ++iy) {
            if (!axis_member(T.ys + ol, T.ye + ol, T.yf + ol, iy)) continue;
            for (int ix = axlo; ix <= axhi; ++ix) {
                if (!axis_member(T.xs + ol, T.xe + ol, T.xf + ol, ix)) continue;
                const int32_t v = __ldg(nl + (iy << l) + ix);
                if (v >= 0) f(v, lane, gid);
            }
        }
    }
}

// shared memory of the count / scatter kernels: [6 * n1 table ints][4^base node->leaf ints][payload]
__device__ __forceinline__ int32_t* ms_load_common(const MsParams& p, int32_t* smem, QtTables& T) {
    if (p.grid_w > 0) { T = p.tab; return smem; }  // tile grid: nothing to stage
    if (p.base_clean && p.meta.num_levels <= p.base_level + 1) {
        T = p.tab;  // never dereferenced: no table look-up at a clean base level, no deeper level
        __syncthreads();
    } else {
        T = load_tables(p.tab, p.n1, smem);  // ends with __syncthreads()
    }
    int32_t* s_leaf = smem + 6 * p.n1;
    const int nb = 1 << (2 * p.base_level);
    const int32_t* src = p.node_leaf + off2(p.base_level);
    for (int i = threadIdx.x; i < nb; i += blockDim.x) s_leaf[i] = src[i];
    return s_leaf;
}

// count:   matrix[c][leaf] = instances of `leaf` in chunk c (one CTA per chunk of C sorted entries)
// scan:    per leaf, exclusive prefix over the chunks + the leaf's list offset (three small kernels, 32 x 32 tiles)
// scatter: position = matrix[c][leaf] + rank inside the chunk (bit matrix)
template <int C>
__global__ void __launch_bounds__(C) ms_count_kernel(const MsParams p) {
    extern __shared__ int32_t smem_ms[];
    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int nl = p.header[G2PC_HDR_NUM_LEAVES];
    QtTables T;
    int32_t* s_leaf = ms_load_common(p, smem_ms, T);
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(s_leaf + (p.grid_w > 0 ? 0 : (1 << (2 * p.base_level))));
    for (int i = threadIdx.x; i < nl; i += C) s_hist[i] = 0u;
    __syncthreads();
    const int64_t k = (int64_t)blockIdx.x * C + threadIdx.x;
    unsigned long long v = (unsigned long long)G2PC_RANGE_EMPTY << 32;
    if (k < p.n) v = p.val_sorted[k];
    for_each_leaf(p, T, s_leaf, (uint32_t)(v >> 32), (uint32_t)v,
                  [&](int leaf, int, uint32_t) { atomicAdd(s_hist + leaf, 1u); });
    __syncthreads();
    uint32_t* row = p.matrix + (int64_t)blockIdx.x * nl;
    for (int i = threadIdx.x; i < nl; i += C) row[i] = s_hist[i];
}

// Column-wise exclusive scan of matrix (rows x num_leaves) in three steps over tiles of 1024 rows x 32 leaves:
//   partial: tile sums -> tile_sum[tile_row][leaf];  blocks: per leaf, scan of the tile sums + the leaf's list offset;
//   apply: every tile rewrites its rows as running offsets.
constexpr int SCAN_ROWS = 1024;  // rows per tile (32 per thread)
__global__ void __launch_bounds__(1024) ms_scan_partial_kernel(const MsParams p, int32_t rows) {
    __shared__ uint32_t s_sum[32][33];
    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int nl = p.header[G2PC_HDR_NUM_LEAVES];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int leaf = blockIdx.x * 32 + tx;
    if (blockIdx.x * 32 >= nl) return;
    const int r0 = blockIdx.y * SCAN_ROWS + ty * 32;
    uint32_t sum = 0;
    if (leaf < nl) {
#pragma unroll 8
        for (int r = r0; r < min(rows, r0 + 32); ++r) sum += p.matrix[(int64_t)r * nl + leaf];
    }
    s_sum[ty][tx] = sum;
    __syncthreads();
    if (ty == 0 && leaf < nl) {
        uint32_t t = 0;
#pragma unroll
        for (int s = 0; s < 32; ++s) t += s_sum[s][tx];
        uint32_t* tile_sum = p.matrix + (int64_t)rows * nl;  // appended behind the rows
        tile_sum[(int64_t)blockIdx.y * nl + leaf] = t;
    }
}

__global__ void __launch_bounds__(256) ms_scan_blocks_kernel(const MsParams p, int32_t rows, int32_t tiles) {
    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int nl = p.header[G2PC_HDR_NUM_LEAVES];
    const int leaf = blockIdx.x * 256 + threadIdx.x;
    if (leaf >= nl) return;
    uint32_t* tile_sum = p.matrix + (int64_t)rows * nl;
    uint32_t run = (uint32_t)p.leaves[leaf].inst_begin;
    for (int t = 0; t < tiles; ++t) {
        const uint32_t v = tile_sum[(int64_t)t * nl + leaf];
        tile_sum[(int64_t)t * nl + leaf] = run;
        run += v;
    }
}

__global__ void __launch_bounds__(1024) ms_scan_apply_kernel(const MsParams p, int32_t rows) {
    __shared__ uint32_t s_sum[32][33];
    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int nl = p.header[G2PC_HDR_NUM_LEAVES];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int leaf = blockIdx.x * 32 + tx;
    if (blockIdx.x * 32 >= nl) return;
    const int r0 = blockIdx.y * SCAN_ROWS + ty * 32, r1 = min(rows, r0 + 32);
    uint32_t v[32];
    uint32_t sum = 0;
#pragma unroll
    for (int q = 0; q < 32; ++q) {
        v[q] = (leaf < nl && r0 + q < r1) ? p.matrix[(int64_t)(r0 + q) * nl + leaf] : 0u;
        sum += v[q];
    }
    s_sum[ty][tx] = sum;
    __syncthreads();
    if (leaf >= nl) return;
    const uint32_t* tile_sum = p.matrix + (int64_t)rows * nl;
    uint32_t run = tile_sum[(int64_t)blockIdx.y * nl + leaf];
    for (int s = 0; s < ty; ++s) run += s_sum[s][tx];
#pragma unroll
    for (int q = 0; q < 32; ++q) {
        if (r0 + q < r1) p.matrix[(int64_t)(r0 + q) * nl + leaf] = run;
        run += v[q];
    }
}

template <int C>
__global__ void __launch_bounds__(C) ms_scatter_kernel(const MsParams p) {
    extern __shared__ int32_t smem_ms[];
    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int nl = p.header[G2PC_HDR_NUM_LEAVES];
    constexpr int WORDS = C / 32;
    QtTables T;
    int32_t* s_leaf = ms_load_common(p, smem_ms, T);
    uint32_t* s_row = reinterpret_cast<uint32_t*>(s_leaf + (p.grid_w > 0 ? 0 : (1 << (2 * p.base_level))));  // [nl]
    uint32_t* s_bits = s_row + p.leaf_cap;                                                                   // [WORDS][nl]
    {
        // the chunk's list offsets (one coalesced row of the matrix) and a zeroed bit matrix; 16-byte stores where the
        // carve-up allows (leaf_cap is a multiple of 4 and the dynamic smem base is 16-byte aligned)
        const uint32_t* grow = p.matrix + (int64_t)blockIdx.x * nl;
        for (int i = threadIdx.x; i < nl; i += C) s_row[i] = grow[i];
        if (((reinterpret_cast<uintptr_t>(s_bits) & 15) == 0) && ((nl & 3) == 0)) {
            uint4* b4 = reinterpret_cast<uint4*>(s_bits);
            for (int i = threadIdx.x; i < WORDS * nl / 4; i += C) b4[i] = make_uint4(0u, 0u, 0u, 0u);
        } else {
            for (int i = threadIdx.x; i < WORDS * nl; i += C) s_bits[i] = 0u;
        }
    }
    __syncthreads();
    const int w = threadIdx.x >> 5;  // the warp = the 32-entry group of the chunk
    uint32_t* mybits = s_bits + w * nl;
    const int64_t k = (int64_t)blockIdx.x * C + threadIdx.x;
    unsigned long long v = (unsigned long long)G2PC_RANGE_EMPTY << 32;
    if (k < p.n) v = p.val_sorted[k];
    const uint32_t range = (uint32_t)(v >> 32), gid = (uint32_t)v;
    // 1. mark (leaf, k) in the bit matrix: order-free
    for_each_leaf(p, T, s_leaf, range, gid, [&](int leaf, int owner, uint32_t) { atomicOr(mybits + leaf, 1u << owner); });
    __syncthreads();
    // 2. every instance finds its place: the chunk's offset for the leaf, the instances of the same leaf in earlier
    //    32-entry groups of the chunk, then the earlier lanes of its own group (bit order = depth order)
    for_each_leaf(p, T, s_leaf, range, gid, [&](int leaf, int owner, uint32_t og) {
        uint32_t pos = s_row[leaf] + (uint32_t)__popc(mybits[leaf] & ((1u << owner) - 1u));
        for (int w2 = 0; w2 < w; ++w2) pos += (uint32_t)__popc(s_bits[w2 * nl + leaf]);
        p.inst_gid[pos] = og;
    });
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

template <int C>
int launch_multisplit(const MsParams& p, int32_t chunks, cudaStream_t st) {
    const size_t common = p.grid_w > 0 ? 0 : ((size_t)6 * p.n1 + ((size_t)1 << (2 * p.base_level))) * sizeof(int32_t);
    const size_t smem_count = common + (size_t)p.leaf_cap * sizeof(uint32_t);
    const size_t smem_scatter = common + (size_t)(C / 32 + 1) * p.leaf_cap * sizeof(uint32_t);
    if (smem_scatter > 200 * 1024 || smem_count > 200 * 1024) {
        g2pc_set_error("g2pc_multisplit: shared memory budget exceeded");
        return G2PC_ERR_INVALID;
    }
    if (smem_count > 48 * 1024)
        G2PC_CUDA(cudaFuncSetAttribute(ms_count_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_count));
    if (smem_scatter > 48 * 1024)
        G2PC_CUDA(cudaFuncSetAttribute(ms_scatter_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_scatter));
    ms_count_kernel<C><<<(unsigned)chunks, C, smem_count, st>>>(p);
    G2PC_CHECK_LAUNCH();
    const int tiles = (chunks + SCAN_ROWS - 1) / SCAN_ROWS;
    const dim3 sgrid((unsigned)((p.leaf_cap + 31) / 32), (unsigned)tiles);
    ms_scan_partial_kernel<<<sgrid, 1024, 0, st>>>(p, chunks);
    G2PC_CHECK_LAUNCH();
    ms_scan_blocks_kernel<<<(unsigned)((p.leaf_cap + 255) / 256), 256, 0, st>>>(p, chunks, tiles);
    G2PC_CHECK_LAUNCH();
    ms_scan_apply_kernel<<<sgrid, 1024, 0, st>>>(p, chunks);
    G2PC_CHECK_LAUNCH();
    ms_scatter_kernel<C><<<(unsigned)chunks, C, smem_scatter, st>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

}  // namespace

extern "C" int g2pc_build_tree(const int32_t* tables, int32_t num_levels, int32_t max_gaussians_per_tile,
                               uint32_t* node_cnt, uint8_t* node_state, int32_t* node_leaf, g2pc_leaf_t* leaves,
                               int32_t* leaf_order, int32_t max_leaves, int64_t inst_capacity, int64_t pix_capacity,
                               int64_t matrix_capacity, int32_t ms_chunks, int32_t frame, int32_t* header,
                               uint32_t* fail, int32_t* work_counters, void* stream) {
    G2PC_CHECK_ARG(tables && node_cnt && node_state && node_leaf && leaves && leaf_order && header && fail &&
                       work_counters, "null pointer");
    G2PC_CHECK_ARG(num_levels >= 1 && num_levels <= G2PC_MAX_LEVELS && max_leaves >= 1, "bad sizes");
    G2PC_CHECK_ARG(frame >= 0 && ms_chunks >= 0, "bad frame / chunk count");
    TreeParams p;
    p.meta.num_levels = num_levels; p.meta.max_gaussians_per_tile = max_gaussians_per_tile;
    p.n1 = (1 << num_levels) - 1;
    p.tab = make_tables(tables, p.n1);
    p.node_cnt = node_cnt; p.node_state = node_state; p.node_leaf = node_leaf; p.leaves = leaves;
    p.leaf_order = leaf_order; p.max_leaves = max_leaves;
    p.inst_capacity = inst_capacity; p.pix_capacity = pix_capacity; p.matrix_capacity = matrix_capacity;
    p.ms_chunks = ms_chunks; p.frame = frame; p.header = header; p.fail = fail; p.work_counters = work_counters;
    p.nodes_2d = ((1 << (2 * num_levels)) - 1) / 3;
    tree_kernel<<<1, TB, 0, (cudaStream_t)stream>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

// workspace layout of g2pc_depth_sort: [keys_out n u32][cub temp]
extern "C" int64_t g2pc_depth_sort_workspace_bytes(int64_t n) {
    size_t sort_b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_b, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (const unsigned long long*)nullptr, (unsigned long long*)nullptr, n);
    return (int64_t)(align256((size_t)n * 4) + align256(sort_b));
}

/* Sort the (depth key, value) pairs by key (stable: ties keep index order) -> val_sorted[k] = value of the k-th nearest
 * Gaussian. */
extern "C" int g2pc_depth_sort(const uint32_t* depth_key, const uint64_t* val, int64_t n, uint64_t* val_sorted,
                               void* workspace, int64_t workspace_bytes, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(depth_key && val && val_sorted && workspace, "null pointer");
    G2PC_CHECK_ARG(workspace_bytes >= g2pc_depth_sort_workspace_bytes(n), "workspace too small");
    char* ws = (char*)workspace;
    uint32_t* keys_out = (uint32_t*)ws;
    void* tmp = ws + align256((size_t)n * 4);
    size_t b = (size_t)workspace_bytes - align256((size_t)n * 4);
    G2PC_CUDA(cub::DeviceRadixSort::SortPairs(tmp, b, depth_key, keys_out, (const unsigned long long*)val,
                                              (unsigned long long*)val_sorted, n, 0, 32, (cudaStream_t)stream));
    return G2PC_OK;
}

extern "C" int32_t g2pc_multisplit_chunk(int32_t leaf_cap) {
    // entries per chunk: the scatter kernel keeps leaf_cap x (chunk bits + one offset) in shared memory.  Prefer a
    // footprint that lets 3 CTAs share an SM (the kernel is a chain of short latency-bound phases: with one resident CTA
    // per SM the 3600-tile grid of the CUDA back-end ran 3.5x slower per instance than the 1024 leaves of the python one)
    const int64_t n = leaf_cap;
    if (n * 36 <= 74 * 1024) return 256;
    if (n * 20 <= 74 * 1024) return 128;
    if (n * 12 <= 110 * 1024) return 64;
    if (n * 20 <= 200 * 1024) return 128;
    if (n * 12 <= 200 * 1024) return 64;
    return 0;
}

extern "C" int32_t g2pc_multisplit_rows(int64_t n, int32_t leaf_cap) {
    // matrix rows the multisplit needs for n entries: one per chunk + one per scan tile of 1024 chunks
    const int C = g2pc_multisplit_chunk(leaf_cap);
    if (C <= 0) return 0;
    const int32_t chunks = (int32_t)((n + C - 1) / C);
    return chunks + (chunks + SCAN_ROWS - 1) / SCAN_ROWS;
}

extern "C" int g2pc_multisplit(const uint64_t* val_sorted, int64_t n, const void* proj, int32_t width, int32_t height,
                               const int32_t* tables, int32_t num_levels, uint32_t level_mask, uint32_t clean_mask,
                               const int32_t* node_leaf,
                               const g2pc_leaf_t* leaves, const int32_t* header, const uint32_t* fail, int32_t frame,
                               int32_t leaf_cap, uint32_t* matrix, uint32_t* inst_gid, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(val_sorted && proj && tables && node_leaf && leaves && header && fail && matrix && inst_gid,
                   "null pointer");
    G2PC_CHECK_ARG(num_levels >= 1 && num_levels <= G2PC_MAX_LEVELS && level_mask != 0u, "bad levels");
    const int C = g2pc_multisplit_chunk(leaf_cap);
    G2PC_CHECK_ARG(C > 0, "too many leaves for the multisplit");
    MsParams p;
    p.val_sorted = (const unsigned long long*)val_sorted; p.n = n; p.proj = (const float4*)proj;
    p.width = width; p.height = height;
    p.meta.num_levels = num_levels; p.meta.max_gaussians_per_tile = 0;
    p.n1 = (1 << num_levels) - 1;
    p.tab = make_tables(tables, p.n1);
    p.level_mask = level_mask; p.base_level = __builtin_ctz(level_mask);
    G2PC_CHECK_ARG(p.base_level <= G2PC_RANGE_MAX_LEVEL, "first leaf-candidate level too deep");
    p.node_leaf = node_leaf; p.header = header; p.fail = fail; p.frame = frame; p.leaves = leaves; p.matrix = matrix;
    p.inst_gid = inst_gid;
    p.leaf_cap = leaf_cap; p.grid_w = 0;
    p.base_clean = (int32_t)((clean_mask >> p.base_level) & 1u);
    p.clean_mask = clean_mask;
    const int32_t chunks = (int32_t)((n + C - 1) / C);
    cudaStream_t st = (cudaStream_t)stream;
    if (C == 256) return launch_multisplit<256>(p, chunks, st);
    if (C == 128) return launch_multisplit<128>(p, chunks, st);
    return launch_multisplit<64>(p, chunks, st);
}

/* The same multisplit over a flat grid of tiles (s7_tiles.cu): leaf = tile index, the packed range is the tile rect. */
extern "C" int g2pc_multisplit_grid(const uint64_t* val_sorted, int64_t n, int32_t grid_w, int32_t grid_h,
                                    const g2pc_leaf_t* leaves, const int32_t* header, const uint32_t* fail,
                                    int32_t frame, int32_t leaf_cap, uint32_t* matrix, uint32_t* inst_gid, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(val_sorted && leaves && header && fail && matrix && inst_gid, "null pointer");
    G2PC_CHECK_ARG(grid_w >= 1 && grid_h >= 1 && grid_w <= 256 && grid_h <= 256 && leaf_cap >= grid_w * grid_h,
                   "bad tile grid / leaf_cap");
    const int C = g2pc_multisplit_chunk(leaf_cap);
    G2PC_CHECK_ARG(C > 0, "too many tiles for the multisplit");
    MsParams p;
    p.val_sorted = (const unsigned long long*)val_sorted; p.n = n; p.proj = nullptr;
    p.width = 0; p.height = 0;
    p.meta.num_levels = 1; p.meta.max_gaussians_per_tile = 0;
    p.n1 = 0;
    p.tab.xs = p.tab.xe = p.tab.xf = p.tab.ys = p.tab.ye = p.tab.yf = nullptr;
    p.level_mask = 1u; p.base_level = 0;
    p.node_leaf = nullptr; p.header = header; p.fail = fail; p.frame = frame; p.leaves = leaves; p.matrix = matrix;
    p.inst_gid = inst_gid;
    p.leaf_cap = leaf_cap; p.grid_w = grid_w; p.base_clean = 1; p.clean_mask = 1u;
    const int32_t chunks = (int32_t)((n + C - 1) / C);
    cudaStream_t st = (cudaStream_t)stream;
    if (C == 256) return launch_multisplit<256>(p, chunks, st);
    if (C == 128) return launch_multisplit<128>(p, chunks, st);
    return launch_multisplit<64>(p, chunks, st);
}
