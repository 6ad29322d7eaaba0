// s7_tiles.cu — the colour stage with the semantics of the reference's CUDA back-end (renderer_type="cuda"):
// fixed 16x16 tiles, near cull z <= 0.2, radius ceil(3 sigma), alpha < 1/255 skipped, a pixel stops at T < 1e-4, depth /
// inverse-depth images, per-pixel mask, per-Gaussian max contribution + arg-max pixel, per-Gaussian minimum distance to
// the predicted surface.
//
// Reference semantics restated (not copied):
//   forward.cu:153-271      preprocessCUDA   (in_frustum auxiliary.h:151-176, computeCov2D :76-111, getRect auxiliary.h:45-55)
//   rasterizer_impl.cu:69-137,285-326        duplicateWithKeys / radix sort / identifyTileRanges  -> per-tile depth-ordered lists
//   forward.cu:303-497      renderCUDA       (blend, max contribution :434-456, surface distance :460-477, mask :334,389,485)
//   gaussian_pointcloud_rasterization/__init__.py:126-158   per-camera accumulator updates
// Nothing of their structure is kept: the depth-ordered lists come from the same depth sort + bit-matrix multisplit as the
// python-semantics path (s4_tree.cu), built per SUPER-TILE of 2x2 tiles (32x32 pixels: 900 lists at 1280x720 instead of
// 3600 — the multisplit's cost grows with the number of lists); the blend of a tile walks its super-tile's list and skips
// the entries whose tile rect (packed into the projection record) does not contain the tile, so every tile still sees
// exactly its own list, in order, and the 256-entry rounds of the surface distance count the tile's own entries;
// the blend is a persistent kernel with TMA-staged id chunks and cp.async record gathers (scalar FP32: the per-pixel keep /
// stop predicates of these semantics do not pack into FP32x2), and every cross-thread reduction is a deterministic max / min (the reference's shared-memory CAS loop, its racing
// `largest_collected_contribution_pixel` store and its non-atomic cross-block updates make its results run-dependent —
// SURVEY.md §2.1).  Deterministic definition of the surface distance (SURVEY.md §8a): after every round of 256 list entries
// of a tile, dist(j) = min over the tile's pixel threads of |depth_j - E_p| with E_p the thread's running un-normalised
// expected depth (threads outside the image hold 0, masked pixels have left the loop), min over tiles and cameras — the
// value the reference's racy compare-and-store aims at.
#include "colour_common.cuh"

namespace {

constexpr int TILE = 16;

struct TilePreParams {
    const float4* geom;    // packed geometry (g2pc_pack_geometry)
    const float* colours;  // (n,3) f32 or null
    const float* shs;      // SH coefficients or null
    int32_t sh_stride, sh_degree, sh_layout;  // layout 0: (n,3,stride) channel-major; 1: (n,stride,3) coefficient-major
    int64_t n;
    float view[16], projm[16], campos[3];
    float tan_fovx, tan_fovy, focal_x, focal_y;
    int32_t W, H, gx, gy, sgx, sgy;  // tile grid, super-tile grid
    float4* proj;
    uint32_t* node_cnt;    // per super-tile
    uint32_t* depth_key;
    unsigned long long* val;
    int32_t* radii;        // (n) int32 or null
    int32_t use_hist;
};

__device__ __forceinline__ float3 sh_eval(const float* __restrict__ sh, int stride, int layout, int deg, float3 d) {
    float out[3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
        out[c] = sh_channel(deg, d, [&](int k) { return layout == 0 ? __ldg(sh + c * stride + k) : __ldg(sh + 3 * k + c); });
    return make_float3(out[0], out[1], out[2]);
}

__global__ void __launch_bounds__(256) preprocess_tiles_kernel(const TilePreParams p) {
    extern __shared__ uint32_t s_hist_t[];
    const int ntiles = p.sgx * p.sgy;
    if (p.use_hist) {
        for (int k = threadIdx.x; k < ntiles; k += blockDim.x) s_hist_t[k] = 0u;
        __syncthreads();
    }
    const int64_t base = (int64_t)blockIdx.x * 1024;
    for (int it = 0; it < 4; ++it) {
        const int64_t i = base + it * 256 + threadIdx.x;
        if (base + it * 256 >= p.n) break;             // uniform: the whole CTA is past the end
        const int64_t il = i < p.n ? i : p.n - 1;      // lanes past the end shadow the last Gaussian and write nothing
        const float4 g0 = __ldg(p.geom + 3 * il), g1 = __ldg(p.geom + 3 * il + 1), g2 = __ldg(p.geom + 3 * il + 2);
        const float* V = p.view;
        const float* M = p.projm;
        const float px_ = g0.x, py_ = g0.y, pz_ = g0.z;
        // p_view = [p,1] * viewmatrix (z forward), near cull (auxiliary.h:151-176)
        const float vx = V[0] * px_ + V[4] * py_ + V[8] * pz_ + V[12];
        const float vy = V[1] * px_ + V[5] * py_ + V[9] * pz_ + V[13];
        const float vz = V[2] * px_ + V[6] * py_ + V[10] * pz_ + V[14];
        float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0, q2 = q0;
        uint32_t range = G2PC_RANGE_EMPTY;
        int radius_out = 0;
        bool ok = (vz > 0.2f) && (i < p.n);
        int rx0 = 1, rx1 = 1, ry0 = 1, ry1 = 1;  // tile rect [rx0, rx1) x [ry0, ry1)
        if (ok) {
            const float hx = M[0] * px_ + M[4] * py_ + M[8] * pz_ + M[12];
            const float hy = M[1] * px_ + M[5] * py_ + M[9] * pz_ + M[13];
            const float hw = M[3] * px_ + M[7] * py_ + M[11] * pz_ + M[15];
            const float pw = 1.0f / (hw + 0.0000001f);
            const float ndx = hx * pw, ndy = hy * pw;
            // EWA covariance (forward.cu:76-111): cov = Jm Wc Sigma Wc^T Jm^T, Wc[r][c] = V[4c + r]
            const float limx = 1.3f * p.tan_fovx, limy = 1.3f * p.tan_fovy;
            const float tx = fminf(limx, fmaxf(-limx, vx / vz)) * vz;
            const float ty = fminf(limy, fmaxf(-limy, vy / vz)) * vz;
            const float ja = p.focal_x / vz, jb = -(p.focal_x * tx) / (vz * vz);
            const float jc = p.focal_y / vz, jd = -(p.focal_y * ty) / (vz * vz);
            float Mr[2][3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Mr[0][c] = ja * V[4 * c + 0] + jb * V[4 * c + 2];
                Mr[1][c] = jc * V[4 * c + 1] + jd * V[4 * c + 2];
            }
            const float S[9] = {g0.w, g1.x, g1.y, g1.x, g1.z, g1.w, g1.y, g1.w, g2.x};
            float A[2][3];
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int c = 0; c < 3; ++c) A[r][c] = Mr[r][0] * S[c] + Mr[r][1] * S[3 + c] + Mr[r][2] * S[6 + c];
            float ca = A[0][0] * Mr[0][0] + A[0][1] * Mr[0][1] + A[0][2] * Mr[0][2];
            const float cb = A[0][0] * Mr[1][0] + A[0][1] * Mr[1][1] + A[0][2] * Mr[1][2];
            float cc = A[1][0] * Mr[1][0] + A[1][1] * Mr[1][1] + A[1][2] * Mr[1][2];
            ca += 0.3f; cc += 0.3f;  // low-pass dilation (forward.cu:217-220)
            const float det = ca * cc - cb * cb;
            ok = det != 0.0f;
            if (ok) {
                const float det_inv = 1.0f / det;
                const float kx = cc * det_inv, ky = -cb * det_inv, kz = ca * det_inv;
                const float mid = 0.5f * (ca + cc);
                const float root = sqrtf(fmaxf(0.1f, mid * mid - det));
                const float my_radius = ceilf(3.0f * sqrtf(fmaxf(mid + root, mid - root)));
                // ndc2Pix is evaluated in double in the reference (auxiliary.h:40-43)
                const float pix_x = (float)((((double)ndx + 1.0) * (double)p.W - 1.0) * 0.5);
                const float pix_y = (float)((((double)ndy + 1.0) * (double)p.H - 1.0) * 0.5);
                const int ir = (int)my_radius;
                rx0 = min(p.gx, max(0, (int)((pix_x - ir) / TILE)));
                ry0 = min(p.gy, max(0, (int)((pix_y - ir) / TILE)));
                rx1 = min(p.gx, max(0, (int)((pix_x + ir + TILE - 1) / TILE)));
                ry1 = min(p.gy, max(0, (int)((pix_y + ir + TILE - 1) / TILE)));
                ok = (rx1 - rx0) * (ry1 - ry0) != 0;
                if (ok) {
                    float3 rgb;
                    if (p.shs) {
                        const float dx = px_ - p.campos[0], dy = py_ - p.campos[1], dz = pz_ - p.campos[2];
                        const float inv = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
                        rgb = sh_eval(p.shs + (int64_t)il * 3 * p.sh_stride, p.sh_stride, p.sh_layout, p.sh_degree,
                                      make_float3(dx * inv, dy * inv, dz * inv));
                    } else {
                        rgb = make_float3(p.colours[3 * il], p.colours[3 * il + 1], p.colours[3 * il + 2]);
                    }
                    // power = -0.5 (kx dx^2 + kz dy^2) - ky dx dy, evaluated by the blend as exp2 of K' terms
                    const float K = -0.72134752044448170368f;  // -0.5 log2(e)
                    q0 = make_float4(pix_x, pix_y, kx * K, 2.0f * ky * K);
                    q1 = make_float4(kz * K, g2.y, rgb.x, rgb.y);
                    // q2.w carries the packed TILE rect (the blend's membership filter)
                    q2 = make_float4(rgb.z, vz, my_radius,
                                     __uint_as_float(g2pc_pack_range(rx0, rx1 - 1, ry0, ry1 - 1)));
                    radius_out = ir;
                    range = g2pc_pack_range(rx0 >> 1, (rx1 - 1) >> 1, ry0 >> 1, (ry1 - 1) >> 1);  // super-tiles
                }
            }
        }
        // Gaussians per tile; large rects are walked by the whole warp (all 32 lanes reach this point)
        warp_for_each_node(range, 0u, [&](int tx_, int ty_, int, uint32_t) {
                               if (p.use_hist) atomicAdd(s_hist_t + ty_ * p.sgx + tx_, 1u);
                               else atomicAdd(p.node_cnt + ty_ * p.sgx + tx_, 1u);
                           });
        if (i < p.n) {
            float4* rec = p.proj + 3 * i;
            rec[0] = q0; rec[1] = q1; rec[2] = q2;
            p.depth_key[i] = ok ? __float_as_uint(vz) : 0xFFFFFFFFu;
            p.val[i] = ((unsigned long long)range << 32) | (unsigned long long)(uint32_t)i;
            if (p.radii) p.radii[i] = radius_out;
        }
    }
    if (p.use_hist) {
        __syncthreads();
        for (int k = threadIdx.x; k < ntiles; k += blockDim.x) {
            const uint32_t v = s_hist_t[k];
            if (v) atomicAdd(p.node_cnt + k, v);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// List table (one CTA): every super-tile is a "leaf" (leaf index = super-tile index, row-major; the leaf rectangle is its
// 32x32 pixels clipped to the image), lists padded to 16 bytes, heaviest first in the launch order, frame header + poison
// exactly as g2pc_build_tree.
constexpr int TB = 1024;
constexpr int SORT_CAP = 8192;

struct TileTreeParams {
    uint32_t* node_cnt;
    g2pc_leaf_t* leaves;
    int32_t* leaf_order;
    int32_t W, H, gx, gy, max_leaves;
    int64_t inst_capacity, matrix_capacity;
    int32_t ms_rows, frame;
    int32_t* header;
    uint32_t* fail;
    int32_t* work_counters;
};

__global__ void __launch_bounds__(TB) tile_tree_kernel(const TileTreeParams p) {
    __shared__ int s_warp[33];
    __shared__ uint32_t s_sort[SORT_CAP];  // (2^19 - 1 - min(count, 2^19 - 1)) << 13 | tile
    if (g2pc_frame_skipped(p.fail, p.frame)) {
        report_skipped_frame(p.fail, p.frame, p.header);
        return;
    }
    const int nt = p.gx * p.gy;  // (gx, gy = super-tile grid here)
    const int nl = nt < p.max_leaves ? nt : p.max_leaves;
    long long inst_total = 0;
    for (int k0 = 0; k0 < nl; k0 += TB) {
        const int i = k0 + threadIdx.x;
        int cnt = 0;
        if (i < nl) cnt = (int)p.node_cnt[i];
        int tc;
        const int pc = block_scan((cnt + 3) & ~3, s_warp, tc);
        if (i < nl) {
            const int ty = i / p.gx, tx = i - ty * p.gx;
            g2pc_leaf_t lf;
            lf.r0 = ty * 2 * TILE; lf.c0 = tx * 2 * TILE;
            lf.w = min(2 * TILE, p.W - lf.c0); lf.h = min(2 * TILE, p.H - lf.r0);
            lf.inst_begin = (int32_t)(inst_total + pc);
            lf.inst_count = cnt;
            lf.pix_offset = 0;
            lf.node = i;
            p.leaves[i] = lf;
        }
        inst_total += tc;
    }
    __syncthreads();
    if (nl <= SORT_CAP) {
        int m = 1;
        while (m < nl) m <<= 1;
        for (int i = threadIdx.x; i < m; i += TB) {
            uint32_t key = 0xFFFFFFFFu;
            if (i < nl) key = ((0x7FFFFu - min(p.node_cnt[i], 0x7FFFFu)) << 13) | (uint32_t)i;
            s_sort[i] = key;
        }
        __syncthreads();
        bitonic_sort<TB>(s_sort, m);
        for (int i = threadIdx.x; i < nl; i += TB) p.leaf_order[i] = (int)(s_sort[i] & 0x1FFFu);
    } else {
        for (int i = threadIdx.x; i < nl; i += TB) p.leaf_order[i] = i;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < nt; k += TB) p.node_cnt[k] = 0u;
    if (threadIdx.x < G2PC_WORK_COUNTERS) p.work_counters[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        const int leaf_over = nt > p.max_leaves ? 1 : 0;
        const int cap_over = (inst_total > p.inst_capacity || (long long)p.ms_rows * (long long)nl > p.matrix_capacity ||
                              inst_total > 0x7FFFFFFFll) ? 1 : 0;
        write_frame_header(p.header, p.fail, p.frame, nt, inst_total, p.W * p.H, 0, leaf_over, cap_over);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Blend: one super-tile (2x2 tiles of 16x16 pixels) per work item, 256 threads: tile s = warps 2s, 2s+1, a thread blends a
// row quad of its tile.  Chunks of 128 list entries go through the same 3-deep pipeline as s5_blend.cu (TMA bulk copy of
// the ids, cp.async gather of the records, blend); the records are fetched once per super-tile and every tile skips the
// entries whose tile rect does not contain it (a warp-uniform branch), so each tile blends exactly its own depth-ordered
// list.  The surface-distance rounds (256 entries of the TILE's list) are counted per tile and flushed with a 64-thread
// named barrier.
constexpr int TBT = 256;
constexpr int TCH = 128;

struct TileBlendParams {
    const g2pc_leaf_t* leaves;
    const int32_t* leaf_order;
    const int32_t* header;
    const uint32_t* fail;
    int32_t frame;
    const uint32_t* inst_gid;
    const float4* proj;
    unsigned long long* cam_best;
    uint32_t* cam_dist;        // per Gaussian: bits of the minimum surface distance of this camera (init FLT_MAX) or null
    const int32_t* mask;       // per pixel (H*W) int32, 0 = ignore, or null
    float* out_color;          // (3,H,W)
    float* out_depth;          // (H,W)
    float* out_invdepth;       // (H,W)
    int32_t W, H;
    float bg[3];
    int32_t* work_counter;
    unsigned long long* stats;
};

__device__ __forceinline__ void pair_sync(int tile) {  // the two warps of one tile (static ids: a register id makes
    switch (tile) {                                     // ptxas reserve all 16 barriers and caps the CTAs per SM)
        case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
        case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
        case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
        default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
    }
}

template <bool SURF>
__global__ void __launch_bounds__(TBT, SURF ? 3 : 4) blend_tiles_kernel(const TileBlendParams p) {
    __shared__ __align__(16) float4 s_q0[2][TCH];
    __shared__ __align__(16) float4 s_q1[2][TCH];
    __shared__ __align__(16) float4 s_q2[2][TCH];  // (blue, depth, radius, packed tile rect)
    __shared__ __align__(16) uint32_t s_gid[3][TCH];
    __shared__ unsigned long long s_best[TBT / 32][TCH];
    __shared__ __align__(8) unsigned long long s_bar[3];
    __shared__ int s_item;
    __shared__ float s_E[SURF ? 4 : 1][SURF ? 256 : 1];       // expected depths of a tile's threads, sorted per round
    __shared__ float s_rdepth[SURF ? 4 : 1][SURF ? 256 : 1];  // depths / ids of the tile's current round
    __shared__ uint32_t s_rgid[SURF ? 4 : 1][SURF ? 256 : 1];
    __shared__ int s_pair_live[SURF ? 4 : 1][2];

    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int num_items = p.header[G2PC_HDR_NUM_LEAVES];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tile = tid >> 6, tt = tid & 63;  // tile of the super-tile, thread of the tile
    if (tid == 0) {
        mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_init(&s_bar[2], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int w = 0; w < TBT / 32; ++w)
        for (int t = tid; t < TCH; t += TBT) s_best[w][t] = 0ull;
    uint32_t phase_bits = 0;
    unsigned long long iters = 0;
    __syncthreads();

  for (;;) {
    if (tid == 0) s_item = atomicAdd(p.work_counter, 1);
    __syncthreads();
    const int item = s_item;
    __syncthreads();
    if (item >= num_items) break;
    const g2pc_leaf_t lf = p.leaves[p.leaf_order[item]];
    const int tc0 = lf.c0 + (tile & 1) * TILE, tr0 = lf.r0 + (tile >> 1) * TILE;  // the tile's origin
    const int tw = max(0, min(TILE, p.W - tc0)), th = max(0, min(TILE, p.H - tr0));
    const uint32_t tix = (uint32_t)(tc0 / TILE), tiy = (uint32_t)(tr0 / TILE);
    const int row = tt >> 2, x0 = (tt & 3) * 4;
    const int gy_ = tr0 + row;
    const bool row_in = row < th;
    // per pixel: inside the image and not masked out -> live; `live` drops to 0 when the pixel stops (T would fall below 1e-4)
    float live[4], T[4], Cr[4], Cg[4], Cb[4], D[4], ID[4], px[4];
    bool valid[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool inside = row_in && (x0 + i < tw);
        bool m = inside;
        if (inside && p.mask) m = p.mask[(int64_t)gy_ * p.W + tc0 + x0 + i] != 0;
        valid[i] = m;
        live[i] = m ? 1.0f : 0.0f;
        T[i] = 1.0f; Cr[i] = Cg[i] = Cb[i] = D[i] = ID[i] = 0.0f;
        px[i] = (float)(tc0 + x0 + i);
    }
    const float py = (float)gy_;
    const int pix_base = gy_ * p.W + tc0 + x0;
    const bool tile_has_outside = (tw < TILE) || (th < TILE);

    const int cnt = lf.inst_count;
    const int nchunks = (cnt + TCH - 1) / TCH;
    const uint32_t* list = p.inst_gid + (int64_t)lf.inst_begin;

    auto issue_ids = [&](int c) {
        const int nl = min(TCH, cnt - c * TCH);
        tma_load_1d(&s_gid[c % 3][0], list + (int64_t)c * TCH, (uint32_t)(((nl + 3) & ~3) * 4), &s_bar[c % 3]);
    };
    auto wait_ids = [&](int c) {
        const int s = c % 3;
        mbar_wait(&s_bar[s], (phase_bits >> s) & 1u);
        phase_bits ^= 1u << s;
    };
    auto issue_records = [&](int c) {
        const int nl = min(TCH, cnt - c * TCH);
        if (tid < nl) {
            const float4* rec = p.proj + 3 * (int64_t)s_gid[c % 3][tid];
            cp_async16(&s_q0[c & 1][tid], rec);
            cp_async16(&s_q1[c & 1][tid], rec + 1);
            cp_async16(&s_q2[c & 1][tid], rec + 2);
        }
        cp_async_commit();
    };
    // end of a round of the tile's list (forward.cu:460-477): distance of every entry of the round to the nearest running
    // expected depth among the tile's 256 threads.  Sort the values once, then binary-search per entry.  Both warps of
    // the tile call this at the same entry.
    auto flush_round = [&](int nround) {
        float* E = s_E[SURF ? tile : 0];
#pragma unroll
        for (int i = 0; i < 4; ++i) E[tt * 4 + i] = valid[i] ? D[i] : 3.0e38f;
        pair_sync(tile);
        for (int k = 2; k <= 256; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tt; i < 256; i += 64) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const float a = E[i], b = E[ixj];
                        const bool up = (i & k) == 0;
                        if ((a > b) == up) { E[i] = b; E[ixj] = a; }
                    }
                }
                pair_sync(tile);
            }
        for (int t = tt; t < nround; t += 64) {
            const float d = s_rdepth[SURF ? tile : 0][t];
            int lo = 0, hi = 256;  // first index with E >= d
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (E[mid] < d) lo = mid + 1; else hi = mid; }
            float best = 3.0e38f;
            if (lo < 256 && E[lo] < 1.0e38f) best = fabsf(E[lo] - d);
            if (lo > 0 && E[lo - 1] < 1.0e38f) best = fminf(best, fabsf(d - E[lo - 1]));
            if (tile_has_outside) best = fminf(best, fabsf(d));  // threads outside the image hold expected depth 0
            if (best < 1.0e38f) atomicMin(p.cam_dist + s_rgid[SURF ? tile : 0][t], __float_as_uint(best));
        }
        pair_sync(tile);
    };

    bool warp_done = false;   // no live pixel left in this warp
    bool tile_left = (tw == 0) || (th == 0);  // the tile has left its list (or lies outside the image)
    int members = 0;          // entries of the tile's own list seen so far
    if (nchunks > 0) {
        if (tid == 0) { issue_ids(0); if (nchunks > 1) issue_ids(1); }
        wait_ids(0);
        issue_records(0);
    }
    for (int c = 0; c < nchunks; ++c) {
        const int nload = min(TCH, cnt - c * TCH);
        const bool more = (c + 1 < nchunks);
        if (more) { wait_ids(c + 1); issue_records(c + 1); }
        if (more) cp_async_wait<1>(); else cp_async_wait<0>();
        const bool all_left = __syncthreads_and((SURF ? tile_left : (tile_left || warp_done)) ? 1 : 0);
        if (all_left) {
            if (more) cp_async_wait<0>();
            break;
        }
        if (tid == 0 && c + 2 < nchunks) issue_ids(c + 2);
        const float4* q0s = s_q0[c & 1];
        const float4* q1s = s_q1[c & 1];
        const float4* q2s = s_q2[c & 1];
        const uint32_t* gids = s_gid[c % 3];
        if (SURF ? !tile_left : !(tile_left || warp_done)) {
            for (int j = 0; j < nload; ++j) {
                const float4 q2 = q2s[j];
                const uint32_t rect = __float_as_uint(q2.w);
                // the tile's own list = the entries whose tile rect contains it (warp-uniform)
                if (tix - (rect & 255u) > ((rect >> 8) & 255u) - (rect & 255u) ||
                    tiy - ((rect >> 16) & 255u) > (rect >> 24) - ((rect >> 16) & 255u))
                    continue;
                if (SURF) {
                    // the reference leaves a tile when all its threads are done at the START of a round (forward.cu:366-369)
                    if ((members & 255) == 0 && members > 0) {
                        const float lmax = fmaxf(fmaxf(live[0], live[1]), fmaxf(live[2], live[3]));
                        const bool warp_live = __any_sync(FULLM, lmax != 0.0f);
                        if (lane == 0) s_pair_live[tile][warp & 1] = warp_live ? 1 : 0;
                        pair_sync(tile);
                        const bool any_live = (s_pair_live[tile][0] | s_pair_live[tile][1]) != 0;
                        pair_sync(tile);
                        if (!any_live) { tile_left = true; break; }
                    }
                    if ((warp & 1) == 0 && lane == 0) {
                        s_rdepth[tile][members & 255] = q2.y;
                        s_rgid[tile][members & 255] = gids[j];
                    }
                }
                ++members;
                if (!warp_done) {
                    const float4 q0 = q0s[j];
                    const float4 q1 = q1s[j];
                    const float dy = py - q0.y;
                    const float Bq = dy * q0.w;
                    const float Cq = dy * dy * q1.x;           // power' without the opacity term
                    const float depth = q2.y, idepth = 1.0f / q2.y;
                    float c4[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float dx = px[i] - q0.x;
                        const float pw = fmaf(dx, fmaf(dx, q0.z, Bq), Cq);  // = power * log2(e)
                        const float alpha = fminf(0.99f, ex2f(pw + q1.y));
                        // power > 0 -> skip; alpha < 1/255 -> skip (forward.cu:404,412)
                        const bool keep = !(pw > 0.0f) && !(alpha < (1.0f / 255.0f));
                        const float cand = T[i] * alpha;
                        const float testT = T[i] * (1.0f - alpha);
                        // the pixel stops BEFORE taking a contribution that would leave T < 1e-4 (forward.cu:414-419)
                        if (keep && testT < 0.0001f) live[i] = 0.0f;
                        const float cc = (keep ? cand : 0.0f) * live[i];
                        const bool take = keep && (live[i] != 0.0f);
                        T[i] = take ? testT : T[i];
                        Cr[i] = fmaf(cc, q1.z, Cr[i]);
                        Cg[i] = fmaf(cc, q1.w, Cg[i]);
                        Cb[i] = fmaf(cc, q2.x, Cb[i]);
                        D[i] = fmaf(cc, depth, D[i]);
                        ID[i] = fmaf(cc, idepth, ID[i]);
                        c4[i] = cc;
                    }
                    const float v = fmaxf(fmaxf(c4[0], c4[1]), fmaxf(c4[2], c4[3]));
                    if (__any_sync(FULLM, v > 0.0f)) {
                        const uint32_t vb = __float_as_uint(v);
                        const uint32_t wm = __reduce_max_sync(FULLM, vb);
                        const int i = (c4[0] == v) ? 0 : (c4[1] == v) ? 1 : (c4[2] == v) ? 2 : 3;
                        const uint32_t pk = (vb == wm) ? (0xFFFFFFFFu - (uint32_t)(pix_base + i)) : 0u;
                        const uint32_t wp = __reduce_max_sync(FULLM, pk);
                        if (lane == 0) s_best[warp][j] = ((unsigned long long)wm << 32) | (unsigned long long)wp;
                    }
                    ++iters;
                }
                if (SURF && (members & 255) == 0) flush_round(256);
            }
            if (!warp_done) {
                const float lmax = fmaxf(fmaxf(live[0], live[1]), fmaxf(live[2], live[3]));
                warp_done = __all_sync(FULLM, lmax == 0.0f);
            }
        }
        __syncthreads();
        // one atomic per entry for the whole super-tile: the best (contribution, pixel) over its warps.  (Tried: every
        // warp straight to the global maximum and a single barrier per chunk — 10 % slower on C4.)
        for (int t = tid; t < nload; t += TBT) {
            unsigned long long best = s_best[0][t];
            s_best[0][t] = 0ull;
#pragma unroll
            for (int w = 1; w < TBT / 32; ++w) {
                const unsigned long long o = s_best[w][t];
                s_best[w][t] = 0ull;
                best = o > best ? o : best;
            }
            if ((best >> 32) != 0ull) atomicMax(p.cam_best + gids[t], best);
        }
    }
    if (SURF && !tile_left && (members & 255) != 0) flush_round(members & 255);  // the last, partial round
    // out_color = C + T * bg, depth, inverse depth for the pixels that are inside the image and not masked (:485-496)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (valid[i]) {
            const int64_t pix = (int64_t)pix_base + i;
            const int64_t hw = (int64_t)p.W * p.H;
            p.out_color[pix] = fmaf(T[i], p.bg[0], Cr[i]);
            p.out_color[hw + pix] = fmaf(T[i], p.bg[1], Cg[i]);
            p.out_color[2 * hw + pix] = fmaf(T[i], p.bg[2], Cb[i]);
            p.out_depth[pix] = D[i];
            p.out_invdepth[pix] = ID[i];
        }
    }
  }
    if (p.stats && lane == 0 && iters) atomicAdd(p.stats + G2PC_STAT_WARP_GAUSSIANS, iters);
}

// fold one camera into the accumulators (__init__.py:128-158): colour of the arg-max pixel from the FINAL image, strict >
// for the maximum, sum of the per-camera maxima, minimum surface distance; clears the per-camera arrays
__global__ void __launch_bounds__(256) accumulate_tiles_kernel(unsigned long long* __restrict__ cam_best,
                                                               uint32_t* __restrict__ cam_dist,
                                                               const float* __restrict__ out_color, int64_t hw, int64_t n,
                                                               float* __restrict__ max_contrib, float* __restrict__ total,
                                                               float* __restrict__ colours, float* __restrict__ min_dist,
                                                               int32_t* __restrict__ first_frame, int32_t frame,
                                                               float* __restrict__ cam_contrib, int32_t* __restrict__ cam_pixel,
                                                               float* __restrict__ cam_surface) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    const unsigned long long b = cam_best[g];
    float v = 0.0f;
    int32_t pix = 0;
    if (b != 0ull) {
        cam_best[g] = 0ull;
        v = __uint_as_float((uint32_t)(b >> 32));
        pix = (int32_t)(0xFFFFFFFFu - (uint32_t)b);
        if (v > max_contrib[g]) {
            max_contrib[g] = v;
            if (first_frame) first_frame[g] = frame;
            colours[3 * g] = out_color[pix];
            colours[3 * g + 1] = out_color[hw + pix];
            colours[3 * g + 2] = out_color[2 * hw + pix];
        }
        total[g] += v;
    }
    if (cam_contrib) { cam_contrib[g] = v; cam_pixel[g] = pix; }
    if (cam_dist) {
        const uint32_t d = cam_dist[g];
        const float df = __uint_as_float(d);
        if (d != 0x7F7FFFFFu) {
            cam_dist[g] = 0x7F7FFFFFu;
            if (df < min_dist[g]) min_dist[g] = df;
        }
        if (cam_surface) cam_surface[g] = df;
    }
}

__global__ void __launch_bounds__(256) fill_u32_kernel(uint32_t* v, uint32_t x, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = x;
}

}  // namespace

extern "C" int g2pc_tiles_preprocess(const void* geom, const float* colours, const float* shs, int32_t sh_stride,
                                     int32_t sh_degree, int32_t sh_layout, int64_t n, const g2pc_raster_t* rs_host,
                                     void* proj, uint32_t* node_cnt, uint32_t* depth_key, uint64_t* val, int32_t* radii,
                                     void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(geom && rs_host && proj && node_cnt && depth_key && val, "null pointer");
    G2PC_CHECK_ARG(n <= 0xFFFFFFFFll, "more than 2^32 Gaussians");
    G2PC_CHECK_ARG((colours != nullptr) != (shs != nullptr), "provide exactly one of colours / shs");
    G2PC_CHECK_ARG(!shs || (sh_degree >= 0 && sh_degree <= 3 && sh_stride >= (sh_degree + 1) * (sh_degree + 1) &&
                            (sh_layout == 0 || sh_layout == 1)), "bad SH arguments");
    G2PC_CHECK_ARG(rs_host->width > 0 && rs_host->height > 0, "bad image size");
    TilePreParams p;
    p.geom = (const float4*)geom; p.colours = colours; p.shs = shs;
    p.sh_stride = sh_stride; p.sh_degree = sh_degree; p.sh_layout = sh_layout; p.n = n;
    for (int i = 0; i < 16; ++i) { p.view[i] = rs_host->viewmatrix[i]; p.projm[i] = rs_host->projmatrix[i]; }
    for (int i = 0; i < 3; ++i) p.campos[i] = rs_host->campos[i];
    p.tan_fovx = rs_host->tan_fovx; p.tan_fovy = rs_host->tan_fovy;
    p.W = rs_host->width; p.H = rs_host->height;
    p.focal_y = (float)p.H / (2.0f * p.tan_fovy);  // rasterizer_impl.cu:229-230
    p.focal_x = (float)p.W / (2.0f * p.tan_fovx);
    p.gx = (p.W + TILE - 1) / TILE; p.gy = (p.H + TILE - 1) / TILE;
    p.sgx = (p.gx + 1) / 2; p.sgy = (p.gy + 1) / 2;
    G2PC_CHECK_ARG(p.gx <= 256 && p.gy <= 256, "image larger than 4096 pixels per side (packed tile rect)");
    p.proj = (float4*)proj; p.node_cnt = node_cnt; p.depth_key = depth_key; p.val = (unsigned long long*)val;
    p.radii = radii;
    const int ntiles = p.sgx * p.sgy;
    p.use_hist = ntiles <= 24 * 1024 ? 1 : 0;
    const size_t smem = p.use_hist ? (size_t)ntiles * sizeof(uint32_t) : 0;
    if (smem > 48 * 1024)
        G2PC_CUDA(cudaFuncSetAttribute(preprocess_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    preprocess_tiles_kernel<<<(unsigned)((n + 1023) / 1024), 256, smem, (cudaStream_t)stream>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_tiles_build(uint32_t* node_cnt, int32_t width, int32_t height, g2pc_leaf_t* leaves,
                                int32_t* leaf_order, int32_t max_leaves, int64_t inst_capacity, int64_t matrix_capacity,
                                int32_t ms_rows, int32_t frame, int32_t* header, uint32_t* fail, int32_t* work_counters,
                                void* stream) {
    G2PC_CHECK_ARG(node_cnt && leaves && leaf_order && header && fail && work_counters, "null pointer");
    G2PC_CHECK_ARG(width > 0 && height > 0 && max_leaves >= 1 && frame >= 0, "bad sizes");
    TileTreeParams p;
    p.node_cnt = node_cnt; p.leaves = leaves; p.leaf_order = leaf_order;
    p.W = width; p.H = height;
    p.gx = ((width + TILE - 1) / TILE + 1) / 2; p.gy = ((height + TILE - 1) / TILE + 1) / 2;  // super-tile grid
    p.max_leaves = max_leaves; p.inst_capacity = inst_capacity; p.matrix_capacity = matrix_capacity;
    p.ms_rows = ms_rows; p.frame = frame; p.header = header; p.fail = fail; p.work_counters = work_counters;
    tile_tree_kernel<<<1, TB, 0, (cudaStream_t)stream>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_tiles_blend(const g2pc_leaf_t* leaves, const int32_t* leaf_order, const int32_t* header,
                                const uint32_t* fail, int32_t frame, const uint32_t* inst_gid, const void* proj, uint64_t* cam_best, uint32_t* cam_dist,
                                const int32_t* mask, float* out_color, float* out_depth, float* out_invdepth,
                                int32_t width, int32_t height, const float* background3_host, int32_t* work_counters,
                                uint64_t* stats, void* stream) {
    G2PC_CHECK_ARG(leaves && leaf_order && header && fail && inst_gid && proj && cam_best && out_color && out_depth &&
                       out_invdepth && background3_host && work_counters, "null pointer");
    G2PC_CHECK_ARG(((uintptr_t)inst_gid & 15) == 0, "inst_gid must be 16-byte aligned (TMA bulk copies)");
    TileBlendParams p;
    p.leaves = leaves; p.leaf_order = leaf_order; p.header = header; p.fail = fail; p.frame = frame;
    p.inst_gid = inst_gid;
    p.proj = (const float4*)proj; p.cam_best = (unsigned long long*)cam_best; p.cam_dist = cam_dist; p.mask = mask;
    p.out_color = out_color; p.out_depth = out_depth; p.out_invdepth = out_invdepth;
    p.W = width; p.H = height;
    for (int i = 0; i < 3; ++i) p.bg[i] = background3_host[i];
    p.work_counter = work_counters; p.stats = (unsigned long long*)stats;
    cudaStream_t st = (cudaStream_t)stream;
    if (cam_dist)
        blend_tiles_kernel<true><<<(unsigned)resident_ctas(blend_tiles_kernel<true>, TBT, 0, 3), TBT, 0, st>>>(p);
    else
        blend_tiles_kernel<false><<<(unsigned)resident_ctas(blend_tiles_kernel<false>, TBT, 0, 4), TBT, 0, st>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_tiles_accumulate(uint64_t* cam_best, uint32_t* cam_dist, const float* out_color, int32_t width,
                                     int32_t height, int64_t n, float* max_contrib, float* total_contrib, float* colours,
                                     float* min_dist, int32_t* first_frame, int32_t frame, float* cam_contrib,
                                     int32_t* cam_pixel, float* cam_surface, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(cam_best && out_color && max_contrib && total_contrib && colours, "null pointer");
    G2PC_CHECK_ARG(!cam_dist || min_dist, "min_dist required with cam_dist");
    G2PC_CHECK_ARG((cam_contrib == nullptr) == (cam_pixel == nullptr), "cam_contrib and cam_pixel go together");
    accumulate_tiles_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (unsigned long long*)cam_best, cam_dist, out_color, (int64_t)width * height, n, max_contrib, total_contrib, colours,
        min_dist, first_frame, frame, cam_contrib, cam_pixel, cam_surface);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_fill_u32(uint32_t* v, uint32_t value, int64_t n, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(v, "null pointer");
    fill_u32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(v, value, n);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}
