// colour_common.cuh — shared pieces of both colour back-ends (S3-S7): quadtree tables in shared memory, range queries, SH
// colours, list-table building blocks (block scan, launch-order sort, frame header), async-copy / TMA helpers.
#pragma once
#include "common.cuh"

constexpr unsigned FULLM = 0xffffffffu;

#define QT_FLAG_DROPPED 1
#define QT_FLAG_BIG 2

// node states written by the tree kernel
#define NODE_NONE 0   // does not exist / dropped
#define NODE_EMPTY 1  // exists, no Gaussian overlaps it (background fill, gauss_render.py:313-315)
#define NODE_SPLIT 2  // exists and was split into 4 children (gauss_render.py:319-335)
#define NODE_LEAF 3   // exists and is rendered

// node range of a Gaussian at the first leaf-candidate level, packed 8 bits per bound
#define G2PC_RANGE_MAX_LEVEL 8
#define G2PC_RANGE_EMPTY 0x00000001u  // xlo = 1 > xhi = 0
__host__ __device__ __forceinline__ uint32_t g2pc_pack_range(int xlo, int xhi, int ylo, int yhi) {
    return (uint32_t)xlo | ((uint32_t)xhi << 8) | ((uint32_t)ylo << 16) | ((uint32_t)yhi << 24);
}
__host__ __device__ __forceinline__ void g2pc_unpack_range(uint32_t r, int& xlo, int& xhi, int& ylo, int& yhi) {
    xlo = (int)(r & 255u); xhi = (int)((r >> 8) & 255u); ylo = (int)((r >> 16) & 255u); yhi = (int)(r >> 24);
}

// Frame failure word shared by the frames in flight (uint32, 0xFFFFFFFF = none, else 1 + the LOWEST frame that did not fit):
// every kernel of frame f does nothing iff f + 1 >= *fail.  Frames of two CUDA streams may be in flight at once, so a
// later frame can fail before an earlier one has finished: the earlier one must still complete.
__device__ __forceinline__ bool g2pc_frame_skipped(const uint32_t* fail, int frame) {
    return (uint32_t)(frame + 1) >= *fail;
}

// Frame header of the list-table kernels (one CTA).  Prologue of a frame that g2pc_frame_skipped: report the poison
// (the kernel then does nothing).
__device__ __forceinline__ void report_skipped_frame(const uint32_t* fail, int frame, int32_t* header) {
    if (threadIdx.x == 0) { header[G2PC_HDR_POISON] = (int32_t)*fail; header[G2PC_HDR_FRAME] = frame; }
}
// Epilogue (one thread): the sizes of the frame, the overflow flags, then the failure word — lowered first if the frame
// did not fit, so the header of a failed frame always names the earliest failure.
__device__ __forceinline__ void write_frame_header(int32_t* header, uint32_t* fail, int frame, int num_leaves,
                                                   long long inst_total, int total_pix, int need_deeper, int leaf_over,
                                                   int cap_over) {
    header[G2PC_HDR_NUM_LEAVES] = num_leaves;
    header[G2PC_HDR_TOTAL_INST] = (int32_t)(inst_total & 0xFFFFFFFFll);
    header[G2PC_HDR_TOTAL_INST_HI] = (int32_t)(inst_total >> 32);
    header[G2PC_HDR_TOTAL_PIX] = total_pix;
    header[G2PC_HDR_NEED_DEEPER] = need_deeper;
    header[G2PC_HDR_LEAF_OVERFLOW] = leaf_over;
    header[G2PC_HDR_CAP_OVERFLOW] = cap_over;
    header[G2PC_HDR_FRAME] = frame;
    if (need_deeper | leaf_over | cap_over) atomicMin(fail, (uint32_t)(frame + 1));
    const uint32_t f = *(volatile uint32_t*)fail;
    header[G2PC_HDR_POISON] = f == 0xFFFFFFFFu ? 0 : (int32_t)f;
}

// block-wide exclusive scan for a CTA of (a multiple of 32, at most 1024) threads; returns the prefix, sets total
__device__ __forceinline__ int block_scan(int v, int* s_warp, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULLM, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULLM, winc, o);
            if (lane >= o) winc += t;
        }
        s_warp[lane] = winc - w;            // exclusive prefix of warp totals
        if (lane == 31) s_warp[32] = winc;  // grand total
    }
    __syncthreads();
    const int res = s_warp[warp] + inc - v;
    total = s_warp[32];
    __syncthreads();
    return res;
}

// Ascending bitonic sort of m keys (a power of two) in shared memory: the heaviest-first launch order of the leaves in
// both list-table kernels.  NT = threads of the CTA, a compile-time constant (the loop stride unrolls against it).
template <int NT, typename K>
__device__ __forceinline__ void bitonic_sort(K* s_sort, int m) {
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < m; i += NT) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const K a = s_sort[i], b = s_sort[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { s_sort[i] = b; s_sort[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
}

// ---- async copies (sm_90+) --------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2f(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  // results below FLT_MIN flush to 0
    return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one elected thread: arm the barrier with the byte count, then start the 1-D bulk copy global -> shared (TMA engine)
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // earlier generic-proxy reads of dst are ordered before
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// CTAs of a persistent grid: every SM filled to the kernel's occupancy (per_sm_fallback if the query fails)
template <typename Kernel>
inline int resident_ctas(Kernel kernel, int threads, size_t smem, int per_sm_fallback) {
    int dev = 0, sms = 148, per_sm = per_sm_fallback;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1)
        per_sm = per_sm_fallback;
    return sms * per_sm;
}

// SH colour of one channel (gauss_render.py:43-99; + 0.5, clamped at 0 as forward.cu:65-72), d = unit view direction.
// coef(k) returns coefficient k of the channel; the caller chooses the loads.
template <typename Coef>
__device__ __forceinline__ float sh_channel(int deg, float3 d, Coef coef) {
    const float C0 = 0.28209479177387814f, C1 = 0.4886025119029199f;
    const float C2[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f, -1.0925484305920792f,
                         0.5462742152960396f};
    const float C3[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f, 0.3731763325901154f,
                         -0.4570457994644658f, 1.445305721320277f, -0.5900435899266435f};
    const float x = d.x, y = d.y, z = d.z;
    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
    float r = C0 * coef(0);
    if (deg > 0) {
        r = r - C1 * y * coef(1) + C1 * z * coef(2) - C1 * x * coef(3);
        if (deg > 1) {
            r = r + C2[0] * xy * coef(4) + C2[1] * yz * coef(5) + C2[2] * (2.0f * zz - xx - yy) * coef(6) +
                C2[3] * xz * coef(7) + C2[4] * (xx - yy) * coef(8);
            if (deg > 2) {
                r = r + C3[0] * y * (3.0f * xx - yy) * coef(9) + C3[1] * xy * z * coef(10) +
                    C3[2] * y * (4.0f * zz - xx - yy) * coef(11) +
                    C3[3] * z * (2.0f * zz - 3.0f * xx - 3.0f * yy) * coef(12) +
                    C3[4] * x * (4.0f * zz - xx - yy) * coef(13) + C3[5] * z * (xx - yy) * coef(14) +
                    C3[6] * x * (xx - 3.0f * yy) * coef(15);
            }
        }
    }
    return fmaxf(r + 0.5f, 0.0f);
}

struct QtMeta {
    int32_t num_levels;  // tabulated levels 0..num_levels-1
    int32_t max_gaussians_per_tile;
};

// per-Gaussian projection record: 3 x float4
//   q0 = (mx, my, c00', c01')     c' = conic * (-0.5 * log2(e));  c01' = (conic01 + conic10)'
//   q1 = (c11', opacity, r, g)
//   q2 = (b, depth, radius, valid)   valid: 1.0f if in front of the camera (gauss_render.py:167), else 0
struct QtTables {
    const int32_t* xs; const int32_t* xe; const int32_t* xf;
    const int32_t* ys; const int32_t* ye; const int32_t* yf;
};

// the 6 arrays of n1 ints of the flat table array (g2pc/quadtree.py QuadtreeTables.flat)
inline QtTables make_tables(const int32_t* tables, int n1) {
    QtTables t;
    t.xs = tables; t.xe = tables + n1; t.xf = tables + 2 * n1;
    t.ys = tables + 3 * n1; t.ye = tables + 4 * n1; t.yf = tables + 5 * n1;
    return t;
}

// first 2-D node of level l (levels 0..l-1 hold (4^l - 1) / 3 nodes)
__device__ __forceinline__ int off2(int l) { return ((1 << (2 * l)) - 1) / 3; }

// copy the 1-D tables (6 arrays of n1 ints) into shared memory; returns pointers into smem
__device__ __forceinline__ QtTables load_tables(const QtTables g, int n1, int32_t* smem) {
    for (int i = threadIdx.x; i < n1; i += blockDim.x) {
        smem[i] = g.xs[i];
        smem[n1 + i] = g.xe[i];
        smem[2 * n1 + i] = g.xf[i];
        smem[3 * n1 + i] = g.ys[i];
        smem[4 * n1 + i] = g.ye[i];
        smem[5 * n1 + i] = g.yf[i];
    }
    __syncthreads();
    QtTables s;
    s.xs = smem; s.xe = smem + n1; s.xf = smem + 2 * n1;
    s.ys = smem + 3 * n1; s.ye = smem + 4 * n1; s.yf = smem + 5 * n1;
    return s;
}

// Members of the interval (rmin, rmax) among the 2^level nodes of one axis at `level`:
//   min(rmax, e_i) > max(rmin, s_i)   (fp32 compares, strict — gauss_render.py:308-310)
//   <=>  rmax > rmin  &&  rmax > s_i  &&  e_i > rmin  &&  e_i > s_i
// starts / ends are non-decreasing within a level, so the candidates form the index range [lo, hi]; nodes inside the
// range that are dropped or degenerate (e_i <= s_i) are filtered by the caller through axis_member().
__device__ __forceinline__ void axis_range(const int32_t* __restrict__ s, const int32_t* __restrict__ e, int level,
                                           float rmin, float rmax, float inv_step, int& lo, int& hi) {
    const int n = 1 << level;
    if (!(rmax > rmin)) { lo = 1; hi = 0; return; }
    // the nodes of a level are (nearly) uniformly spaced: start from the arithmetic guess and walk to the exact answer
    // (0-2 steps in practice) instead of a binary search.  inv_step = 2^level / extent.
    // lo = first i with e_i > rmin
    int a = min(n - 1, max(0, (int)(rmin * inv_step)));
    while (a < n && !((float)e[a] > rmin)) ++a;
    while (a > 0 && (float)e[a - 1] > rmin) --a;
    lo = a;
    // hi = last i with s_i < rmax
    a = min(n - 1, max(0, (int)(rmax * inv_step)));
    while (a >= 0 && !((float)s[a] < rmax)) --a;
    while (a + 1 < n && (float)s[a + 1] < rmax) ++a;
    hi = a;
}

__device__ __forceinline__ bool axis_member(const int32_t* __restrict__ s, const int32_t* __restrict__ e,
                                            const int32_t* __restrict__ f, int i) {
    return !(f[i] & QT_FLAG_DROPPED) && e[i] > s[i];
}

// Warp-cooperative walk over per-lane node rectangles.  Every lane brings a packed rectangle (g2pc_pack_range; empty if
// xlo > xhi) and a 32-bit payload; f(ix, iy, owner_lane, owner_payload) is called once per (lane, node).  Rectangles of up
// to WARP_SMALL_AREA nodes are walked by their own lane; larger ones (a few huge splats cover hundreds of tiles) are
// walked by the whole warp — the lanes tile the rectangle with a power-of-two number of columns, so no division is
// needed — otherwise the warp runs at the speed of its largest rectangle (ncu r02a: 6.9 of 32 threads active in the
// multisplit).  Must be called by all 32 lanes.
// (a cooperative iteration costs ~45 instructions of shuffles / loop control, a private node ~12: the break-even rectangle
// is ~10 nodes; with a threshold of 4 the typical 2x3 / 3x3 rectangles all went the slow cooperative way)
constexpr int WARP_SMALL_AREA = 12;
template <typename F>
__device__ __forceinline__ void warp_for_each_node(uint32_t range, uint32_t payload, F f) {
    const int lane = threadIdx.x & 31;
    int xlo, xhi, ylo, yhi;
    g2pc_unpack_range(range, xlo, xhi, ylo, yhi);
    const int area = (xlo > xhi || ylo > yhi) ? 0 : (xhi - xlo + 1) * (yhi - ylo + 1);
    if (area > 0 && area <= WARP_SMALL_AREA)
        for (int iy = ylo; iy <= yhi; ++iy)
            for (int ix = xlo; ix <= xhi; ++ix) f(ix, iy, lane, payload);
    unsigned big = __ballot_sync(0xffffffffu, area > WARP_SMALL_AREA);
    while (big) {
        const int b = __ffs(big) - 1;
        big &= big - 1u;
        const uint32_t br = __shfl_sync(0xffffffffu, range, b);
        const uint32_t bp = __shfl_sync(0xffffffffu, payload, b);
        int bx, bxh, by, byh;
        g2pc_unpack_range(br, bx, bxh, by, byh);
        const int bw = bxh - bx + 1, bh = byh - by + 1;
        const int sh = bw <= 1 ? 0 : 32 - __clz(bw - 1);  // ceil(log2(width))
        if (sh >= 5) {
            for (int ry = 0; ry < bh; ++ry)
                for (int rx = lane; rx < bw; rx += 32) f(bx + rx, by + ry, b, bp);
        } else {
            const int rx = lane & ((1 << sh) - 1);
            if (rx < bw)
                for (int ry = lane >> sh; ry < bh; ry += 32 >> sh) f(bx + rx, by + ry, b, bp);
        }
    }
}

// rect of a Gaussian (gauss_render.py:182-193): [mean -+ radius] clipped to [0, W-1] x [0, H-1]
__device__ __forceinline__ void gaussian_rect(float mx, float my, float radius, int W, int H, float& x0, float& x1,
                                              float& y0, float& y1) {
    const float wm = (float)W - 1.0f, hm = (float)H - 1.0f;
    x0 = fminf(fmaxf(mx - radius, 0.0f), wm);
    x1 = fminf(fmaxf(mx + radius, 0.0f), wm);
    y0 = fminf(fmaxf(my - radius, 0.0f), hm);
    y1 = fminf(fmaxf(my + radius, 0.0f), hm);
}
