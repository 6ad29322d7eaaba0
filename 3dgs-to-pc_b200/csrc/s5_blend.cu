// s5_blend.cu — S5: per-leaf front-to-back blend with per-Gaussian max-contribution tracking; S6: accumulate; image.
//
// Reference semantics restated (not copied), renderer_type=python, gauss_render.py:337-402:
//   every Gaussian of a leaf's depth-ordered list contributes to EVERY pixel of the leaf (no 1/255 cut, no early
//   termination, no per-pixel radius test):
//     weight = exp(-0.5 (dx^2 c00 + dy^2 c11 + dx dy c01 + dx dy c10)),  alpha = min(0.99, weight * opacity),
//     contribution = T * alpha,  T <- T (1 - alpha),  pixel = sum contribution * colour + (1 - sum contribution) * bg
//   per Gaussian: the largest contribution over the leaf's pixels and the pixel where it occurs; where that beats the
//   Gaussian's running maximum (strict >, over leaves in BFS order and cameras in call order) the maximum and the
//   blended colour of that pixel are stored (:371-395).
// Role of renderCUDA (forward.cu:303-497) in the reference's CUDA back-end; none of its structure is kept.
//
// Kernel shape: persistent CTAs of 128 threads pull (leaf, slab) items, heaviest leaf first; a CTA owns up to 128 quads
// (4 consecutive pixels of one row) of a leaf and walks the leaf's depth-ordered id list in chunks of 128 Gaussians
// through a 3-deep software pipeline:
//   stage A  the id chunk c+2 is brought into shared memory by ONE TMA bulk copy (cp.async.bulk + mbarrier
//            complete_tx; the lists are 16-byte aligned by the tree kernel)                  — "TMA staging of tile lists"
//   stage B  the 48-byte projection records of chunk c+1 are gathered by cp.async (LDGSTS, 16-byte copies addressed by
//            the staged ids) straight into shared memory, no register round trip
//   stage C  chunk c is blended
// so the dependent id -> record latency of the next chunks hides under the arithmetic of the current one.  Per thread
// and Gaussian the row-dependent terms are formed once; the per-pixel arithmetic runs on the packed FP32x2 pipe (FADD2 /
// FFMA2 / FMUL2, two pixels per instruction, scalar broadcast operands): 8 packed ops + 2 EX2 + 2 FMNMX per pixel pair.
// The per-Gaussian maximum is a redux.sync (u32 max of the non-negative float bits) per warp, merged across warps in
// shared memory and published with ONE 64-bit atomicMax per (CTA, Gaussian): key = (contribution bits << 32) |
// ~(leaf-pixel index), so ties go to the earliest leaf / lowest pixel, deterministically.
// Short-cuts: (i) a warp stops once ALL its pixels have T below t_stop (checked every 32 Gaussians): every contribution
// it skips is < t_stop and so is their sum per pixel; t_stop = FLT_MIN in strict-parity runs; (ii) the arg-max
// bookkeeping of a Gaussian is skipped by a warp when none of its contributions exceeds the maximum the Gaussian already
// holds from earlier cameras (the update rule is a strict >, so such contributions can never be recorded).
#include "colour_common.cuh"

namespace {

constexpr int BT = 128;
constexpr int CH = 128;
constexpr int SUB = 32;   // Gaussians between two transmittance checks

struct BlendParams {
    const g2pc_leaf_t* leaves;
    const int32_t* leaf_order;
    const int32_t* header;
    const uint32_t* fail;
    int32_t frame;
    const uint32_t* inst_gid;
    const float4* proj;
    unsigned long long* cam_best;
    const float* max_contrib;  // running per-Gaussian maxima of the earlier cameras (threshold for the bookkeeping)
    float* leaf_colour;
    uint32_t* owner;
    int32_t W, H;
    float bg;
    float t_stop;
    int32_t* work_counter;  // cleared by the tree kernel: dynamic (leaf, slab) work distribution
    int32_t slabs;
    int32_t compact;        // 1: compact warp footprints (blocks), 0: row strips
    unsigned long long* stats;
};

__global__ void __launch_bounds__(BT, 8) blend_kernel(const BlendParams p) {
    __shared__ __align__(16) float4 s_q0[2][CH];
    __shared__ __align__(16) float4 s_q1[2][CH];
    __shared__ __align__(8) float2 s_b[2][CH];           // (blue, threshold)
    __shared__ __align__(16) uint32_t s_gid[3][CH];      // id chunks, filled by the TMA engine
    __shared__ unsigned long long s_best[BT / 32][CH];
    __shared__ __align__(8) unsigned long long s_bar[3];
    __shared__ int s_item;

    if (g2pc_frame_skipped(p.fail, p.frame)) return;
    const int num_items = p.header[G2PC_HDR_NUM_LEAVES] * p.slabs;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_init(&s_bar[2], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int w = 0; w < BT / 32; ++w) s_best[w][tid] = 0ull;
    uint32_t phase_bits = 0;  // parity of the next completion of each id barrier (bit s)
    const float t_stop = p.t_stop;
    unsigned long long iters = 0;
    __syncthreads();

    // persistent CTAs: work items (leaf, slab) are handed out heaviest-leaf-first from a global counter, so the tail of
    // the launch is at most one item long
  for (;;) {
    if (tid == 0) s_item = atomicAdd(p.work_counter, 1);
    __syncthreads();
    const int item = s_item;
    __syncthreads();
    if (item >= num_items) break;
    const g2pc_leaf_t lf = p.leaves[p.leaf_order[item / p.slabs]];
    const int qpr = (lf.w + 3) >> 2;
    bool active;
    int row, x0;
    if (p.compact) {
        // compact warp footprints: a warp owns a block of tw quad columns x th rows (<= 32 quads, e.g. 20 x 6 pixels of a
        // 40 x 23 leaf) instead of a strip of full rows — the pixels of a block reach the transmittance stop together
        const int ncb = (qpr + 4) / 5;                 // blocks across
        const int tw = (qpr + ncb - 1) / ncb;          // <= 5 quad columns per block
        const int th = 32 / tw;                        // rows per block
        const int nrb = (lf.h + th - 1) / th;
        const int wblock = (item % p.slabs) * (BT / 32) + warp;   // block of this warp
        if ((item % p.slabs) * (BT / 32) >= ncb * nrb) continue;  // uniform: no block left for this slab
        const int bx = wblock % ncb, by = wblock / ncb;
        const int lr = lane / tw, lc = lane - lr * tw;
        row = by * th + lr;
        const int qc = bx * tw + lc;
        active = wblock < ncb * nrb && lr < th && row < lf.h && qc < qpr;
        x0 = qc * 4;
        if (!active) { row = 0; x0 = 0; }
    } else {
        const int nquads = qpr * lf.h;
        const int quad0 = (item % p.slabs) * BT;
        if (quad0 >= nquads) continue;
        const int quad = quad0 + tid;
        active = quad < nquads;
        row = active ? quad / qpr : 0;
        x0 = active ? (quad - row * qpr) * 4 : 0;
    }

    // two pixel pairs per thread: Blackwell's packed FP32x2 pipe (FADD2 / FMUL2 / FFMA2) takes a scalar broadcast operand,
    // so the per-Gaussian scalars feed both pixels of a pair without extra moves
    float2 T01, T23, px01, px23;
    float2 Cr01 = make_float2(0.f, 0.f), Cr23 = Cr01, Cg01 = Cr01, Cg23 = Cr01, Cb01 = Cr01, Cb23 = Cr01;
    {
        float Tv[4], pxv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const bool valid = active && (x0 + i < lf.w);
            Tv[i] = valid ? 1.0f : 0.0f;  // T = 0 makes every contribution of a padding pixel exactly 0
            pxv[i] = (float)(lf.c0 + x0 + i);
        }
        T01 = make_float2(Tv[0], Tv[1]); T23 = make_float2(Tv[2], Tv[3]);
        px01 = make_float2(pxv[0], pxv[1]); px23 = make_float2(pxv[2], pxv[3]);
    }
    const float py = (float)(lf.r0 + row);
    const int pix_row = row * lf.w + x0;

    const int cnt = lf.inst_count;
    const int nchunks = (cnt + CH - 1) / CH;
    const uint32_t* list = p.inst_gid + (int64_t)lf.inst_begin;  // 16-byte aligned (tree kernel)

    // ---- pipeline helpers ------------------------------------------------------------------------------------------
    auto issue_ids = [&](int c) {  // thread 0 only
        const int nl = min(CH, cnt - c * CH);
        const uint32_t bytes = (uint32_t)(((nl + 3) & ~3) * 4);  // whole 16-byte units (the lists are padded)
        tma_load_1d(&s_gid[c % 3][0], list + (int64_t)c * CH, bytes, &s_bar[c % 3]);
    };
    auto wait_ids = [&](int c) {
        const int s = c % 3;
        mbar_wait(&s_bar[s], (phase_bits >> s) & 1u);
        phase_bits ^= 1u << s;
    };
    auto issue_records = [&](int c) {
        const int nl = min(CH, cnt - c * CH);
        if (tid < nl) {
            const uint32_t gid = s_gid[c % 3][tid];
            const float4* rec = p.proj + 3 * (int64_t)gid;
            cp_async16(&s_q0[c & 1][tid], rec);
            cp_async16(&s_q1[c & 1][tid], rec + 1);
            cp_async4(&s_b[c & 1][tid].x, rec + 2);
            cp_async4(&s_b[c & 1][tid].y, p.max_contrib + gid);
        }
        cp_async_commit();
    };

    bool warp_done = false;
    if (nchunks > 0) {
        if (tid == 0) { issue_ids(0); if (nchunks > 1) issue_ids(1); }
        wait_ids(0);
        issue_records(0);
    }
    for (int c = 0; c < nchunks; ++c) {
        const int nload = min(CH, cnt - c * CH);
        const bool more = (c + 1 < nchunks);
        if (more) { wait_ids(c + 1); issue_records(c + 1); }
        if (more) cp_async_wait<1>(); else cp_async_wait<0>();
        // records of chunk c visible to the CTA; every thread is past the merge of chunk c - 1 (its id buffer is free)
        const bool all_done = __syncthreads_and(warp_done ? 1 : 0);
        if (all_done) {
            if (more) cp_async_wait<0>();  // drain the gather in flight before the buffers are reused by the next item
            break;
        }
        if (tid == 0 && c + 2 < nchunks) issue_ids(c + 2);
        const float4* q0s = s_q0[c & 1];
        const float4* q1s = s_q1[c & 1];
        const float2* bs = s_b[c & 1];
        if (!warp_done) {
            for (int j0 = 0; j0 < nload; j0 += SUB) {
                const int j1 = min(nload, j0 + SUB);
                for (int j = j0; j < j1; ++j) {
                    const float4 q0 = q0s[j];
                    const float4 q1 = q1s[j];
                    const float2 bt = bs[j];
                    const float bl = bt.x;
                    const float dy = py - q0.y;
                    const float Bq = dy * q0.w;
                    const float Cq = fmaf(dy * dy, q1.x, q1.y);  // + log2(opacity): alpha = min(0.99, exp2(e))
                    const float nmx = -q0.x;
                    const float2 dx01 = __fadd2_rn(px01, make_float2(nmx, nmx));
                    const float2 dx23 = __fadd2_rn(px23, make_float2(nmx, nmx));
                    const float2 e01 = __ffma2_rn(dx01, __ffma2_rn(dx01, make_float2(q0.z, q0.z), make_float2(Bq, Bq)),
                                                  make_float2(Cq, Cq));
                    const float2 e23 = __ffma2_rn(dx23, __ffma2_rn(dx23, make_float2(q0.z, q0.z), make_float2(Bq, Bq)),
                                                  make_float2(Cq, Cq));
                    const float2 a01 = make_float2(fminf(0.99f, ex2f(e01.x)), fminf(0.99f, ex2f(e01.y)));
                    const float2 a23 = make_float2(fminf(0.99f, ex2f(e23.x)), fminf(0.99f, ex2f(e23.y)));
                    const float2 c01 = __fmul2_rn(T01, a01);
                    const float2 c23 = __fmul2_rn(T23, a23);
                    Cr01 = __ffma2_rn(c01, make_float2(q1.z, q1.z), Cr01);
                    Cr23 = __ffma2_rn(c23, make_float2(q1.z, q1.z), Cr23);
                    Cg01 = __ffma2_rn(c01, make_float2(q1.w, q1.w), Cg01);
                    Cg23 = __ffma2_rn(c23, make_float2(q1.w, q1.w), Cg23);
                    Cb01 = __ffma2_rn(c01, make_float2(bl, bl), Cb01);
                    Cb23 = __ffma2_rn(c23, make_float2(bl, bl), Cb23);
                    T01 = __ffma2_rn(c01, make_float2(-1.0f, -1.0f), T01);  // T - T*alpha (one rounding)
                    T23 = __ffma2_rn(c23, make_float2(-1.0f, -1.0f), T23);
                    // arg-max bookkeeping only if some contribution can beat what the Gaussian already holds
                    const float v = fmaxf(fmaxf(c01.x, c01.y), fmaxf(c23.x, c23.y));
                    if (__any_sync(FULLM, v > bt.y)) {
                        // warp max of the (non-negative) contributions, then the lowest pixel index among the lanes holding it
                        const uint32_t vb = __float_as_uint(v);
                        const uint32_t wm = __reduce_max_sync(FULLM, vb);
                        const int i = (c01.x == v) ? 0 : (c01.y == v) ? 1 : (c23.x == v) ? 2 : 3;
                        const uint32_t pk = (vb == wm) ? (0xFFFFFFFFu - (uint32_t)(pix_row + i)) : 0u;
                        const uint32_t wp = __reduce_max_sync(FULLM, pk);
                        if (lane == 0) s_best[warp][j] = ((unsigned long long)wm << 32) | (unsigned long long)wp;
                    }
                }
                iters += (unsigned long long)(j1 - j0);
                const float tmax = fmaxf(fmaxf(T01.x, T01.y), fmaxf(T23.x, T23.y));
                warp_done = __all_sync(FULLM, tmax < t_stop);
                if (warp_done) break;
            }
        }
        __syncthreads();  // s_best complete; every warp is past its reads of the record buffers of chunk c
        if (tid < nload) {
            unsigned long long best = s_best[0][tid];
            s_best[0][tid] = 0ull;
#pragma unroll
            for (int w = 1; w < BT / 32; ++w) {
                const unsigned long long o = s_best[w][tid];
                s_best[w][tid] = 0ull;
                best = o > best ? o : best;
            }
            if ((best >> 32) != 0ull) {
                // leaf-local pixel -> index into the concatenated leaf-colour buffer (earlier leaf => smaller index)
                const uint32_t pix = 0xFFFFFFFFu - (uint32_t)best;
                const unsigned long long packed = (best & 0xFFFFFFFF00000000ull) |
                                                  (unsigned long long)(0xFFFFFFFFu - (uint32_t)(lf.pix_offset + pix));
                atomicMax(p.cam_best + s_gid[c % 3][tid], packed);
            }
        }
    }
    // final pixel colours: sum + (1 - sum of contributions) * bg; the second factor equals the final T
    if (active) {
        const float T[4] = {T01.x, T01.y, T23.x, T23.y};
        const float Cr[4] = {Cr01.x, Cr01.y, Cr23.x, Cr23.y};
        const float Cg[4] = {Cg01.x, Cg01.y, Cg23.x, Cg23.y};
        const float Cb[4] = {Cb01.x, Cb01.y, Cb23.x, Cb23.y};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (x0 + i < lf.w) {
                const int64_t lp = (int64_t)lf.pix_offset + pix_row + i;
                float* o = p.leaf_colour + 3 * lp;
                o[0] = fmaf(T[i], p.bg, Cr[i]);
                o[1] = fmaf(T[i], p.bg, Cg[i]);
                o[2] = fmaf(T[i], p.bg, Cb[i]);
                // overlapping leaves: the later BFS entry wins the image pixel (gauss_render.py:369)
                atomicMax(p.owner + (int64_t)(lf.r0 + row) * p.W + (lf.c0 + x0 + i), (uint32_t)lp + 1u);
            }
        }
    }
  }  // work-item loop
    if (p.stats && lane == 0 && iters) atomicAdd(p.stats + G2PC_STAT_WARP_GAUSSIANS, iters);
}

// S6: fold one camera's per-Gaussian winners into the running maxima (strict >, earlier camera wins ties) and fetch
// the blended colour of the winning pixel (gauss_render.py:387-395); clears cam_best for the next camera.
__global__ void __launch_bounds__(256) accumulate_kernel(unsigned long long* __restrict__ cam_best,
                                                         const float* __restrict__ leaf_colour, int64_t n,
                                                         float* __restrict__ max_contrib, float* __restrict__ colours,
                                                         int32_t* __restrict__ first_frame, int32_t frame) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    const unsigned long long b = cam_best[g];
    if (b == 0ull) return;
    cam_best[g] = 0ull;
    const float v = __uint_as_float((uint32_t)(b >> 32));
    if (v > max_contrib[g]) {
        max_contrib[g] = v;
        if (first_frame) first_frame[g] = frame;
        const int64_t idx = (int64_t)(0xFFFFFFFFu - (uint32_t)b);
        colours[3 * g] = leaf_colour[3 * idx];
        colours[3 * g + 1] = leaf_colour[3 * idx + 1];
        colours[3 * g + 2] = leaf_colour[3 * idx + 2];
    }
}

// image = leaf colours where a leaf covers the pixel, else background; flipped left-right (gauss_render.py:402)
__global__ void __launch_bounds__(256) compose_kernel(uint32_t* __restrict__ owner, const float* __restrict__ leaf_colour,
                                                      int W, int H, float bg, float* __restrict__ image) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)W * H) return;
    const int y = (int)(i / W), x = (int)(i - (int64_t)y * W);
    const uint32_t o = owner[i];
    owner[i] = 0u;
    float r = bg, g = bg, b = bg;
    if (o) { const float* c = leaf_colour + 3 * (int64_t)(o - 1u); r = c[0]; g = c[1]; b = c[2]; }
    float* out = image + 3 * ((int64_t)y * W + (W - 1 - x));
    out[0] = r; out[1] = g; out[2] = b;
}

}  // namespace

static int g_blend_compact = 1;
/* experiment switch (bench / tests): 1 = compact warp footprints (default), 0 = row strips */
extern "C" void g2pc_blend_set_compact(int on) { g_blend_compact = on ? 1 : 0; }

extern "C" int g2pc_blend(const g2pc_leaf_t* leaves, const int32_t* leaf_order, const int32_t* header,
                          const uint32_t* fail, int32_t frame, int32_t max_leaf_pixels_quads, const uint32_t* inst_gid,
                          const void* proj,
                          uint64_t* cam_best, const float* max_contrib, float* leaf_colour, uint32_t* owner,
                          int32_t width, int32_t height, float background, float t_stop, int32_t* work_counters,
                          uint64_t* stats, void* stream) {
    G2PC_CHECK_ARG(leaves && leaf_order && header && fail && inst_gid && proj && cam_best && max_contrib && leaf_colour &&
                       owner && work_counters, "null pointer");
    G2PC_CHECK_ARG(max_leaf_pixels_quads >= 1, "max_leaf_pixels_quads < 1");
    G2PC_CHECK_ARG(t_stop >= 0.0f && t_stop < 1.0f, "t_stop must be in [0, 1)");
    G2PC_CHECK_ARG(((uintptr_t)inst_gid & 15) == 0, "inst_gid must be 16-byte aligned (TMA bulk copies)");
    BlendParams p;
    p.leaves = leaves; p.leaf_order = leaf_order; p.header = header; p.fail = fail; p.frame = frame;
    p.inst_gid = inst_gid;
    p.proj = (const float4*)proj;
    p.cam_best = (unsigned long long*)cam_best; p.max_contrib = max_contrib; p.leaf_colour = leaf_colour;
    p.owner = owner;
    p.W = width; p.H = height; p.bg = background;
    p.t_stop = t_stop > 1.17549435e-38f ? t_stop : 1.17549435e-38f;
    p.compact = g_blend_compact;
    // slabs: CTAs per leaf.  Row strips: ceil(quads / 128).  Blocks: a leaf of max_tile_size has at most
    // ceil(qpr / 5) x ceil(h / 6) blocks of <= 32 quads; the caller's bound is quads = ceil(w / 4) * h <= 15 * h.
    p.slabs = p.compact ? (max_leaf_pixels_quads + 4 * 25 - 1) / (4 * 25) + 1 : (max_leaf_pixels_quads + BT - 1) / BT;
    p.work_counter = work_counters;
    p.stats = (unsigned long long*)stats;
    static int resident = 0;  // persistent grid: every SM filled to the kernel's occupancy (device constant)
    if (resident == 0) resident = resident_ctas(blend_kernel, BT, 0, 8);
    blend_kernel<<<(unsigned)resident, BT, 0, (cudaStream_t)stream>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_accumulate(uint64_t* cam_best, const float* leaf_colour, int64_t n, float* max_contrib,
                               float* colours, int32_t* first_frame, int32_t frame, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(cam_best && leaf_colour && max_contrib && colours, "null pointer");
    accumulate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (unsigned long long*)cam_best, leaf_colour, n, max_contrib, colours, first_frame, frame);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_compose_image(uint32_t* owner, const float* leaf_colour, int32_t width, int32_t height,
                                  float background, float* image, void* stream) {
    G2PC_CHECK_ARG(width > 0 && height > 0, "bad image size");
    G2PC_CHECK_ARG(owner && leaf_colour && image, "null pointer");
    const int64_t n = (int64_t)width * height;
    compose_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(owner, leaf_colour, width, height,
                                                                                    background, image);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}
