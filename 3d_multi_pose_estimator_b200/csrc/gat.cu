// Stage 2a: fused attention logits + edge-softmax + neighbour aggregation of one GAT layer.
//
// Reference behaviour restated (skeleton_matching/gat2.py):
//   :59-61,78-81  a[e]   = LeakyReLU_alpha(a1[src] + a2[dst])                 (apply_edges UDF)
//   :63,83-88     s[e]   = exp(a[e] - max_dst) / sum_dst exp(...)             (dgl.ops.edge_softmax, by dst)
//   :66           out[v] = sum_{u->v} s[e] * ft2[u]                           (update_all u_mul_e / sum)
//   :141-142      next input = LeakyReLU_0.01(out.flatten(1));  :144-145 sigmoid on the last layer
//
// Four kernels, one arithmetic (softmax through the SFU, sums in ascending reference edge id unless noted):
//   gat_aggregate_frame_kernel  frames of at most 32 heads whose plan fits in shared memory (the Panoptic-sized case):
//                               one CTA per frame, head rows resident, edge-node rows streamed once through a bulk-copy
//                               ring, warp per destination, head accumulators in registers. The product path at 1024 frames.
//   gat_aggregate_large_kernel  frames of more than 48 heads (10 views x 16 persons) and batches of a few frames: edge
//                               units with staged head rows and per-warp cp.async rings, head units with a one-pass
//                               fixed-reference softmax (reassociated sums: equal to fp32 rounding, not bitwise).
//   gat_aggregate_kernel        the general gather kernel: warp per destination over the CSR, any graph.
//   gat_aggregate_scalar_kernel the last layer (one output per node) with the sigmoid fused.
// The host function at the bottom picks one (impl 0) or takes the caller's choice (A/B runs, tests).
//
// gat_aggregate_kernel: one CTA per (frame, chunk of destinations), one warp per destination node walking its CSR row.
// When a frame's heads fit (at most 48 rows) their z rows (and, for layer 0, the single shared edge-node row) are staged
// in shared memory: every edge-node destination reads two head rows and every head reads its own, so 2/3 of the row
// gathers are served on chip; edge-node rows come through the read-only path. Lanes own 4 (or 2) consecutive feature
// columns, so every row read is a coalesced, vectorised sweep.
#include "common.cuh"

namespace b200pose {

struct AggParams {
    int n_frames, n_heads_total;
    const int* head_off; const int* node_off; const int* row_ptr; const int* col;
    const float* z; int ldz; int heads, dim, layer0;
    float alpha, act_slope;
    float* raw_f32; __nv_bfloat16* act_hi; __nv_bfloat16* act_lo; int ld_planes;
    const float* res; int ld_res;   // residual term added to the aggregate before the activation (gat2.py:70-75: res_fc(h)), gather / scalar kernels only
    int stage_rows;     // z rows of shared memory available per CTA for staging
    int chunk;          // destination nodes per CTA (work unit = frame x chunk)
    int n_chunks;       // chunks per frame (grid = n_frames * n_chunks)
    int max_deg;        // largest in-degree (sizes the per-warp attention scratch)
    int stage_cap;      // large-frame kernel: z rows of shared memory per CTA
    int edge_units;     // large-frame kernel: edge-node work units per frame
    int head_units;     // large-frame kernel: head work units per frame
};

template <int VEC> __device__ __forceinline__ void load_vec(const float* p, float (&v)[VEC]) {
    if constexpr (VEC == 4) { float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    else if constexpr (VEC == 2) { float2 t = *reinterpret_cast<const float2*>(p); v[0] = t.x; v[1] = t.y; }
    else v[0] = *p;
}

// Softmax arithmetic of both aggregation kernels: exp(x) for x <= 0 through the SFU (ex2.approx, ~2 ulp) and the
// normalisation through the SFU reciprocal - a softmax weight that is off by 1e-7 relative moves a score by far less
// than the 1e-4 tolerance, and the precise expf/IEEE division cost ~25 issue slots per weight in issue-bound kernels.
// Written as PTX so that every aggregation kernel executes exactly these instructions (their outputs are compared
// bit for bit): ex2.approx.ftz of x*log2(e) - two instructions, no denormal range code - and one SFU reciprocal per
// denominator, shared by the weights that are divided by it (the asm is not volatile: the compiler merges equal rcp's).
__device__ __forceinline__ float soft_exp(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
    return y;
}
__device__ __forceinline__ float soft_rcp(float d) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
    return r;
}
__device__ __forceinline__ float soft_div(float x, float d) { return x * soft_rcp(d); }

constexpr int kAggWarps = 8;

// VEC consecutive columns per lane, KMAX column vectors per lane (heads*dim <= 32*VEC*KMAX)
template <int VEC, int KMAX>
__global__ void __launch_bounds__(kAggWarps * 32) gat_aggregate_kernel(AggParams p)
{
    extern __shared__ __align__(128) float smem_f[];
    // chunk index fastest: the CTAs working on one frame run together, so the z rows of a frame that several of
    // them gather (every edge-node row is read by itself and by its two heads) are served from L2
    const int b = blockIdx.x / p.n_chunks;
    const int n0 = p.node_off[b];
    const int Nb = p.node_off[b + 1] - n0;
    const int v_begin = (blockIdx.x - b * p.n_chunks) * p.chunk;
    if (v_begin >= Nb) return;
    const int v_end = min(Nb, v_begin + p.chunk);
    const int h0 = p.head_off[b];
    const int Hb = p.head_off[b + 1] - h0;
    const int H = p.heads, D = p.dim, HD = H * D;
    const int ldz = p.ldz;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* zs = smem_f;                                                     // staged z rows
    float* att = smem_f + (size_t)p.stage_rows * ldz + (size_t)warp * p.max_deg * H;   // this warp's [deg][H] scratch

    // ---- stage the frame's head rows (layer 0: + the shared edge-node row) ------------------------
    int n_stage;
    bool all_staged = false;
    if (p.layer0) {
        all_staged = (Hb + 1 <= p.stage_rows);
        n_stage = all_staged ? Hb + 1 : 0;
    } else {
        n_stage = min(Hb, p.stage_rows);
    }
    {
        const int vec_per_row = ldz / 4;                       // ldz is a multiple of 4
        const int total = n_stage * vec_per_row;
        for (int i = threadIdx.x; i < total; i += blockDim.x) {
            const int r = i / vec_per_row, c = i - r * vec_per_row;
            size_t grow;
            if (p.layer0) grow = (r < Hb) ? (size_t)(h0 + r) : (size_t)p.n_heads_total;
            else grow = (size_t)(n0 + r);
            reinterpret_cast<float4*>(zs)[i] = __ldg(reinterpret_cast<const float4*>(p.z + grow * ldz) + c);
        }
    }
    __syncthreads();

    auto row_of = [&](int u_global) -> const float* {         // z row of a source node
        const int l = u_global - n0;
        if (p.layer0) {
            if (all_staged) return zs + (size_t)(l < Hb ? l : Hb) * ldz;
            return p.z + (size_t)(l < Hb ? h0 + l : p.n_heads_total) * ldz;
        }
        if (l < n_stage) return zs + (size_t)l * ldz;
        return p.z + (size_t)u_global * ldz;
    };

    const int n_vec = HD / VEC;
    int head_of[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) head_of[k] = min(H - 1, ((lane + 32 * k) * VEC) / D);

    for (int v = v_begin + warp; v < v_end; v += kAggWarps) {
        const int gv = n0 + v;
        const int beg = p.row_ptr[gv];
        const int deg = min(p.row_ptr[gv + 1] - beg, p.max_deg);
        const float* rowv = row_of(gv);
        float acc[KMAX][VEC];
        if (deg == 3 && 3 * H <= 32) {
            // edge-node destination (two heads + self loop): lane t = i * H + h holds the logit and then the softmax
            // weight of in-edge i, attention head h; the three rows are loaded together. Same operation order as below.
            const int i = min(lane / H, 2), h = lane - (lane / H) * H;
            const float* r3[3];
#pragma unroll
            for (int u = 0; u < 3; ++u) r3[u] = row_of(__ldg(p.col + beg + u));
            const float* rme = i == 0 ? r3[0] : (i == 1 ? r3[1] : r3[2]);
            float f[3][KMAX][VEC];
#pragma unroll
            for (int u = 0; u < 3; ++u)
#pragma unroll
                for (int k = 0; k < KMAX; ++k) {
                    const int cv = lane + 32 * k;
                    if (cv < n_vec) load_vec<VEC>(r3[u] + cv * VEC, f[u][k]);
                }
            const float e = lane < 3 * H ? leaky(rme[HD + h] + rowv[HD + H + h], p.alpha) : 0.f;
            const float e0 = __shfl_sync(0xffffffffu, e, h), e1 = __shfl_sync(0xffffffffu, e, H + h), e2 = __shfl_sync(0xffffffffu, e, 2 * H + h);
            const float m = fmaxf(fmaxf(e0, e1), e2);
            const float x0 = soft_exp(e0 - m), x1 = soft_exp(e1 - m), x2 = soft_exp(e2 - m);
            const float den = (x0 + x1) + x2;
            const float wgt = soft_div(i == 0 ? x0 : (i == 1 ? x1 : x2), den);
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                float a[3];
#pragma unroll
                for (int u = 0; u < 3; ++u) a[u] = __shfl_sync(0xffffffffu, wgt, u * H + head_of[k]);
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    float s = fmaf(a[0], f[0][k][q], 0.f);
                    s = fmaf(a[1], f[1][k][q], s);
                    acc[k][q] = fmaf(a[2], f[2][k][q], s);
                }
            }
        } else {
        // 1. attention logits e[i][h] = LeakyReLU(a1[u_i][h] + a2[v][h])            (gat2.py:78-81)
        const int npair = deg * H;
        for (int t = lane; t < npair; t += 32) {
            const int i = t / H, h = t - i * H;
            const float* ru = row_of(__ldg(p.col + beg + i));
            att[t] = leaky(ru[HD + h] + rowv[HD + H + h], p.alpha);
        }
        __syncwarp();
        // 2. softmax over the in-edges of v, per head                                  (gat2.py:83-88)
        float mh = -INFINITY;
        if (lane < H) for (int i = 0; i < deg; ++i) mh = fmaxf(mh, att[i * H + lane]);
        for (int t0 = 0; t0 < npair; t0 += 32) {                // uniform trip count: every lane takes part in the shuffle
            const int t = t0 + lane;
            const float m = __shfl_sync(0xffffffffu, mh, t % H);
            if (t < npair) att[t] = soft_exp(att[t] - m);
        }
        __syncwarp();
        float dh = 0.f;
        if (lane < H) for (int i = 0; i < deg; ++i) dh += att[i * H + lane];
        for (int t0 = 0; t0 < npair; t0 += 32) {
            const int t = t0 + lane;
            const float d = __shfl_sync(0xffffffffu, dh, t % H);
            if (t < npair) att[t] = soft_div(att[t], d);
        }
        __syncwarp();
        // 3. out[v] = sum_i s[i][h] * ft2[u_i]                                        (gat2.py:66)
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[k][i] = 0.f;
        // neighbours in batches of 4: the row loads of a batch are independent and issued together (a head of a
        // 10-view frame has ~145 in-edges; one L2 round trip per neighbour would serialise them), the FMAs keep the
        // ascending-edge order
        for (int i0 = 0; i0 < deg; i0 += 4) {
            const float* ru[4];
            float f[4][KMAX][VEC];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = min(i0 + u, deg - 1);
                ru[u] = row_of(__ldg(p.col + beg + i));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int k = 0; k < KMAX; ++k) {
                    const int cv = lane + 32 * k;
                    if (cv < n_vec) load_vec<VEC>(ru[u] + cv * VEC, f[u][k]);
                }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (i0 + u >= deg) break;
                const float* w = att + (i0 + u) * H;
#pragma unroll
                for (int k = 0; k < KMAX; ++k) {
                    const int cv = lane + 32 * k;
                    if (cv < n_vec) {
                        const float a = w[head_of[k]];
#pragma unroll
                        for (int q = 0; q < VEC; ++q) acc[k][q] = fmaf(a, f[u][k][q], acc[k][q]);
                    }
                }
            }
        }
        __syncwarp();                                           // att is reused by the next destination
        }
        // 4. outputs
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            const int cv = lane + 32 * k;
            if (cv >= n_vec) continue;
            if (p.res) {                                        // ret = resval + ret (gat2.py:75)
                const float* rr = p.res + (size_t)gv * p.ld_res + cv * VEC;
#pragma unroll
                for (int q = 0; q < VEC; ++q) acc[k][q] = rr[q] + acc[k][q];
            }
            if (p.raw_f32) {
                float* o = p.raw_f32 + (size_t)gv * HD + cv * VEC;
#pragma unroll
                for (int q = 0; q < VEC; ++q) o[q] = acc[k][q];
            }
            if (p.act_hi) {
                __nv_bfloat16 hi[VEC], lo[VEC];
#pragma unroll
                for (int q = 0; q < VEC; ++q) split_bf16(leaky(acc[k][q], p.act_slope), hi[q], lo[q]);
                __nv_bfloat16* oh = p.act_hi + (size_t)gv * p.ld_planes + cv * VEC;
                __nv_bfloat16* ol = p.act_lo + (size_t)gv * p.ld_planes + cv * VEC;
                if constexpr (VEC == 4) {
                    *reinterpret_cast<uint2*>(oh) = make_uint2(pack_bf16x2(hi[0], hi[1]), pack_bf16x2(hi[2], hi[3]));
                    *reinterpret_cast<uint2*>(ol) = make_uint2(pack_bf16x2(lo[0], lo[1]), pack_bf16x2(lo[2], lo[3]));
                } else if constexpr (VEC == 2) {
                    *reinterpret_cast<uint32_t*>(oh) = pack_bf16x2(hi[0], hi[1]);
                    *reinterpret_cast<uint32_t*>(ol) = pack_bf16x2(lo[0], lo[1]);
                } else {
                    oh[0] = hi[0]; ol[0] = lo[0];
                }
            }
        }
        if (p.act_hi) {                                         // K padding of the planes stays zero
            for (int c = HD + lane; c < p.ld_planes; c += 32) {
                p.act_hi[(size_t)gv * p.ld_planes + c] = __float2bfloat16_rn(0.f);
                p.act_lo[(size_t)gv * p.ld_planes + c] = __float2bfloat16_rn(0.f);
            }
        }
    }
}


// ------------------------------------------------------------------------------------------------
// Frame-resident kernel (the product path whenever a frame's plan fits in shared memory).
//
// One CTA per frame: 16 consumer warps + 1 producer warp. Every z row of the frame leaves HBM exactly once
// per layer:
//   * the head rows (and their a1|a2 attention scalars) are staged in shared memory for the whole frame;
//   * the edge-node rows - one contiguous block of M_b rows - stream through a kSlots-deep shared-memory ring
//     in chunks of kChunkRows rows, fetched by 1-D bulk async copies (cp.async.bulk, mbarrier complete_tx)
//     issued by the producer warp; consumer warps hand a slot back through an "empty" mbarrier, so there is
//     no CTA-wide barrier in the steady state and the copies of later chunks overlap the arithmetic;
//   * per chunk, consumer warp w takes (a) edge-node destination k0+w - warp per destination: two head rows +
//     the node's own row from shared memory, its three softmax weights computed on the fly from the a1|a2
//     columns of those rows - and (b) the contributions of the chunk's rows to the head destinations it owns
//     (heads w and w+16; their accumulators stay in registers across chunks, their in-edge lists are walked in
//     ascending edge id with weights precomputed in phase 1).
// Lanes own VEC consecutive columns of KMAX column groups: every row access is a coalesced vector sweep.
// The summation order per output element is ascending reference edge id, exactly as in the gather kernel.
//   phase 1: stage head rows, a1|a2 of heads, a1 of edge-nodes, in-edge lists of the heads; one thread per
//            (head destination, attention head) computes the softmax weights of its in-edges (gat2.py:78-88)
//   phase 2: chunk loop as above
// ------------------------------------------------------------------------------------------------
constexpr int kFrameWarps = 16;                             // consumer warps
constexpr int kFrameThreads = (kFrameWarps + 1) * 32;       // + the producer warp
constexpr int kFrameOwn = 2;                                // head destinations per consumer warp
constexpr int kChunkRows = kFrameWarps;                     // one edge-node destination per consumer warp and chunk
constexpr int kSlots = 4;

__device__ __forceinline__ uint32_t agg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void agg_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void agg_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void agg_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void agg_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        if (clock64() - t0 > 4000000000LL) __trap();      // a lost copy becomes an error, not a hang
    }
}
__device__ __forceinline__ void agg_cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void agg_cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void agg_bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

struct FramePlan {          // shared-memory plan of one frame (element offsets into a float array)
    int ring, zh, ze, ah, a1e, wh, lsth, prs, total_floats;
};

__host__ __device__ inline FramePlan frame_plan(int max_heads, int max_enodes, int HD, int H, int ldz) {
    FramePlan f;
    const int hd4 = (HD + 3) & ~3;
    const int e_heads = max_heads + 2 * max_enodes;                     // in-edges of all head destinations of a frame
    int o = 0;
    f.ring = o; o += kSlots * kChunkRows * ldz;                         // bulk-copy destinations first: 16-byte aligned
    f.zh = o; o += max_heads * hd4;
    f.ze = o; o += ldz;                                                 // layer 0: the shared edge-node row, a1|a2 included
    f.ah = o; o += (max_heads * 2 * H + 3) & ~3;                        // a1|a2 of the heads
    f.a1e = o; o += (max_enodes * H + 3) & ~3;                          // a1 of the edge-nodes (phase 1)
    f.wh = o; o += (e_heads * H + 3) & ~3;                              // softmax weights of the heads' in-edges, CSR order
    f.lsth = o; o += (e_heads + 3) & ~3;                                // frame-local sources of the heads' in-edges
    f.prs = o; o += (2 * max_enodes + 3) & ~3;                          // (h1, h2) of every edge-node
    f.total_floats = o;
    return f;
}

template <int VEC> struct VecT;
template <> struct VecT<4> { using type = float4; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<1> { using type = float; };

template <int VEC> __device__ __forceinline__ void store_out(const AggParams& p, bool slope_le1, int gv, int c0, const float (&v)[VEC]) {
    if (p.raw_f32) {
        float* o = p.raw_f32 + (size_t)gv * (p.heads * p.dim) + c0;
#pragma unroll
        for (int q = 0; q < VEC; ++q) o[q] = v[q];
    }
    if (p.act_hi) {
        float a[VEC];
        if (slope_le1) {
#pragma unroll
            for (int q = 0; q < VEC; ++q) a[q] = leaky_le1(v[q], p.act_slope);
        } else {
#pragma unroll
            for (int q = 0; q < VEC; ++q) a[q] = leaky(v[q], p.act_slope);
        }
        __nv_bfloat16* oh = p.act_hi + (size_t)gv * p.ld_planes + c0;
        __nv_bfloat16* ol = p.act_lo + (size_t)gv * p.ld_planes + c0;
        if constexpr (VEC == 4) {
            uint32_t h0, l0, h1, l1;
            split_pack2(a[0], a[1], h0, l0);
            split_pack2(a[2], a[3], h1, l1);
            *reinterpret_cast<uint2*>(oh) = make_uint2(h0, h1);
            *reinterpret_cast<uint2*>(ol) = make_uint2(l0, l1);
        } else if constexpr (VEC == 2) {
            uint32_t h0, l0;
            split_pack2(a[0], a[1], h0, l0);
            *reinterpret_cast<uint32_t*>(oh) = h0;
            *reinterpret_cast<uint32_t*>(ol) = l0;
        } else {
            __nv_bfloat16 h, l;
            split_bf16(a[0], h, l);
            oh[0] = h; ol[0] = l;
        }
    }
}

template <int VEC, int KMAX>
__global__ void __launch_bounds__(kFrameThreads, 1) gat_aggregate_frame_kernel(AggParams p, int max_heads, int max_enodes)
{
    extern __shared__ __align__(128) float smem_f[];
    __shared__ __align__(8) uint64_t bar_full[kSlots];
    __shared__ __align__(8) uint64_t bar_empty[kSlots];
    __shared__ __align__(8) uint64_t bar_wh;                  // the heads' softmax weights (phase 1b) are complete
    const int b = blockIdx.x;
    const int n0 = p.node_off[b];
    const int Nb = p.node_off[b + 1] - n0;
    if (Nb == 0) return;
    const int h0 = p.head_off[b];
    const int Hb = p.head_off[b + 1] - h0;
    const int Mb = Nb - Hb;
    const int Eh = Hb + 2 * Mb;                             // in-edges of the head destinations (CSR: head rows come first)
    const int e0 = h0 + 5 * (n0 - h0);                      // first edge (CSR position) of the frame
    const int H = p.heads, D = p.dim, HD = H * D, ldz = p.ldz;
    const int hd4 = (HD + 3) & ~3;
    const FramePlan f = frame_plan(max_heads, max_enodes, HD, H, ldz);
    float* ring = smem_f + f.ring;
    float* zh = smem_f + f.zh;
    float* zE = smem_f + f.ze;
    float* ah = smem_f + f.ah;
    float* a1e = smem_f + f.a1e;
    float* wh = smem_f + f.wh;
    int* lsth = reinterpret_cast<int*>(smem_f + f.lsth);
    int* prs = reinterpret_cast<int*>(smem_f + f.prs);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const bool streamed = !p.layer0 && Mb > 0;
    const int n_chunks = (Mb + kChunkRows - 1) / kChunkRows;
    const float* zen = p.z + (size_t)(n0 + Hb) * ldz;       // first edge-node row of the frame (not layer 0)
    auto issue_chunk = [&](int c) {                         // one thread: bulk copy of chunk c into ring slot c % kSlots
        const int rows = min(kChunkRows, Mb - c * kChunkRows);
        const uint32_t bytes = (uint32_t)rows * (uint32_t)ldz * 4u;
        const uint32_t bar = agg_smem_u32(&bar_full[c % kSlots]);
        agg_mbar_expect_tx(bar, bytes);
        agg_bulk_load(agg_smem_u32(ring + (size_t)(c % kSlots) * kChunkRows * ldz), zen + (size_t)c * kChunkRows * ldz, bytes, bar);
    };
    if (tid == kFrameWarps * 32) {                          // lane 0 of the producer warp
#pragma unroll
        for (int s = 0; s < kSlots; ++s) { agg_mbar_init(agg_smem_u32(&bar_full[s]), 1); agg_mbar_init(agg_smem_u32(&bar_empty[s]), kFrameWarps); }
        agg_mbar_init(agg_smem_u32(&bar_wh), kFrameWarps + 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (streamed)
            for (int c = 0; c < kSlots && c < n_chunks; ++c) issue_chunk(c);
    }
    // z row of frame-local node l
    auto zrow = [&](int l) -> const float* {
        if (p.layer0) return p.z + (size_t)(l < Hb ? h0 + l : p.n_heads_total) * ldz;
        return p.z + (size_t)(n0 + l) * ldz;
    };
    // ---- phase 1a: stage the head rows, a1|a2 of the heads, a1 of the edge-nodes, the heads' in-edge lists ----
    // Everything goes through cp.async (global -> shared without a register round trip): the five tables are issued
    // back to back and waited for once, instead of paying one global-memory latency per table. The CSR columns are
    // staged raw (global node ids); n0 is subtracted where they are used.
    {
        const int vec_per_row = hd4 / 4;                    // ldz % 4 == 0 and columns [HD, hd4) exist in the row (a1 follows)
        for (int i = tid; i < Hb * vec_per_row; i += kFrameThreads) {
            const int r = i / vec_per_row, c = i - r * vec_per_row;
            agg_cp_async16(agg_smem_u32(zh + (size_t)r * hd4 + 4 * c), zrow(r) + 4 * c);
        }
        if (p.layer0)
            for (int i = tid; i < ldz / 4; i += kFrameThreads) agg_cp_async16(agg_smem_u32(zE + 4 * i), zrow(Hb) + 4 * i);
    }
    for (int i = tid; i < Hb * 2 * H; i += kFrameThreads) {
        const int r = i / (2 * H), c = i - r * 2 * H;
        agg_cp_async4(agg_smem_u32(ah + i), zrow(r) + HD + c);
    }
    if (!p.layer0)
        for (int i = tid; i < Mb * H; i += kFrameThreads) {
            const int r = i / H, c = i - r * H;
            agg_cp_async4(agg_smem_u32(a1e + i), zen + (size_t)r * ldz + HD + c);
        }
    for (int i = tid; i < Eh; i += kFrameThreads) agg_cp_async4(agg_smem_u32(lsth + i), p.col + e0 + i);
    for (int k = tid; k < Mb; k += kFrameThreads) {
        const int q = e0 + Eh + 3 * k;                      // CSR: 3 in-edges per edge-node after the head rows: h1, h2, self
        agg_cp_async4(agg_smem_u32(prs + 2 * k), p.col + q);
        agg_cp_async4(agg_smem_u32(prs + 2 * k + 1), p.col + q + 1);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    // ---- phase 1b: softmax weights of the heads' in-edges, per attention head (gat2.py:78-88) ----
    for (int q = tid; q < Hb * H; q += kFrameThreads) {
        const int v = q / H, hh = q - v * H;
        const int beg = __ldg(p.row_ptr + n0 + v) - e0;
        const int deg = __ldg(p.row_ptr + n0 + v + 1) - e0 - beg;
        const float a2v = ah[v * 2 * H + H + hh];
        float* wv = wh + (size_t)beg * H + hh;
        float m = -INFINITY;
        for (int i = 0; i < deg; ++i) {
            const int u = lsth[beg + i] - n0;
            const float a1u = (u < Hb) ? ah[u * 2 * H + hh] : (p.layer0 ? zE[HD + hh] : a1e[(u - Hb) * H + hh]);
            const float e = leaky(a1u + a2v, p.alpha);
            wv[i * H] = e;
            m = fmaxf(m, e);
        }
        float den = 0.f;
        for (int i = 0; i < deg; ++i) {
            const float e = soft_exp(wv[i * H] - m);
            wv[i * H] = e;
            den += e;
        }
        for (int i = 0; i < deg; ++i) wv[i * H] = soft_div(wv[i * H], den);
    }
    // no CTA barrier here: only part (b) of the chunk loop reads the heads' weights, so every warp just reports its share
    // of phase 1b done and the consumers wait for all reports after the edge-node destinations of their first chunk
    __syncwarp();
    if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_wh));
    // ---- phase 2 ----
    if (wid == kFrameWarps) {
        // ===== producer warp: refill a slot as soon as all consumer warps have released it =====
        if (lane == 0 && streamed) {
            for (int c = kSlots; c < n_chunks; ++c) {
                const int s = c % kSlots;
                agg_mbar_wait(agg_smem_u32(&bar_empty[s]), (uint32_t)(c / kSlots - 1) & 1u);
                issue_chunk(c);
            }
        }
        return;
    }
    const int n_vec = HD / VEC;
    using V = typename VecT<VEC>::type;
    const bool slope_le1 = p.act_slope >= 0.f && p.act_slope <= 1.f;
    int cj[KMAX], hj[KMAX];
    bool okj[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
        const int cv = lane + 32 * j;
        okj[j] = cv < n_vec;
        cj[j] = okj[j] ? cv * VEC : 0;
        hj[j] = cj[j] / D;
    }
    // owned head destinations: accumulators in registers, initialised with the self loop (first in-edge of the row) once the
    // heads' weights are known
    float acc[kFrameOwn][KMAX][VEC];
    int hbeg[kFrameOwn], hdeg[kFrameOwn], hcur[kFrameOwn];
#pragma unroll
    for (int t = 0; t < kFrameOwn; ++t) {
        const int h = wid + t * kFrameWarps;
        hbeg[t] = 0; hdeg[t] = 0; hcur[t] = 1;
        if (h < Hb) {
            hbeg[t] = __ldg(p.row_ptr + n0 + h) - e0;
            hdeg[t] = __ldg(p.row_ptr + n0 + h + 1) - e0 - hbeg[t];
        }
    }
    auto init_acc = [&]() {
        agg_mbar_wait(agg_smem_u32(&bar_wh), 0u);
#pragma unroll
        for (int t = 0; t < kFrameOwn; ++t) {
            const int h = wid + t * kFrameWarps;
#pragma unroll
            for (int j = 0; j < KMAX; ++j) {
                float zv[VEC];
#pragma unroll
                for (int q = 0; q < VEC; ++q) zv[q] = 0.f;
                float a = 0.f;
                if (h < Hb && okj[j]) {
                    *reinterpret_cast<V*>(zv) = *reinterpret_cast<const V*>(zh + (size_t)h * hd4 + cj[j]);
                    a = wh[(size_t)hbeg[t] * H + hj[j]];
                }
#pragma unroll
                for (int q = 0; q < VEC; ++q) acc[t][j][q] = fmaf(a, zv[q], 0.f);
            }
        }
    };
    if (n_chunks == 0) init_acc();
    const int lh = lane < H ? lane : 0;                     // attention head whose edge-node softmax this lane computes
    for (int c = 0; c < n_chunks; ++c) {
        const int k0 = c * kChunkRows, k1 = min(Mb, k0 + kChunkRows);
        const int slot = c % kSlots;
        const float* rows = zE;
        int rstride = 0;
        if (!p.layer0) {
            agg_mbar_wait(agg_smem_u32(&bar_full[slot]), (uint32_t)(c / kSlots) & 1u);
            rows = ring + (size_t)slot * kChunkRows * ldz;
            rstride = ldz;
        }
        // (a) the edge-node destination of this warp: in-edges (h1 -> e), (h2 -> e), (e -> e)
        const int k = k0 + wid;
        if (k < k1) {
            const int h1 = prs[2 * k] - n0, h2 = prs[2 * k + 1] - n0;
            const float* re = rows + (size_t)(k - k0) * rstride;
            // softmax of the three logits, attention head lh (lanes >= H repeat head 0; nobody reads them)
            const float a2e = re[HD + H + lh];
            const float e1 = leaky(ah[h1 * 2 * H + lh] + a2e, p.alpha);
            const float e2 = leaky(ah[h2 * 2 * H + lh] + a2e, p.alpha);
            const float e3 = leaky(re[HD + lh] + a2e, p.alpha);
            const float m = fmaxf(fmaxf(e1, e2), e3);
            const float x1 = soft_exp(e1 - m), x2 = soft_exp(e2 - m), x3 = soft_exp(e3 - m);
            const float den = (0.f + x1 + x2) + x3;
            const float s1 = soft_div(x1, den), s2 = soft_div(x2, den), s3 = soft_div(x3, den);
#pragma unroll
            for (int j = 0; j < KMAX; ++j) {
                const float w1 = __shfl_sync(0xffffffffu, s1, hj[j]);
                const float w2 = __shfl_sync(0xffffffffu, s2, hj[j]);
                const float w3 = __shfl_sync(0xffffffffu, s3, hj[j]);
                if (!okj[j]) continue;
                float z1[VEC], z2[VEC], ze[VEC], o[VEC];
                *reinterpret_cast<V*>(z1) = *reinterpret_cast<const V*>(zh + (size_t)h1 * hd4 + cj[j]);
                *reinterpret_cast<V*>(z2) = *reinterpret_cast<const V*>(zh + (size_t)h2 * hd4 + cj[j]);
                *reinterpret_cast<V*>(ze) = *reinterpret_cast<const V*>(re + cj[j]);
#pragma unroll
                for (int q = 0; q < VEC; ++q) o[q] = fmaf(w3, ze[q], fmaf(w2, z2[q], fmaf(w1, z1[q], 0.f)));
                store_out<VEC>(p, slope_le1, n0 + Hb + k, cj[j], o);
            }
        }
        // (b) contributions of the chunk's rows to the owned heads, ascending edge id
        if (c == 0) init_acc();
#pragma unroll
        for (int t = 0; t < kFrameOwn; ++t) {
            while (hcur[t] < hdeg[t]) {
                const int pos = hbeg[t] + hcur[t];
                const int kk = lsth[pos] - n0 - Hb;
                if (kk >= k1) break;
                const float* re = rows + (size_t)(kk - k0) * rstride;
                const float* wp = wh + (size_t)pos * H;
#pragma unroll
                for (int j = 0; j < KMAX; ++j) {
                    if (!okj[j]) continue;
                    float ze[VEC];
                    *reinterpret_cast<V*>(ze) = *reinterpret_cast<const V*>(re + cj[j]);
                    const float a = wp[hj[j]];
#pragma unroll
                    for (int q = 0; q < VEC; ++q) acc[t][j][q] = fmaf(a, ze[q], acc[t][j][q]);
                }
                ++hcur[t];
            }
        }
        if (streamed) {                                     // this warp is done with the slot
            __syncwarp();
            if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_empty[slot]));
        }
    }
#pragma unroll
    for (int t = 0; t < kFrameOwn; ++t) {
        const int h = wid + t * kFrameWarps;
        if (h >= Hb) continue;
#pragma unroll
        for (int j = 0; j < KMAX; ++j)
            if (okj[j]) store_out<VEC>(p, slope_le1, n0 + h, cj[j], acc[t][j]);
    }
    if (p.act_hi && p.ld_planes > HD) {                     // K padding of the planes stays zero
        const int padc = p.ld_planes - HD;
        const int nthr = kFrameWarps * 32;
        if ((HD & 7) == 0) {                                // 16-byte stores (ld_planes is a multiple of 64)
            const int pv = padc / 8;
            for (int i = tid; i < Nb * pv; i += nthr) {
                const int r = i / pv, cc = HD + 8 * (i - r * pv);
                *reinterpret_cast<uint4*>(p.act_hi + (size_t)(n0 + r) * p.ld_planes + cc) = make_uint4(0, 0, 0, 0);
                *reinterpret_cast<uint4*>(p.act_lo + (size_t)(n0 + r) * p.ld_planes + cc) = make_uint4(0, 0, 0, 0);
            }
        } else {
            for (int i = tid; i < Nb * padc; i += nthr) {
                const int r = i / padc, cc = HD + (i - r * padc);
                p.act_hi[(size_t)(n0 + r) * p.ld_planes + cc] = __float2bfloat16_rn(0.f);
                p.act_lo[(size_t)(n0 + r) * p.ld_planes + cc] = __float2bfloat16_rn(0.f);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Shape-specialised frame-resident kernel: the product path for the layer shapes of the shipped model
// (heads x dim = 10x40, 8x40, 5x30; train_skeleton_matching.py:45-46). Same algorithm, same summation order and the
// same arithmetic as gat_aggregate_frame_kernel above - the outputs are bit-identical - but every size is a
// compile-time constant and the instruction stream is cut down, because the generic kernel is issue-bound, not
// memory-bound (ncu, profiles/r02_agg_before.md: 56 % issue-slot utilisation at 3.9 warps per scheduler, 125 k
// warp-instructions per frame of which 11 % are the FMAs):
//   * the head rows arrive as ONE bulk copy (they are contiguous, a1|a2 tails included: no separate attention table);
//   * row / plane addresses are formed once per destination, column offsets are immediates;
//   * the K padding of the output planes is written by the lanes that idle in the last column group (no extra pass);
//   * barrier waits poll without reading the clock; no fp32 side output (that takes the generic kernel).
// ------------------------------------------------------------------------------------------------
template <int H, int D> struct FrameShape {
    static constexpr int HD = H * D;
    static constexpr int LDZ = (HD + 2 * H + 3) & ~3;
    static constexpr int VEC = (HD % 4 == 0) ? 4 : ((HD % 2 == 0) ? 2 : 1);
    static constexpr int NV = HD / VEC;                       // column vectors per row
    static constexpr int KMAX = (NV + 31) / 32;               // column vectors per lane
    static constexpr int LDP = (HD + 63) / 64 * 64;           // row pitch of the output planes
    static constexpr int NVP = LDP / VEC;                     // column vectors per plane row, K padding included
};

struct FramePlanS { int ring, zh, ze, a1e, wh, lsth, prs, total_floats; };

template <int H, int D>
__host__ __device__ inline FramePlanS frame_plan_s(int max_heads, int max_enodes) {
    using S = FrameShape<H, D>;
    FramePlanS f;
    const int e_heads = max_heads + 2 * max_enodes;
    int o = 0;
    f.ring = o; o += kSlots * kChunkRows * S::LDZ;            // bulk-copy destinations first: 16-byte aligned
    f.zh = o; o += max_heads * S::LDZ;                        // head rows, a1|a2 included
    f.ze = o; o += S::LDZ;                                    // layer 0: the shared edge-node row
    f.a1e = o; o += (max_enodes * H + 3) & ~3;
    f.wh = o; o += (e_heads * H + 3) & ~3;
    f.lsth = o; o += (e_heads + 3) & ~3;
    f.prs = o; o += (2 * max_enodes + 3) & ~3;
    f.total_floats = o;
    return f;
}

__device__ __forceinline__ void agg_mbar_wait_spin(uint32_t bar, uint32_t parity, uint32_t hint = 1000u) {
    uint32_t done = 0, spins = 0;
    while (true) {
        // the hint lets the hardware park the warp for up to ~1 us instead of returning to the polling loop at once
        // (the persistent kernel measured the same with hints from 0 to 100000 ns)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity), "r"(hint) : "memory");
        if (done) break;
        if (++spins == (1u << 24)) __trap();                  // a lost copy becomes an error, not a hang
    }
}

template <int VEC> __device__ __forceinline__ void store_planes_vec(__nv_bfloat16* oh, __nv_bfloat16* ol, const float (&a)[VEC]) {
    if constexpr (VEC == 4) {
        uint32_t h0, l0, h1, l1;
        split_pack2(a[0], a[1], h0, l0);
        split_pack2(a[2], a[3], h1, l1);
        *reinterpret_cast<uint2*>(oh) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(ol) = make_uint2(l0, l1);
    } else if constexpr (VEC == 2) {
        uint32_t h0, l0;
        split_pack2(a[0], a[1], h0, l0);
        *reinterpret_cast<uint32_t*>(oh) = h0;
        *reinterpret_cast<uint32_t*>(ol) = l0;
    } else {
        __nv_bfloat16 h, l;
        split_bf16(a[0], h, l);
        oh[0] = h; ol[0] = l;
    }
}
template <int VEC> __device__ __forceinline__ void store_planes_zero(__nv_bfloat16* oh, __nv_bfloat16* ol) {
    if constexpr (VEC == 4) { *reinterpret_cast<uint2*>(oh) = make_uint2(0, 0); *reinterpret_cast<uint2*>(ol) = make_uint2(0, 0); }
    else if constexpr (VEC == 2) { *reinterpret_cast<uint32_t*>(oh) = 0u; *reinterpret_cast<uint32_t*>(ol) = 0u; }
    else { oh[0] = __float2bfloat16_rn(0.f); ol[0] = __float2bfloat16_rn(0.f); }
}

template <int H, int D, bool L0>
__global__ void __launch_bounds__(kFrameThreads, 1) gat_aggregate_frame_s_kernel(AggParams p, int max_heads, int max_enodes)
{
    using S = FrameShape<H, D>;
    constexpr int HD = S::HD, LDZ = S::LDZ, VEC = S::VEC, NV = S::NV, KMAX = S::KMAX, LDP = S::LDP, NVP = S::NVP;
    using V = typename VecT<VEC>::type;
    extern __shared__ __align__(128) float smem_f[];
    __shared__ __align__(8) uint64_t bar_full[kSlots];
    __shared__ __align__(8) uint64_t bar_empty[kSlots];
    __shared__ __align__(8) uint64_t bar_wh;                  // the heads' softmax weights (phase 1b) are complete
    __shared__ __align__(8) uint64_t bar_heads;               // the head rows (bulk copy) have landed
    const int b = blockIdx.x;
    const int n0 = __ldg(p.node_off + b);
    const int Nb = __ldg(p.node_off + b + 1) - n0;
    if (Nb == 0) return;
    const int h0 = __ldg(p.head_off + b);
    const int Hb = __ldg(p.head_off + b + 1) - h0;
    const int Mb = Nb - Hb;
    const int Eh = Hb + 2 * Mb;                             // in-edges of the head destinations (CSR: head rows come first)
    const int e0 = h0 + 5 * (n0 - h0);                      // first edge (CSR position) of the frame
    const FramePlanS f = frame_plan_s<H, D>(max_heads, max_enodes);
    float* ring = smem_f + f.ring;
    float* zh = smem_f + f.zh;
    float* zE = smem_f + f.ze;
    float* a1e = smem_f + f.a1e;
    float* wh = smem_f + f.wh;
    int* lsth = reinterpret_cast<int*>(smem_f + f.lsth);
    int* prs = reinterpret_cast<int*>(smem_f + f.prs);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const bool streamed = !L0 && Mb > 0;
    const int n_chunks = (Mb + kChunkRows - 1) / kChunkRows;
    // the frame's head rows are contiguous (layer 0: rows h0.. of the compact matrix), its edge-node rows follow them
    const float* zheads = p.z + (size_t)(L0 ? h0 : n0) * LDZ;
    const float* zen = L0 ? p.z + (size_t)p.n_heads_total * LDZ : p.z + (size_t)(n0 + Hb) * LDZ;
    auto issue_chunk = [&](int c) {                         // one thread: bulk copy of chunk c into ring slot c % kSlots
        const int rows = min(kChunkRows, Mb - c * kChunkRows);
        const uint32_t bytes = (uint32_t)rows * (uint32_t)(LDZ * 4);
        const uint32_t bar = agg_smem_u32(&bar_full[c % kSlots]);
        agg_mbar_expect_tx(bar, bytes);
        agg_bulk_load(agg_smem_u32(ring + (size_t)(c % kSlots) * kChunkRows * LDZ), zen + (size_t)c * kChunkRows * LDZ, bytes, bar);
    };
    if (tid == kFrameWarps * 32) {                          // lane 0 of the producer warp
#pragma unroll
        for (int s = 0; s < kSlots; ++s) { agg_mbar_init(agg_smem_u32(&bar_full[s]), 1); agg_mbar_init(agg_smem_u32(&bar_empty[s]), kFrameWarps); }
        agg_mbar_init(agg_smem_u32(&bar_wh), kFrameWarps + 1);
        agg_mbar_init(agg_smem_u32(&bar_heads), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t hb_bytes = (uint32_t)Hb * (uint32_t)(LDZ * 4);
        agg_mbar_expect_tx(agg_smem_u32(&bar_heads), hb_bytes + (L0 ? (uint32_t)(LDZ * 4) : 0u));
        agg_bulk_load(agg_smem_u32(zh), zheads, hb_bytes, agg_smem_u32(&bar_heads));
        if (L0) agg_bulk_load(agg_smem_u32(zE), zen, (uint32_t)(LDZ * 4), agg_smem_u32(&bar_heads));
        if (streamed)
            for (int c = 0; c < kSlots && c < n_chunks; ++c) issue_chunk(c);
    }
    // the CSR bounds phase 1b needs are requested now, so their latency overlaps the staging
    const float alpha = p.alpha, act_slope = p.act_slope;
    int rp_beg = 0, rp_end = 0;
    if (tid < Hb * H) { rp_beg = __ldg(p.row_ptr + n0 + tid / H); rp_end = __ldg(p.row_ptr + n0 + tid / H + 1); }
    // ---- phase 1a: a1 of the edge-nodes, the heads' in-edge lists, (h1, h2) of every edge-node: small gathers through
    // cp.async, issued back to back and waited for once ----
    if (!L0)
        for (int i = tid; i < Mb * H; i += kFrameThreads) {
            const int r = i / H, c = i - r * H;
            agg_cp_async4(agg_smem_u32(a1e + i), zen + (size_t)r * LDZ + HD + c);
        }
    for (int i = tid; i < Eh; i += kFrameThreads) agg_cp_async4(agg_smem_u32(lsth + i), p.col + e0 + i);
    for (int k = tid; k < Mb; k += kFrameThreads) {
        const int q = e0 + Eh + 3 * k;                      // CSR: 3 in-edges per edge-node after the head rows: h1, h2, self
        agg_cp_async4(agg_smem_u32(prs + 2 * k), p.col + q);
        agg_cp_async4(agg_smem_u32(prs + 2 * k + 1), p.col + q + 1);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();                                        // tables visible; the barriers are initialised past this point
    agg_mbar_wait_spin(agg_smem_u32(&bar_heads), 0u);
    // ---- phase 1b: softmax weights of the heads' in-edges, per attention head (gat2.py:78-88) ----
    for (int q = tid; q < Hb * H; q += kFrameThreads) {
        const int v = q / H, hh = q - v * H;
        const int beg = (q == tid ? rp_beg : __ldg(p.row_ptr + n0 + v)) - e0;
        const int deg = (q == tid ? rp_end : __ldg(p.row_ptr + n0 + v + 1)) - e0 - beg;
        const float a2v = zh[v * LDZ + HD + H + hh];
        float* wv = wh + (size_t)beg * H + hh;
        float m = -INFINITY;
        for (int i = 0; i < deg; ++i) {
            const int u = lsth[beg + i] - n0;
            const float a1u = (u < Hb) ? zh[u * LDZ + HD + hh] : (L0 ? zE[HD + hh] : a1e[(u - Hb) * H + hh]);
            const float e = leaky_le1(a1u + a2v, alpha);
            wv[i * H] = e;
            m = fmaxf(m, e);
        }
        float den = 0.f;
        for (int i = 0; i < deg; ++i) {
            const float e = soft_exp(wv[i * H] - m);
            wv[i * H] = e;
            den += e;
        }
        for (int i = 0; i < deg; ++i) wv[i * H] = soft_div(wv[i * H], den);
    }
    __syncwarp();
    if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_wh));
    // ---- phase 2 ----
    if (wid == kFrameWarps) {
        if (lane == 0 && streamed) {
            for (int c = kSlots; c < n_chunks; ++c) {
                const int s = c % kSlots;
                agg_mbar_wait_spin(agg_smem_u32(&bar_empty[s]), (uint32_t)(c / kSlots - 1) & 1u);
                issue_chunk(c);
            }
        }
        return;
    }
    // lane geometry: column vector cv = lane + 32 j, first column cv * VEC, attention head of that column
    int hj[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) hj[j] = min(H - 1, ((lane + 32 * j) * VEC) / D);
    const int lcol = lane * VEC;
    auto col_ok = [&](int j) -> bool { return 32 * (j + 1) <= NV ? true : lane + 32 * j < NV; };      // compile-time true for full groups
    auto pad_ok = [&](int j) -> bool { return lane + 32 * j < NVP; };
    float acc[kFrameOwn][KMAX][VEC];
    int hbeg[kFrameOwn], hdeg[kFrameOwn], hcur[kFrameOwn];
#pragma unroll
    for (int t = 0; t < kFrameOwn; ++t) {
        const int h = wid + t * kFrameWarps;
        hbeg[t] = 0; hdeg[t] = 0; hcur[t] = 1;
        if (h < Hb) {
            hbeg[t] = __ldg(p.row_ptr + n0 + h) - e0;
            hdeg[t] = __ldg(p.row_ptr + n0 + h + 1) - e0 - hbeg[t];
        }
    }
    auto init_acc = [&]() {
        agg_mbar_wait_spin(agg_smem_u32(&bar_wh), 0u);
#pragma unroll
        for (int t = 0; t < kFrameOwn; ++t) {
            const int h = wid + t * kFrameWarps;
            const float* zr = zh + (size_t)(h < Hb ? h : 0) * LDZ + lcol;
            const float* wr = wh + (size_t)hbeg[t] * H;
#pragma unroll
            for (int j = 0; j < KMAX; ++j) {
                float zv[VEC];
#pragma unroll
                for (int q = 0; q < VEC; ++q) zv[q] = 0.f;
                float a = 0.f;
                if (h < Hb && col_ok(j)) {
                    *reinterpret_cast<V*>(zv) = *reinterpret_cast<const V*>(zr + 32 * VEC * j);
                    a = wr[hj[j]];
                }
#pragma unroll
                for (int q = 0; q < VEC; ++q) acc[t][j][q] = fmaf(a, zv[q], 0.f);
            }
        }
    };
    if (n_chunks == 0) init_acc();
    const int lh = lane < H ? lane : 0;                     // attention head whose edge-node softmax this lane computes
    __nv_bfloat16* const out_hi = p.act_hi + (size_t)n0 * LDP + lcol;
    __nv_bfloat16* const out_lo = p.act_lo + (size_t)n0 * LDP + lcol;
    for (int c = 0; c < n_chunks; ++c) {
        const int k0 = c * kChunkRows, k1 = min(Mb, k0 + kChunkRows);
        const int slot = c % kSlots;
        const float* rows = zE;
        if (!L0) {
            agg_mbar_wait_spin(agg_smem_u32(&bar_full[slot]), (uint32_t)(c / kSlots) & 1u);
            rows = ring + (size_t)slot * kChunkRows * LDZ;
        }
        // (a) the edge-node destination of this warp: in-edges (h1 -> e), (h2 -> e), (e -> e)
        const int k = k0 + wid;
        if (k < k1) {
            const int h1 = prs[2 * k] - n0, h2 = prs[2 * k + 1] - n0;
            const float* re = L0 ? rows : rows + (size_t)(k - k0) * LDZ;
            const float* r1 = zh + (size_t)h1 * LDZ;
            const float* r2 = zh + (size_t)h2 * LDZ;
            const float a2e = re[HD + H + lh];
            const float e1 = leaky_le1(r1[HD + lh] + a2e, alpha);        // 0 <= alpha <= 1 here (dispatch): same value as leaky()
            const float e2 = leaky_le1(r2[HD + lh] + a2e, alpha);
            const float e3 = leaky_le1(re[HD + lh] + a2e, alpha);
            const float m = fmaxf(fmaxf(e1, e2), e3);
            const float x1 = soft_exp(e1 - m), x2 = soft_exp(e2 - m), x3 = soft_exp(e3 - m);
            const float den = (0.f + x1 + x2) + x3;
            const float s1 = soft_div(x1, den), s2 = soft_div(x2, den), s3 = soft_div(x3, den);
            __nv_bfloat16* oh = out_hi + (size_t)(Hb + k) * LDP;
            __nv_bfloat16* ol = out_lo + (size_t)(Hb + k) * LDP;
#pragma unroll
            for (int j = 0; j < KMAX; ++j) {
                const float w1 = __shfl_sync(0xffffffffu, s1, hj[j]);
                const float w2 = __shfl_sync(0xffffffffu, s2, hj[j]);
                const float w3 = __shfl_sync(0xffffffffu, s3, hj[j]);
                if (col_ok(j)) {
                    float z1[VEC], z2[VEC], ze[VEC], o[VEC];
                    *reinterpret_cast<V*>(z1) = *reinterpret_cast<const V*>(r1 + lcol + 32 * VEC * j);
                    *reinterpret_cast<V*>(z2) = *reinterpret_cast<const V*>(r2 + lcol + 32 * VEC * j);
                    *reinterpret_cast<V*>(ze) = *reinterpret_cast<const V*>(re + lcol + 32 * VEC * j);
#pragma unroll
                    for (int q = 0; q < VEC; ++q) o[q] = leaky_le1(fmaf(w3, ze[q], fmaf(w2, z2[q], fmaf(w1, z1[q], 0.f))), act_slope);
                    store_planes_vec<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j, o);
                } else if (NVP > NV && pad_ok(j)) {
                    store_planes_zero<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j);        // K padding of the planes stays zero
                }
            }
        }
        // (b) contributions of the chunk's rows to the owned heads, ascending edge id
        if (c == 0) init_acc();
#pragma unroll
        for (int t = 0; t < kFrameOwn; ++t) {
            while (hcur[t] < hdeg[t]) {
                const int pos = hbeg[t] + hcur[t];
                const int kk = lsth[pos] - n0 - Hb;
                if (kk >= k1) break;
                const float* re = (L0 ? rows : rows + (size_t)(kk - k0) * LDZ) + lcol;
                const float* wp = wh + (size_t)pos * H;
#pragma unroll
                for (int j = 0; j < KMAX; ++j) {
                    if (!col_ok(j)) continue;
                    float ze[VEC];
                    *reinterpret_cast<V*>(ze) = *reinterpret_cast<const V*>(re + 32 * VEC * j);
                    const float a = wp[hj[j]];
#pragma unroll
                    for (int q = 0; q < VEC; ++q) acc[t][j][q] = fmaf(a, ze[q], acc[t][j][q]);
                }
                ++hcur[t];
            }
        }
        if (streamed) {                                     // this warp is done with the slot
            __syncwarp();
            if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_empty[slot]));
        }
    }
#pragma unroll
    for (int t = 0; t < kFrameOwn; ++t) {
        const int h = wid + t * kFrameWarps;
        if (h >= Hb) continue;
        __nv_bfloat16* oh = out_hi + (size_t)h * LDP;
        __nv_bfloat16* ol = out_lo + (size_t)h * LDP;
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
            if (col_ok(j)) {
                float o[VEC];
#pragma unroll
                for (int q = 0; q < VEC; ++q) o[q] = leaky_le1(acc[t][j][q], act_slope);
                store_planes_vec<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j, o);
            } else if (NVP > NV && pad_ok(j)) {
                store_planes_zero<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Persistent form of the shape-specialised kernel: one CTA per SM walks frames b = blockIdx.x, += gridDim.x with the
// per-frame set-up taken off the consumers' path. 18 warps:
//   warps 0..15  consumers  - exactly the chunk loop of gat_aggregate_frame_s_kernel (same order, same arithmetic:
//                             bit-identical outputs);
//   warp 16      streamer   - bulk copies of the edge-node rows into the ring, one running chunk sequence across frame
//                             boundaries, so the first chunks of frame f+1 are in flight while frame f is finished;
//   warp 17      preparer   - for frame f+1, into the other of two table sets: head rows (bulk copy), a1 of the
//                             edge-nodes, in-edge lists, (h1, h2) pairs, CSR bounds and the heads' softmax weights.
// With one CTA per frame those ~4 us of dependent loads, staging and weights sat in front of every frame's streaming at
// 4 warps per scheduler; here they run beside the previous frame's arithmetic.
// ------------------------------------------------------------------------------------------------

struct FramePlanP { int ring, set0, set_stride, zh, ze, wh, lsth, prs, meta, a1e, total_floats; };   // zh..a1e: offsets inside a set

template <int H, int D, int W>
__host__ __device__ inline FramePlanP frame_plan_p(int max_heads, int max_enodes, int slots) {
    using S = FrameShape<H, D>;
    FramePlanP f;
    const int e_heads = max_heads + 2 * max_enodes;
    int o = 0;
    f.ring = o; o += slots * W * S::LDZ;                      // a chunk = one edge-node row per consumer warp
    f.set0 = o;
    int q = 0;
    f.zh = q; q += max_heads * S::LDZ;
    f.ze = q; q += S::LDZ;
    f.wh = q; q += (e_heads * H + 3) & ~3;
    f.lsth = q; q += (e_heads + 3) & ~3;
    f.prs = q; q += (2 * max_enodes + 3) & ~3;
    f.meta = q; q += (8 + 2 * max_heads + 3) & ~3;           // n0, h0, Hb, Mb, e0, then (beg, deg) of every head's CSR row
    f.a1e = q; q += (max_enodes * H + 3) & ~3;               // a1 of the edge-nodes (input of the heads' softmax weights)
    f.set_stride = q;
    o += 2 * q;
    f.total_floats = o;
    return f;
}

// W consumer warps, each owning OWN head destinations (frames of at most W * OWN heads): 20 x 1 for frames of up to 20
// heads (5 views x 4 persons) - one head per warp balances part (b), and 22 warps hide the per-chunk latency chain
// better than 18 - and 16 x 2 up to 32 heads (the register file holds 18 warps with two heads' accumulators each).
template <int H, int D, bool L0, int W, int OWN>
__global__ void __launch_bounds__((W + 2) * 32, 1) gat_aggregate_frame_p_kernel(AggParams p, int max_heads, int max_enodes, int slots)
{
    using S = FrameShape<H, D>;
    constexpr int HD = S::HD, LDZ = S::LDZ, VEC = S::VEC, NV = S::NV, KMAX = S::KMAX, LDP = S::LDP, NVP = S::NVP;
    using V = typename VecT<VEC>::type;
    extern __shared__ __align__(128) float smem_f[];
    __shared__ __align__(8) uint64_t bar_full[kSlots];
    __shared__ __align__(8) uint64_t bar_empty[kSlots];
    __shared__ __align__(8) uint64_t bar_rows[2];             // head rows of a set have landed (bulk copy)
    __shared__ __align__(8) uint64_t bar_tab_full[2];         // a set is complete (preparer -> consumers)
    __shared__ __align__(8) uint64_t bar_tab_empty[2];        // a set is free again (consumers -> preparer)
    __shared__ __align__(8) uint64_t bar_wh[2];               // the heads' softmax weights of a set are complete (consumers -> consumers)
    const FramePlanP f = frame_plan_p<H, D, W>(max_heads, max_enodes, slots);
    float* ring = smem_f + f.ring;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int G = gridDim.x;
    if (tid == 0) {
        for (int s = 0; s < kSlots; ++s) { agg_mbar_init(agg_smem_u32(&bar_full[s]), 1); agg_mbar_init(agg_smem_u32(&bar_empty[s]), W); }
        for (int k = 0; k < 2; ++k) {
            agg_mbar_init(agg_smem_u32(&bar_rows[k]), 1);
            agg_mbar_init(agg_smem_u32(&bar_tab_full[k]), 1);
            agg_mbar_init(agg_smem_u32(&bar_tab_empty[k]), W);
            agg_mbar_init(agg_smem_u32(&bar_wh[k]), W);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const float alpha = p.alpha, act_slope = p.act_slope;

    if (wid == W) {
        // ===================== streamer: the ring, one chunk sequence over all frames of this CTA =====================
        if (L0 || lane != 0) return;
        int g = 0;                                                        // running chunk index
        for (int b = blockIdx.x; b < p.n_frames; b += G) {
            const int n0 = __ldg(p.node_off + b), n1 = __ldg(p.node_off + b + 1);
            const int Hb = __ldg(p.head_off + b + 1) - __ldg(p.head_off + b);
            const int Mb = n1 - n0 - Hb;
            const float* zen = p.z + (size_t)(n0 + Hb) * LDZ;
            const int n_chunks = (Mb + W - 1) / W;
            for (int c = 0; c < n_chunks; ++c, ++g) {
                const int s = g % slots;
                if (g >= slots) agg_mbar_wait_spin(agg_smem_u32(&bar_empty[s]), (uint32_t)(g / slots - 1) & 1u);
                const int rows = min(W, Mb - c * W);
                const uint32_t bytes = (uint32_t)rows * (uint32_t)(LDZ * 4);
                const uint32_t bar = agg_smem_u32(&bar_full[s]);
                agg_mbar_expect_tx(bar, bytes);
                agg_bulk_load(agg_smem_u32(ring + (size_t)s * W * LDZ), zen + (size_t)c * W * LDZ, bytes, bar);
            }
        }
        return;
    }
    if (wid == W + 1) {
        // ===================== preparer: table set (i & 1) of local frame i =====================
        int i = 0;
        for (int b = blockIdx.x; b < p.n_frames; b += G, ++i) {
            const int k = i & 1;
            float* set = smem_f + f.set0 + (size_t)k * f.set_stride;
            float* zh = set + f.zh; float* zE = set + f.ze; float* a1e = set + f.a1e;
            int* lsth = reinterpret_cast<int*>(set + f.lsth);
            int* prs = reinterpret_cast<int*>(set + f.prs);
            int* meta = reinterpret_cast<int*>(set + f.meta);
            if (i >= 2) agg_mbar_wait_spin(agg_smem_u32(&bar_tab_empty[k]), (uint32_t)(i / 2 - 1) & 1u);
            const int n0 = __ldg(p.node_off + b), Nb = __ldg(p.node_off + b + 1) - n0;
            const int h0 = __ldg(p.head_off + b), Hb = __ldg(p.head_off + b + 1) - h0;
            const int Mb = Nb - Hb, Eh = Hb + 2 * Mb, e0 = h0 + 5 * (n0 - h0);
            const float* zheads = p.z + (size_t)(L0 ? h0 : n0) * LDZ;
            const float* zen = L0 ? p.z + (size_t)p.n_heads_total * LDZ : p.z + (size_t)(n0 + Hb) * LDZ;
            if (Nb > 0) {
                if (lane == 0) {
                    const uint32_t hb_bytes = (uint32_t)Hb * (uint32_t)(LDZ * 4);
                    const uint32_t bar = agg_smem_u32(&bar_rows[k]);
                    agg_mbar_expect_tx(bar, hb_bytes + (L0 ? (uint32_t)(LDZ * 4) : 0u));
                    agg_bulk_load(agg_smem_u32(zh), zheads, hb_bytes, bar);
                    if (L0) agg_bulk_load(agg_smem_u32(zE), zen, (uint32_t)(LDZ * 4), bar);
                }
                // CSR bounds of the head rows (requested first: phase 1b and the consumers need them)
                for (int v = lane; v < Hb; v += 32) {
                    const int beg = __ldg(p.row_ptr + n0 + v) - e0;
                    meta[8 + 2 * v] = beg;
                    meta[8 + 2 * v + 1] = __ldg(p.row_ptr + n0 + v + 1) - e0 - beg;
                }
                if (!L0)
                    for (int t = lane; t < Mb * H; t += 32) {
                        const int r = t / H, c = t - r * H;
                        agg_cp_async4(agg_smem_u32(a1e + t), zen + (size_t)r * LDZ + HD + c);
                    }
                for (int t = lane; t < Eh; t += 32) agg_cp_async4(agg_smem_u32(lsth + t), p.col + e0 + t);
                for (int t = lane; t < Mb; t += 32) {
                    const int q = e0 + Eh + 3 * t;
                    agg_cp_async4(agg_smem_u32(prs + 2 * t), p.col + q);
                    agg_cp_async4(agg_smem_u32(prs + 2 * t + 1), p.col + q + 1);
                }
                asm volatile("cp.async.wait_all;" ::: "memory");
                __syncwarp();
            }
            if (lane == 0) {
                meta[0] = n0; meta[1] = h0; meta[2] = Hb; meta[3] = Mb; meta[4] = e0;
                if (Nb == 0) agg_mbar_arrive(agg_smem_u32(&bar_rows[k]));      // an empty frame still uses up one phase of its set's barriers
            }
            __syncwarp();
            if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_tab_full[k]));
        }
        return;
    }
    // ===================== consumers =====================
    int hj[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) hj[j] = min(H - 1, ((lane + 32 * j) * VEC) / D);
    const int lcol = lane * VEC;
    auto col_ok = [&](int j) -> bool { return 32 * (j + 1) <= NV ? true : lane + 32 * j < NV; };
    auto pad_ok = [&](int j) -> bool { return lane + 32 * j < NVP; };
    const int lh = lane < H ? lane : 0;
    int g = 0;                                                            // running chunk index (matches the streamer's)
    int i = 0;
    for (int b = blockIdx.x; b < p.n_frames; b += G, ++i) {
        const int ks = i & 1;
        float* set = smem_f + f.set0 + (size_t)ks * f.set_stride;
        const float* zh = set + f.zh; const float* zE = set + f.ze; float* wh = set + f.wh; const float* a1e = set + f.a1e;
        const int* lsth = reinterpret_cast<const int*>(set + f.lsth);
        const int* prs = reinterpret_cast<const int*>(set + f.prs);
        const int* meta = reinterpret_cast<const int*>(set + f.meta);
        agg_mbar_wait_spin(agg_smem_u32(&bar_tab_full[ks]), (uint32_t)(i / 2) & 1u);
        const int n0 = meta[0], Hb = meta[2], Mb = meta[3];
        if (Hb + Mb > 0) {
            agg_mbar_wait_spin(agg_smem_u32(&bar_rows[ks]), (uint32_t)(i / 2) & 1u);     // acquires the copied head rows
            const int n_chunks = (Mb + W - 1) / W;
            // softmax weights of the heads' in-edges, per attention head (gat2.py:78-88): the consumers' own share, reported
            // through bar_wh; only part (b) below reads them, so nobody waits before its first edge-node destination is done
            for (int q = tid; q < Hb * H; q += W * 32) {
                const int v = q / H, hh = q - v * H;
                const int beg = meta[8 + 2 * v], deg = meta[8 + 2 * v + 1];
                const float a2v = zh[v * LDZ + HD + H + hh];
                float* wv = wh + (size_t)beg * H + hh;
                float m = -INFINITY;
                for (int t = 0; t < deg; ++t) {
                    const int u = lsth[beg + t] - n0;
                    const float a1u = (u < Hb) ? zh[u * LDZ + HD + hh] : (L0 ? zE[HD + hh] : a1e[(u - Hb) * H + hh]);
                    const float e = leaky_le1(a1u + a2v, alpha);
                    wv[t * H] = e;
                    m = fmaxf(m, e);
                }
                float den = 0.f;
                for (int t = 0; t < deg; ++t) {
                    const float e = soft_exp(wv[t * H] - m);
                    wv[t * H] = e;
                    den += e;
                }
                for (int t = 0; t < deg; ++t) wv[t * H] = soft_div(wv[t * H], den);
            }
            __syncwarp();
            if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_wh[ks]));
            float acc[OWN][KMAX][VEC];
            int hbeg[OWN], hdeg[OWN], hcur[OWN];
#pragma unroll
            for (int t = 0; t < OWN; ++t) {
                const int h = wid + t * W;
                hbeg[t] = 0; hdeg[t] = 0; hcur[t] = 1;
                if (h < Hb) { hbeg[t] = meta[8 + 2 * h]; hdeg[t] = meta[8 + 2 * h + 1]; }
            }
            auto init_acc = [&]() {
                agg_mbar_wait_spin(agg_smem_u32(&bar_wh[ks]), (uint32_t)(i / 2) & 1u);
#pragma unroll
                for (int t = 0; t < OWN; ++t) {
                    const int h = wid + t * W;
                    const float* zr = zh + (size_t)(h < Hb ? h : 0) * LDZ + lcol;
                    const float* wr = wh + (size_t)hbeg[t] * H;
#pragma unroll
                    for (int j = 0; j < KMAX; ++j) {
                        float zv[VEC];
#pragma unroll
                        for (int q = 0; q < VEC; ++q) zv[q] = 0.f;
                        float a = 0.f;
                        if (h < Hb && col_ok(j)) {
                            *reinterpret_cast<V*>(zv) = *reinterpret_cast<const V*>(zr + 32 * VEC * j);
                            a = wr[hj[j]];
                        }
#pragma unroll
                        for (int q = 0; q < VEC; ++q) acc[t][j][q] = fmaf(a, zv[q], 0.f);
                    }
                }
            };
            if (n_chunks == 0) init_acc();
            __nv_bfloat16* const out_hi = p.act_hi + (size_t)n0 * LDP + lcol;
            __nv_bfloat16* const out_lo = p.act_lo + (size_t)n0 * LDP + lcol;
            for (int c = 0; c < n_chunks; ++c) {
                const int k0 = c * W, k1 = min(Mb, k0 + W);
                const float* rows = zE;
                int slot = 0;
                if (!L0) {
                    slot = g % slots;
                    agg_mbar_wait_spin(agg_smem_u32(&bar_full[slot]), (uint32_t)(g / slots) & 1u);
                    rows = ring + (size_t)slot * W * LDZ;
                }
                // (a) the edge-node destination of this warp: in-edges (h1 -> e), (h2 -> e), (e -> e)
                const int k = k0 + wid;
                if (k < k1) {
                    const int h1 = prs[2 * k] - n0, h2 = prs[2 * k + 1] - n0;
                    const float* re = L0 ? rows : rows + (size_t)(k - k0) * LDZ;
                    const float* r1 = zh + (size_t)h1 * LDZ;
                    const float* r2 = zh + (size_t)h2 * LDZ;
                    const float a2e = re[HD + H + lh];
                    const float e1 = leaky_le1(r1[HD + lh] + a2e, alpha);
                    const float e2 = leaky_le1(r2[HD + lh] + a2e, alpha);
                    const float e3 = leaky_le1(re[HD + lh] + a2e, alpha);
                    const float m = fmaxf(fmaxf(e1, e2), e3);
                    const float x1 = soft_exp(e1 - m), x2 = soft_exp(e2 - m), x3 = soft_exp(e3 - m);
                    const float den = (0.f + x1 + x2) + x3;
                    const float s1 = soft_div(x1, den), s2 = soft_div(x2, den), s3 = soft_div(x3, den);
                    __nv_bfloat16* oh = out_hi + (size_t)(Hb + k) * LDP;
                    __nv_bfloat16* ol = out_lo + (size_t)(Hb + k) * LDP;
#pragma unroll
                    for (int j = 0; j < KMAX; ++j) {
                        const float w1 = __shfl_sync(0xffffffffu, s1, hj[j]);
                        const float w2 = __shfl_sync(0xffffffffu, s2, hj[j]);
                        const float w3 = __shfl_sync(0xffffffffu, s3, hj[j]);
                        if (col_ok(j)) {
                            float z1[VEC], z2[VEC], ze[VEC], o[VEC];
                            *reinterpret_cast<V*>(z1) = *reinterpret_cast<const V*>(r1 + lcol + 32 * VEC * j);
                            *reinterpret_cast<V*>(z2) = *reinterpret_cast<const V*>(r2 + lcol + 32 * VEC * j);
                            *reinterpret_cast<V*>(ze) = *reinterpret_cast<const V*>(re + lcol + 32 * VEC * j);
#pragma unroll
                            for (int q = 0; q < VEC; ++q) o[q] = leaky_le1(fmaf(w3, ze[q], fmaf(w2, z2[q], fmaf(w1, z1[q], 0.f))), act_slope);
                            store_planes_vec<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j, o);
                        } else if (NVP > NV && pad_ok(j)) {
                            store_planes_zero<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j);
                        }
                    }
                }
                // (b) contributions of the chunk's rows to the owned heads, ascending edge id
                if (c == 0) init_acc();
#pragma unroll
                for (int t = 0; t < OWN; ++t) {
                    while (hcur[t] < hdeg[t]) {
                        const int pos = hbeg[t] + hcur[t];
                        const int kk = lsth[pos] - n0 - Hb;
                        if (kk >= k1) break;
                        const float* re = (L0 ? rows : rows + (size_t)(kk - k0) * LDZ) + lcol;
                        const float* wp = wh + (size_t)pos * H;
#pragma unroll
                        for (int j = 0; j < KMAX; ++j) {
                            if (!col_ok(j)) continue;
                            float ze[VEC];
                            *reinterpret_cast<V*>(ze) = *reinterpret_cast<const V*>(re + 32 * VEC * j);
                            const float a = wp[hj[j]];
#pragma unroll
                            for (int q = 0; q < VEC; ++q) acc[t][j][q] = fmaf(a, ze[q], acc[t][j][q]);
                        }
                        ++hcur[t];
                    }
                }
                if (!L0) {                                      // this warp is done with the slot
                    __syncwarp();
                    if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_empty[slot]));
                    ++g;
                }
            }
#pragma unroll
            for (int t = 0; t < OWN; ++t) {
                const int h = wid + t * W;
                if (h >= Hb) continue;
                __nv_bfloat16* oh = out_hi + (size_t)h * LDP;
                __nv_bfloat16* ol = out_lo + (size_t)h * LDP;
#pragma unroll
                for (int j = 0; j < KMAX; ++j) {
                    if (col_ok(j)) {
                        float o[VEC];
#pragma unroll
                        for (int q = 0; q < VEC; ++q) o[q] = leaky_le1(acc[t][j][q], act_slope);
                        store_planes_vec<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j, o);
                    } else if (NVP > NV && pad_ok(j)) {
                        store_planes_zero<VEC>(oh + 32 * VEC * j, ol + 32 * VEC * j);
                    }
                }
            }
        }
        else if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_wh[ks]));          // an empty frame still uses up one phase of its set's barriers
        __syncwarp();
        if (lane == 0) agg_mbar_arrive(agg_smem_u32(&bar_tab_empty[ks]));       // the set may be overwritten
    }
}

// last layer (heads*dim == 1): one thread per destination node, sigmoid fused (gat2.py:143-145)
__global__ void __launch_bounds__(256) gat_aggregate_scalar_kernel(
    int n_nodes_total, const int* __restrict__ row_ptr, const int* __restrict__ col,
    const float* __restrict__ z, int ldz, float alpha, float* __restrict__ raw_f32, float* __restrict__ scores,
    const float* __restrict__ res, int ld_res)
{
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes_total) return;
    const int beg = row_ptr[v], end = row_ptr[v + 1];
    const float a2v = z[(size_t)v * ldz + 2];
    float m = -INFINITY;
    for (int e = beg; e < end; ++e) m = fmaxf(m, leaky(z[(size_t)col[e] * ldz + 1] + a2v, alpha));
    float den = 0.f;
    for (int e = beg; e < end; ++e) den += expf(leaky(z[(size_t)col[e] * ldz + 1] + a2v, alpha) - m);
    float acc = 0.f;
    for (int e = beg; e < end; ++e) {
        const float* ru = z + (size_t)col[e] * ldz;
        acc = fmaf(expf(leaky(ru[1] + a2v, alpha) - m) / den, ru[0], acc);
    }
    if (res) acc = res[(size_t)v * ld_res] + acc;             // residual (gat2.py:75)
    if (raw_f32) raw_f32[v] = acc;
    if (scores) scores[v] = 1.0f / (1.0f + expf(-acc));
}

// ------------------------------------------------------------------------------------------------
// Large frames (more heads than the frame-resident plan holds: a 10-view x 16-person frame has 160 heads, 11520
// edge-nodes and 19.6 MB of z rows). Work unit = (frame, u), the units of a frame adjacent in the grid:
//   u <  edge_units : kLargeChunk consecutive edge-node destinations. Edge-nodes are ordered by pair block
//                     (group gi < gj) and row-major inside it, so a chunk touches a handful of distinct head rows
//                     (4 + 16 for 16-person views). The CTA marks the heads its destinations reference and stages
//                     those rows in shared memory once; every warp streams the rows of its destinations' third
//                     in-edge (the self loop - the only row that has to come from HBM) through a private
//                     kEdgeRing-deep cp.async ring, and holds the 3-in-edge softmax in registers.
//   u >= edge_units : kLargeHeads head destinations, kAggWarps / kLargeHeads warps each. A head's in-edges are its
//                     self loop and one edge-node per head of every other view (145 rows) - rows the edge units of
//                     the same frame have just pulled through L2. Each warp streams a contiguous part of the in-edges
//                     through a kHeadRing-deep cp.async ring with a running-max softmax (one pass: no separate logit
//                     sweep over 145 rows); the warps' partial (max, denominator, sum) triples are merged in warp
//                     order. Mathematically the reference's edge_softmax + sum; fp32 rounding differs from the
//                     one-warp gather by reassociation and the exp(m_w - M) rescale (~1e-7 relative).
// Every z row is read from HBM once per layer and every output row written once.
// ------------------------------------------------------------------------------------------------
constexpr int kLargeChunk = 64;        // edge-node destinations per edge unit
constexpr int kLargeHeads = 4;         // head destinations per head unit
constexpr int kLargeStageCap = 32;     // staged head rows per edge unit
constexpr int kEdgeRing = 4;           // rows in flight per warp, edge units
constexpr int kHeadRing = 6;           // rows in flight per warp, head units
constexpr int kWarpsPerHead = kAggWarps / kLargeHeads;
constexpr int kRowIters = 5;           // 16-byte copies per lane and row: ldz <= 640
constexpr float kRescaleAt = 30.f;     // head units: the running softmax reference moves when a logit exceeds it by this much
static_assert(kLargeChunk / kAggWarps * 3 <= 32, "edge units: one lane per (destination, in-edge)");
static_assert(kLargeChunk / kAggWarps >= kEdgeRing, "edge ring deeper than a warp's destinations");

template <int N> __device__ __forceinline__ void agg_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void agg_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// one z row (ldz4 16-byte pieces) by the 32 lanes of a warp: constant strides, so the addresses fold into immediates
__device__ __forceinline__ void agg_row_async(uint32_t dst_lane, const float* src_lane, int ldz4, int lane) {
#pragma unroll
    for (int it = 0; it < kRowIters; ++it)
        if (lane + 32 * it < ldz4) agg_cp_async16(dst_lane + 512 * it, src_lane + 128 * it);
}
template <int VEC> __device__ __forceinline__ void lds_vec(uint32_t addr, float (&v)[VEC]) {
    if constexpr (VEC == 4) asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
    else if constexpr (VEC == 2) asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(addr));
    else asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v[0]) : "r"(addr));
}
__device__ __forceinline__ float lds_f32(uint32_t addr) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v; }

struct LargePlan { int stage, slots, idx, ring, part, pm, pd, shared, hidx, total_floats; };
__host__ __device__ inline LargePlan large_plan(int max_heads, int HD, int ldz, int vec) {
    LargePlan f;
    f.ring = 0;                                    // edge: [kAggWarps][kEdgeRing][ldz]; head: [kAggWarps][kHeadRing][ldz]
    const int ring_rows = kAggWarps * (kHeadRing > kEdgeRing ? kHeadRing : kEdgeRing);
    // the head units have no staged rows: their deeper ring overlays the edge units' ring + stage area
    f.stage = kAggWarps * kEdgeRing * ldz;         // [kLargeStageCap + 1][ldz]
    int edge_end = f.stage + (kLargeStageCap + 1) * ldz;
    f.slots = edge_end; edge_end += (max_heads + 1) / 2 + 1;          // short[max_heads]
    f.idx = edge_end; edge_end += 3 * kLargeChunk;                    // int[kLargeChunk][3]
    int head_end = ring_rows * ldz;
    f.part = head_end; head_end += kAggWarps * HD;                    // [kAggWarps][HD]
    f.pm = head_end; head_end += kAggWarps * (HD / vec);              // [kAggWarps][n_vec]
    f.pd = head_end; head_end += kAggWarps * (HD / vec);
    f.shared = head_end; head_end += ldz;                             // layer 0: the row all edge-nodes share
    f.hidx = head_end; head_end += kAggWarps * (max_heads / kWarpsPerHead + 2);   // sources of each warp's in-edges
    f.total_floats = (edge_end > head_end ? edge_end : head_end) + 4;
    return f;
}

// outputs of one destination row held as KMAX vectors per lane; `last` = this lane's last vector exists
template <int VEC, int KMAX>
__device__ __forceinline__ void store_row(const AggParams& p, bool slope_le1, int gv, int lane, bool last, int HD, const float (&acc)[KMAX][VEC])
{
    if (p.raw_f32) {
        float* o = p.raw_f32 + (size_t)gv * HD + lane * VEC;
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
            if (k < KMAX - 1 || last) {
                if constexpr (VEC == 4) *reinterpret_cast<float4*>(o + 128 * k) = make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]);
                else if constexpr (VEC == 2) *reinterpret_cast<float2*>(o + 64 * k) = make_float2(acc[k][0], acc[k][1]);
                else o[32 * k] = acc[k][0];
            }
    }
    if (p.act_hi) {
        __nv_bfloat16* oh = p.act_hi + (size_t)gv * p.ld_planes + lane * VEC;
        __nv_bfloat16* ol = p.act_lo + (size_t)gv * p.ld_planes + lane * VEC;
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
            if (k < KMAX - 1 || last) {
                float a[VEC];
#pragma unroll
                for (int q = 0; q < VEC; ++q) a[q] = slope_le1 ? leaky_le1(acc[k][q], p.act_slope) : leaky(acc[k][q], p.act_slope);
                if constexpr (VEC == 4) {
                    uint32_t h0, l0, h1, l1;
                    split_pack2(a[0], a[1], h0, l0);
                    split_pack2(a[2], a[3], h1, l1);
                    *reinterpret_cast<uint2*>(oh + 128 * k) = make_uint2(h0, h1);
                    *reinterpret_cast<uint2*>(ol + 128 * k) = make_uint2(l0, l1);
                } else if constexpr (VEC == 2) {
                    uint32_t h0, l0;
                    split_pack2(a[0], a[1], h0, l0);
                    *reinterpret_cast<uint32_t*>(oh + 64 * k) = h0;
                    *reinterpret_cast<uint32_t*>(ol + 64 * k) = l0;
                } else {
                    __nv_bfloat16 h, l;
                    split_bf16(a[0], h, l);
                    oh[32 * k] = h; ol[32 * k] = l;
                }
            }
        // K padding of the planes stays zero (HD and ld_planes even unless VEC == 1)
        const int pad = p.ld_planes - HD;
        __nv_bfloat16* zh = p.act_hi + (size_t)gv * p.ld_planes + HD;
        __nv_bfloat16* zl = p.act_lo + (size_t)gv * p.ld_planes + HD;
        if constexpr (VEC == 1) {
            for (int c = lane; c < pad; c += 32) { zh[c] = __float2bfloat16_rn(0.f); zl[c] = __float2bfloat16_rn(0.f); }
        } else {
            for (int c = lane; 2 * c < pad; c += 32) { reinterpret_cast<uint32_t*>(zh)[c] = 0u; reinterpret_cast<uint32_t*>(zl)[c] = 0u; }
        }
    }
}

template <int VEC, int KMAX>
__global__ void __launch_bounds__(kAggWarps * 32, 2) gat_aggregate_large_kernel(AggParams p, int max_heads)
{
    extern __shared__ __align__(16) float smem_l[];
    __shared__ int s_all_staged;
    const int units = p.edge_units + p.head_units;
    const int b = blockIdx.x / units, u = blockIdx.x - b * units;
    const int n0 = p.node_off[b], Nb = p.node_off[b + 1] - n0;
    const int h0 = p.head_off[b], Hb = p.head_off[b + 1] - h0;
    const int H = p.heads, D = p.dim, HD = H * D, ldz = p.ldz, ldz4 = ldz >> 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_vec = HD / VEC;
    const bool last = lane + 32 * (KMAX - 1) < n_vec;          // 32 * (KMAX - 1) < n_vec <= 32 * KMAX (host)
    const bool slope_le1 = p.act_slope >= 0.f && p.act_slope <= 1.f;
    const bool alpha_le1 = p.alpha >= 0.f && p.alpha <= 1.f;
    auto lrelu = [&](float x) { return alpha_le1 ? leaky_le1(x, p.alpha) : leaky(x, p.alpha); };
    if (Hb > max_heads) return;                                // outside the sized plan (caller contract: max_heads covers every frame)
    const LargePlan plan = large_plan(max_heads, HD, ldz, VEC);
    const uint32_t smem_base = agg_smem_u32(smem_l);
    int head_of[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) head_of[k] = min(H - 1, ((lane + 32 * k) * VEC) / D);
    auto grow_of = [&](int l) -> const float* {                // z row of local node l, in global memory
        if (p.layer0) return p.z + (size_t)(l < Hb ? h0 + l : p.n_heads_total) * ldz;
        return p.z + (size_t)(n0 + l) * ldz;
    };

    if (u < p.edge_units) {
        // ---------------- edge-node destinations ----------------
        const int v_begin = Hb + u * kLargeChunk;
        if (v_begin >= Nb) return;
        const int v_end = min(Nb, v_begin + kLargeChunk);
        float* zs = smem_l + plan.stage;
        const uint32_t zs_u32 = smem_base + 4u * plan.stage;
        const uint32_t ring_u32 = smem_base + 4u * (plan.ring + warp * kEdgeRing * ldz);
        short* slot_of = reinterpret_cast<short*>(smem_l + plan.slots);
        int* idx = reinterpret_cast<int*>(smem_l + plan.idx);                 // [kLargeChunk][3] local in-edge sources, -1 = skip
        // in-edges of the chunk: thread t < 3 * kLargeChunk takes in-edge t % 3 of destination t / 3
        int my_l = -1;
        if (tid < 3 * kLargeChunk) {
            const int j = tid / 3, e = tid - 3 * j;
            if (v_begin + j < v_end) {
                const int beg = p.row_ptr[n0 + v_begin + j];
                if (p.row_ptr[n0 + v_begin + j + 1] - beg == 3) my_l = __ldg(p.col + beg + e) - n0;   // build_graph: 3 in-edges per edge-node
            }
        }
        for (int l = tid; l < Hb; l += blockDim.x) slot_of[l] = -1;
        __syncthreads();
        if (tid < 3 * kLargeChunk) {
            idx[tid] = my_l;
            if (my_l >= 0 && my_l < Hb && tid % 3 != 2) slot_of[my_l] = 0;    // heads this chunk references
        }
        __syncthreads();
        // every warp starts the stream of its destinations' third-in-edge rows (warp w takes destinations w, w + 8, ..)
        const int n_mine = v_begin + warp < v_end ? (v_end - v_begin - warp + kAggWarps - 1) / kAggWarps : 0;
        auto fetch = [&](int j) {                                            // row of in-edge 2 of my destination j -> ring slot j % kEdgeRing
            if (j < n_mine && !p.layer0) {
                const int l2 = idx[3 * (warp + kAggWarps * j) + 2];
                if (l2 >= 0) agg_row_async(ring_u32 + 4u * ((j % kEdgeRing) * ldz) + 16u * lane, grow_of(l2) + 4 * lane, ldz4, lane);
            }
            agg_cp_async_commit();
        };
#pragma unroll
        for (int j = 0; j < kEdgeRing; ++j) fetch(j);
        if (warp == 0) {                                                      // staging slots in head order, up to stage_cap
            int base = 0;
            for (int l0 = 0; l0 < Hb; l0 += 32) {
                const int l = l0 + lane;
                const bool need = l < Hb && slot_of[l] == 0;
                const unsigned m = __ballot_sync(0xffffffffu, need);
                const int slot = base + __popc(m & ((1u << lane) - 1u));
                if (l < Hb) slot_of[l] = (need && slot < p.stage_cap) ? (short)slot : (short)-1;
                base += __popc(m);
            }
            if (lane == 0) s_all_staged = base <= p.stage_cap;
        }
        __syncthreads();
        for (int l = warp; l < Hb; l += kAggWarps) {
            const int slot = slot_of[l];
            if (slot >= 0) agg_row_async(zs_u32 + 4u * (slot * ldz) + 16u * lane, grow_of(l) + 4 * lane, ldz4, lane);
        }
        if (p.layer0 && warp == kAggWarps - 1)                                // the row all edge-nodes share in layer 0
            agg_row_async(zs_u32 + 4u * (p.stage_cap * ldz) + 16u * lane, p.z + (size_t)p.n_heads_total * ldz + 4 * lane, ldz4, lane);
        agg_cp_async_commit();
        agg_cp_async_wait<0>();
        __syncthreads();
        const bool all_staged = s_all_staged != 0;
        auto head_row = [&](int l) -> const float* {                          // general path: staged or global
            if (l < Hb) { const int slot = slot_of[l]; return slot >= 0 ? zs + (size_t)slot * ldz : grow_of(l); }
            return p.layer0 ? zs + (size_t)p.stage_cap * ldz : grow_of(l);
        };
        const int i_edge = min(lane / H, 2), h_att = lane - (lane / H) * H;
        const uint32_t col_b = 4u * VEC * lane;                               // byte offset of this lane's first vector in a row
        for (int j = 0; j < n_mine; ++j) {
            // groups committed so far: kEdgeRing + 1 + j; row j is complete once at most kEdgeRing - 1 are pending
            if (j > 0) { agg_cp_async_wait<kEdgeRing - 1>(); __syncwarp(); }
            const int jj = warp + kAggWarps * j;
            const int v = v_begin + jj;
            const int l0 = idx[3 * jj], l1 = idx[3 * jj + 1], l2 = idx[3 * jj + 2];
            if (l0 >= 0) {
                float acc[KMAX][VEC];
                if (all_staged && l0 < Hb && l1 < Hb && (p.layer0 ? l2 >= Hb : l2 == v)) {
                    // the usual case: both heads staged, the third in-edge is the self loop - shared memory only
                    const uint32_t r0 = zs_u32 + 4u * (slot_of[l0] * ldz), r1 = zs_u32 + 4u * (slot_of[l1] * ldz);
                    const uint32_t r2 = p.layer0 ? zs_u32 + 4u * (p.stage_cap * ldz) : ring_u32 + 4u * ((j % kEdgeRing) * ldz);
                    const float a1 = lds_f32((i_edge == 0 ? r0 : (i_edge == 1 ? r1 : r2)) + 4u * (HD + h_att));
                    const float a2 = lds_f32(r2 + 4u * (HD + H + h_att));
                    const float e_l = lrelu(a1 + a2);
                    const float e0 = __shfl_sync(0xffffffffu, e_l, h_att), e1 = __shfl_sync(0xffffffffu, e_l, H + h_att),
                                e2 = __shfl_sync(0xffffffffu, e_l, 2 * H + h_att);
                    const float m = fmaxf(fmaxf(e0, e1), e2);
                    const float x0 = soft_exp(e0 - m), x1 = soft_exp(e1 - m), x2 = soft_exp(e2 - m);
                    const float den = (x0 + x1) + x2;
                    const float wgt = soft_div(i_edge == 0 ? x0 : (i_edge == 1 ? x1 : x2), den);
#pragma unroll
                    for (int k = 0; k < KMAX; ++k) {
                        float a[3];
#pragma unroll
                        for (int e = 0; e < 3; ++e) a[e] = __shfl_sync(0xffffffffu, wgt, e * H + head_of[k]);
                        if (k < KMAX - 1 || last) {
                            float f0[VEC], f1[VEC], f2[VEC];
                            lds_vec<VEC>(r0 + col_b + 128u * VEC * k, f0);
                            lds_vec<VEC>(r1 + col_b + 128u * VEC * k, f1);
                            lds_vec<VEC>(r2 + col_b + 128u * VEC * k, f2);
#pragma unroll
                            for (int q = 0; q < VEC; ++q) {
                                float t = fmaf(a[0], f0[q], 0.f);
                                t = fmaf(a[1], f1[q], t);
                                acc[k][q] = fmaf(a[2], f2[q], t);
                            }
                        }
                    }
                } else {
                    const float* r0 = head_row(l0);
                    const float* r1 = head_row(l1);
                    const float* r2 = p.layer0 ? head_row(l2) : smem_l + plan.ring + (size_t)(warp * kEdgeRing + j % kEdgeRing) * ldz;
                    const float a1 = (i_edge == 0 ? r0 : (i_edge == 1 ? r1 : r2))[HD + h_att];
                    const float a2 = (l2 == v) ? r2[HD + H + h_att] : head_row(v)[HD + H + h_att];    // the destination's own row
                    const float e_l = lrelu(a1 + a2);
                    const float e0 = __shfl_sync(0xffffffffu, e_l, h_att), e1 = __shfl_sync(0xffffffffu, e_l, H + h_att),
                                e2 = __shfl_sync(0xffffffffu, e_l, 2 * H + h_att);
                    const float m = fmaxf(fmaxf(e0, e1), e2);
                    const float x0 = soft_exp(e0 - m), x1 = soft_exp(e1 - m), x2 = soft_exp(e2 - m);
                    const float den = (x0 + x1) + x2;
                    const float wgt = soft_div(i_edge == 0 ? x0 : (i_edge == 1 ? x1 : x2), den);
#pragma unroll
                    for (int k = 0; k < KMAX; ++k) {
                        const int cv = lane + 32 * k;
                        float a[3];
#pragma unroll
                        for (int e = 0; e < 3; ++e) a[e] = __shfl_sync(0xffffffffu, wgt, e * H + head_of[k]);
                        if (k < KMAX - 1 || last) {
                            float f0[VEC], f1[VEC], f2[VEC];
                            load_vec<VEC>(r0 + cv * VEC, f0); load_vec<VEC>(r1 + cv * VEC, f1); load_vec<VEC>(r2 + cv * VEC, f2);
#pragma unroll
                            for (int q = 0; q < VEC; ++q) {
                                float t = fmaf(a[0], f0[q], 0.f);
                                t = fmaf(a[1], f1[q], t);
                                acc[k][q] = fmaf(a[2], f2[q], t);
                            }
                        }
                    }
                }
                store_row<VEC, KMAX>(p, slope_le1, n0 + v, lane, last, HD, acc);
            }
            __syncwarp();                                                     // the slot is free: next row into it
            fetch(j + kEdgeRing);
        }
        agg_cp_async_wait<0>();
        return;
    }

    // ---------------- head destinations ----------------
    const int hh = warp / kWarpsPerHead, part_w = warp - hh * kWarpsPerHead;
    const int v = (u - p.edge_units) * kLargeHeads + hh;
    const uint32_t ring_u32 = smem_base + 4u * (plan.ring + warp * kHeadRing * ldz);
    const uint32_t zsh_u32 = smem_base + 4u * plan.shared;
    float* part = smem_l + plan.part;
    float* pm = smem_l + plan.pm;
    float* pd = smem_l + plan.pd;
    const int hidx_cap = max_heads / kWarpsPerHead + 2;
    int* hidx = reinterpret_cast<int*>(smem_l + plan.hidx) + warp * hidx_cap;
    float m_run[KMAX], d_run[KMAX], acc[KMAX][VEC];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        m_run[k] = 0.f; d_run[k] = 0.f;
#pragma unroll
        for (int q = 0; q < VEC; ++q) acc[k][q] = 0.f;
    }
    if (p.layer0) {       // 145 of a head's 146 in-edges are this one row: one copy per CTA instead of one per in-edge
        for (int c = tid; c < ldz4; c += kAggWarps * 32)
            agg_cp_async16(zsh_u32 + 16u * c, p.z + (size_t)p.n_heads_total * ldz + 4 * c);
        agg_cp_async_commit();
        agg_cp_async_wait<0>();
        __syncthreads();
    }
    int n_rows = 0;
    if (v < Hb) {
        const int gv = n0 + v;
        const int beg = p.row_ptr[gv];
        const int deg = p.row_ptr[gv + 1] - beg;
        const int seg = min((deg + kWarpsPerHead - 1) / kWarpsPerHead, hidx_cap);   // deg <= max_heads (build_graph)
        const int i_beg = part_w * seg, i_end = min(deg, i_beg + seg);
        n_rows = max(0, i_end - i_beg);
        for (int i = lane; i < n_rows; i += 32) hidx[i] = __ldg(p.col + beg + i_beg + i) - n0;
        float a2v[KMAX];
        {
            const float* rowv = grow_of(v);
#pragma unroll
            for (int k = 0; k < KMAX; ++k) a2v[k] = rowv[HD + H + head_of[k]];
        }
        __syncwarp();
        auto fetch = [&](int i) {                                            // in-edge i_beg + i -> ring slot i % kHeadRing
            if (i < n_rows) {
                const int l = hidx[i];
                if (!(p.layer0 && l >= Hb)) agg_row_async(ring_u32 + 4u * ((i % kHeadRing) * ldz) + 16u * lane, grow_of(l) + 4 * lane, ldz4, lane);
            }
            agg_cp_async_commit();
        };
#pragma unroll
        for (int i = 0; i < kHeadRing; ++i) fetch(i);
        const uint32_t col_b = 4u * VEC * lane;
        uint32_t a1_b[KMAX];
#pragma unroll
        for (int k = 0; k < KMAX; ++k) a1_b[k] = 4u * (HD + head_of[k]);
        for (int i = 0; i < n_rows; ++i) {
            agg_cp_async_wait<kHeadRing - 1>();
            __syncwarp();
            const uint32_t r = (p.layer0 && hidx[i] >= Hb) ? zsh_u32 : ring_u32 + 4u * ((i % kHeadRing) * ldz);
            // Softmax weights relative to a per-warp reference logit m_run (the first in-edge's, moved only when a
            // logit exceeds it by kRescaleAt): softmax is shift invariant, the merge below rebases the warps on a
            // common maximum, and exp(x) for x <= 30 is far from fp32 overflow - so the per-row work is one exp and
            // VEC FMAs per vector instead of a rescale of the whole accumulator.
            float e[KMAX];
            bool move = false;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                e[k] = lrelu(lds_f32(r + a1_b[k]) + a2v[k]);                           // gat2.py:78-81
                if (i == 0) m_run[k] = e[k];
                move |= (e[k] - m_run[k] > kRescaleAt);
            }
            if (__any_sync(0xffffffffu, move)) {
#pragma unroll
                for (int k = 0; k < KMAX; ++k) {
                    const float m_new = fmaxf(m_run[k], e[k]);
                    const float sc = soft_exp(m_run[k] - m_new);
                    d_run[k] *= sc;
#pragma unroll
                    for (int q = 0; q < VEC; ++q) acc[k][q] *= sc;
                    m_run[k] = m_new;
                }
            }
#pragma unroll
            for (int k = 0; k < KMAX; ++k)
                if (k < KMAX - 1 || last) {
                    const float w = soft_exp(e[k] - m_run[k]);
                    float f[VEC];
                    lds_vec<VEC>(r + col_b + 128u * VEC * k, f);
                    d_run[k] += w;
#pragma unroll
                    for (int q = 0; q < VEC; ++q) acc[k][q] = fmaf(w, f[q], acc[k][q]);
                }
            __syncwarp();
            fetch(i + kHeadRing);
        }
        agg_cp_async_wait<0>();
    }
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        const int cv = lane + 32 * k;
        if (k < KMAX - 1 || last) {
            pm[warp * n_vec + cv] = n_rows > 0 ? m_run[k] : -INFINITY;
            pd[warp * n_vec + cv] = d_run[k];
#pragma unroll
            for (int q = 0; q < VEC; ++q) part[(size_t)warp * HD + cv * VEC + q] = acc[k][q];
        }
    }
    __syncthreads();
    // merge the partial (reference, denominator, sum) triples of a head's warps in warp order; outputs (gat2.py:66, :141-142)
    for (int t = tid; t < kLargeHeads * HD; t += kAggWarps * 32) {
        const int hq = t / HD, c = t - hq * HD, cv = c / VEC;
        const int vq = (u - p.edge_units) * kLargeHeads + hq;
        if (vq >= Hb) break;
        const int w0 = hq * kWarpsPerHead;
        float M = -INFINITY;
#pragma unroll
        for (int w = 0; w < kWarpsPerHead; ++w) M = fmaxf(M, pm[(w0 + w) * n_vec + cv]);
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int w = 0; w < kWarpsPerHead; ++w) {
            const float sc = soft_exp(pm[(w0 + w) * n_vec + cv] - M);
            num = fmaf(part[(size_t)(w0 + w) * HD + c], sc, num);
            den = fmaf(pd[(w0 + w) * n_vec + cv], sc, den);
        }
        const float val = soft_div(num, den);
        const int gq = n0 + vq;
        if (p.raw_f32) p.raw_f32[(size_t)gq * HD + c] = val;
        if (p.act_hi) {
            __nv_bfloat16 hb, lb;
            split_bf16(leaky(val, p.act_slope), hb, lb);
            p.act_hi[(size_t)gq * p.ld_planes + c] = hb;
            p.act_lo[(size_t)gq * p.ld_planes + c] = lb;
        }
    }
    if (p.act_hi) {
        const int pad = p.ld_planes - HD;
        for (int t = tid; t < kLargeHeads * pad; t += kAggWarps * 32) {
            const int hq = t / pad, c = HD + t - hq * pad;
            const int vq = (u - p.edge_units) * kLargeHeads + hq;
            if (vq >= Hb) break;
            p.act_hi[(size_t)(n0 + vq) * p.ld_planes + c] = __float2bfloat16_rn(0.f);
            p.act_lo[(size_t)(n0 + vq) * p.ld_planes + c] = __float2bfloat16_rn(0.f);
        }
    }
}

}  // namespace b200pose

using namespace b200pose;

static int gat_aggregate_impl(int32_t n_frames, int32_t n_nodes_total, int32_t n_heads_total,
                              const int32_t* head_off, const int32_t* node_off,
                              const int32_t* row_ptr, const int32_t* col,
                              const float* z, int32_t ldz, int32_t heads, int32_t dim, int32_t layer0,
                              int32_t max_heads_per_frame, int32_t max_enodes_per_frame, float alpha, float act_slope,
                              float* raw_f32, uint16_t* act_hi, uint16_t* act_lo, int32_t ld_planes,
                              float* scores, int32_t impl, void* stream, const float* res, int32_t ld_res)
{
    if (res) {
        B2_CHECK_ARG(!layer0, "gat_aggregate_res: the first layer has no residual (gat2.py:118)");
        B2_CHECK_ARG(ld_res >= heads * dim, "gat_aggregate_res: ld_res < heads * dim");
        B2_CHECK_ARG(impl == 0 || impl == 1, "gat_aggregate_res: the residual term is added by the gather kernel (impl 0 or 1)");
        impl = 1;
    }
    B2_CHECK_ARG(head_off && node_off && row_ptr && col && z, "gat_aggregate: null input");
    B2_CHECK_ARG(heads >= 1 && dim >= 1 && ldz >= heads * dim + 2 * heads, "gat_aggregate: ldz too small");
    B2_CHECK_ARG(heads <= 32, "gat_aggregate: more than 32 attention heads");
    B2_CHECK_ARG((act_hi == nullptr) == (act_lo == nullptr), "gat_aggregate: planes go together");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_frames == 0 || n_nodes_total == 0) return B200POSE_OK;
    const int HD = heads * dim;
    if (HD == 1) {
        B2_CHECK_ARG(!layer0 && !act_hi, "gat_aggregate: scalar layer cannot be layer 0 / produce planes");
        gat_aggregate_scalar_kernel<<<ceil_div(n_nodes_total, 256), 256, 0, st>>>(n_nodes_total, row_ptr, col, z, ldz,
                                                                                  alpha, raw_f32, scores, res, ld_res);
        B2_CHECK_LAUNCH();
        return B200POSE_OK;
    }
    B2_CHECK_ARG(scores == nullptr, "gat_aggregate: scores need heads*dim == 1");
    B2_CHECK_ARG(ldz % 4 == 0, "gat_aggregate: ldz must be a multiple of 4");
    if (act_hi) B2_CHECK_ARG(ld_planes % 64 == 0 && ld_planes >= HD, "gat_aggregate: bad ld_planes");
    AggParams p;
    p.n_frames = n_frames; p.n_heads_total = n_heads_total; p.head_off = head_off; p.node_off = node_off;
    p.row_ptr = row_ptr; p.col = col; p.z = z; p.ldz = ldz; p.heads = heads; p.dim = dim; p.layer0 = layer0;
    p.alpha = alpha; p.act_slope = act_slope; p.raw_f32 = raw_f32;
    p.act_hi = reinterpret_cast<__nv_bfloat16*>(act_hi); p.act_lo = reinterpret_cast<__nv_bfloat16*>(act_lo);
    p.ld_planes = ld_planes;
    p.res = res; p.ld_res = ld_res;
    p.stage_cap = 0; p.edge_units = 0; p.head_units = 0;
    const int vec = (dim % 4 == 0) ? 4 : (dim % 2 == 0 ? 2 : 1);
    // A live frame or two (fewer frames than an eighth of the SMs): one CTA per frame would leave the GPU idle and pay one
    // CTA's serial latency (25 us per layer for a Panoptic frame); the large-frame kernel spreads a frame over its edge and
    // head units (8 CTAs for 20 heads / 160 edge-nodes: 10-16 us), so tiny batches take it.
    const bool tiny_batch = impl == 0 && n_frames * 8 <= 148 && 3 * heads <= 32;
    // ---- frame-resident kernels: one CTA per frame, whenever the frame plan fits in shared memory ----
    const bool frame_path = ((impl == 0 && !tiny_batch) || impl == 3 || impl == 5 || impl == 6) && max_heads_per_frame > 0 && max_enodes_per_frame > 0 &&
                            max_heads_per_frame <= kFrameOwn * kFrameWarps && HD / vec <= 32 * 4;
    // shape-specialised kernel (the shipped layer shapes, planes out, LeakyReLU slope in [0, 1]); impl 5 forces the generic one
    if (frame_path && impl != 5 && act_hi && !raw_f32 && act_slope >= 0.f && act_slope <= 1.f && alpha >= 0.f && alpha <= 1.f) {
        auto launch_s = [&](auto kern, const FramePlanS f, int ldz_s, int ldp_s, bool* taken) -> int {
            *taken = false;
            const size_t smem_s = (size_t)f.total_floats * sizeof(float);
            if (ldz != ldz_s || ld_planes != ldp_s || smem_s > 220 * 1024) return B200POSE_OK;
            *taken = true;
            B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s));
            kern<<<n_frames, kFrameThreads, smem_s, st>>>(p, max_heads_per_frame, max_enodes_per_frame);
            B2_CHECK_LAUNCH();
            return B200POSE_OK;
        };
        // persistent form first (one CTA per SM, set-up of frame f+1 beside the arithmetic of frame f); impl 6 forces the
        // one-CTA-per-frame form
        auto launch_p = [&](auto kern, auto plan_fn, int warps, int ldz_s, int ldp_s, bool* taken) -> int {
            *taken = false;
            if (impl == 6 || ldz != ldz_s || ld_planes != ldp_s) return B200POSE_OK;
            int slots = kSlots;
            size_t smem_p = 0;
            for (; slots >= 2; --slots) {
                smem_p = (size_t)plan_fn(max_heads_per_frame, max_enodes_per_frame, slots).total_floats * sizeof(float);
                if (smem_p <= 226 * 1024) break;
            }
            if (slots < 2) return B200POSE_OK;
            *taken = true;
            int dev = 0, sms = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            const int grid = n_frames < sms ? n_frames : sms;
            B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p));
            kern<<<grid, (warps + 2) * 32, smem_p, st>>>(p, max_heads_per_frame, max_enodes_per_frame, slots);
            B2_CHECK_LAUNCH();
            return B200POSE_OK;
        };
        bool taken = false;
        int rc = B200POSE_OK;
        // consumer warps: one per head where the register file allows it (measured on 1024 Panoptic frames, 20 heads each:
        // 16 warps x 2 heads 0.470 ms, 20 x 1 0.422 ms, 24 x 1 0.436 ms per step)
        const bool w20 = max_heads_per_frame <= 20;
        const bool w24 = !w20 && max_heads_per_frame <= 24;
#define B2_TRY_SHAPE_P(HH, DD)                                                                                                      \
        if (!taken && heads == HH && dim == DD) {                                                                                   \
            using S_ = FrameShape<HH, DD>;                                                                                           \
            if (w24) rc = layer0 ? launch_p(gat_aggregate_frame_p_kernel<HH, DD, true, 24, 1>, frame_plan_p<HH, DD, 24>, 24, S_::LDZ, S_::LDP, &taken)  \
                                 : launch_p(gat_aggregate_frame_p_kernel<HH, DD, false, 24, 1>, frame_plan_p<HH, DD, 24>, 24, S_::LDZ, S_::LDP, &taken); \
            else if (w20) rc = layer0 ? launch_p(gat_aggregate_frame_p_kernel<HH, DD, true, 20, 1>, frame_plan_p<HH, DD, 20>, 20, S_::LDZ, S_::LDP, &taken)  \
                                 : launch_p(gat_aggregate_frame_p_kernel<HH, DD, false, 20, 1>, frame_plan_p<HH, DD, 20>, 20, S_::LDZ, S_::LDP, &taken); \
            else rc = layer0 ? launch_p(gat_aggregate_frame_p_kernel<HH, DD, true, 16, 2>, frame_plan_p<HH, DD, 16>, 16, S_::LDZ, S_::LDP, &taken)      \
                             : launch_p(gat_aggregate_frame_p_kernel<HH, DD, false, 16, 2>, frame_plan_p<HH, DD, 16>, 16, S_::LDZ, S_::LDP, &taken);     \
            if (rc != B200POSE_OK) return rc;                                                                                        \
        }
        B2_TRY_SHAPE_P(10, 40)
        B2_TRY_SHAPE_P(8, 40)
        B2_TRY_SHAPE_P(5, 30)
#undef B2_TRY_SHAPE_P
        if (taken) return B200POSE_OK;
#define B2_TRY_SHAPE(HH, DD)                                                                                                        \
        if (!taken && heads == HH && dim == DD) {                                                                                   \
            using S_ = FrameShape<HH, DD>;                                                                                           \
            rc = layer0 ? launch_s(gat_aggregate_frame_s_kernel<HH, DD, true>, frame_plan_s<HH, DD>(max_heads_per_frame, max_enodes_per_frame), S_::LDZ, S_::LDP, &taken) \
                        : launch_s(gat_aggregate_frame_s_kernel<HH, DD, false>, frame_plan_s<HH, DD>(max_heads_per_frame, max_enodes_per_frame), S_::LDZ, S_::LDP, &taken); \
            if (rc != B200POSE_OK) return rc;                                                                                        \
        }
        B2_TRY_SHAPE(10, 40)
        B2_TRY_SHAPE(8, 40)
        B2_TRY_SHAPE(5, 30)
#undef B2_TRY_SHAPE
        if (taken) return B200POSE_OK;
    }
    if (frame_path) {
        const FramePlan f = frame_plan(max_heads_per_frame, max_enodes_per_frame, HD, heads, ldz);
        const size_t smem_frame = (size_t)f.total_floats * sizeof(float);
        if (smem_frame <= 220 * 1024) {
            auto launch_frame = [&](auto kern) -> int {
                B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_frame));
                kern<<<n_frames, kFrameThreads, smem_frame, st>>>(p, max_heads_per_frame, max_enodes_per_frame);
                B2_CHECK_LAUNCH();
                return B200POSE_OK;
            };
            const int n_vec_f = HD / vec;
            if (vec == 4) return n_vec_f <= 64 ? launch_frame(gat_aggregate_frame_kernel<4, 2>) : launch_frame(gat_aggregate_frame_kernel<4, 4>);
            if (vec == 2) return n_vec_f <= 64 ? launch_frame(gat_aggregate_frame_kernel<2, 2>) : launch_frame(gat_aggregate_frame_kernel<2, 4>);
            return launch_frame(gat_aggregate_frame_kernel<1, 4>);
        }
    }
    if (impl == 3 || impl == 5 || impl == 6) {
        set_error("gat_aggregate: impl 3 / 5 / 6 (frame-resident kernels) need frames of at most %d heads whose plan fits in shared memory "
                  "(%d heads, %d edge-nodes per frame here)", kFrameOwn * kFrameWarps, max_heads_per_frame, max_enodes_per_frame);
        return B200POSE_E_UNSUPPORTED;
    }
    B2_CHECK_ARG(impl >= 0 && impl <= 2, "gat_aggregate: impl must be 0 (auto), 1 (gather kernel), 2 (large-frame kernel), 3 (frame-resident kernel, "
                 "frames of at most 32 heads whose plan fits in shared memory) 5 (its generic, not shape-specialised form) or 6 (shape-specialised, one CTA per frame instead of persistent)");
    // ---- gather kernel: work unit = (frame, chunk of destination nodes). ---- In-degree of a head is 1 + H_b - n_g <= H_b and of an
    // edge-node 3; the frame with the most heads also has the most nodes: N_b <= H_b + H_b^2/2.
    const int mh = max_heads_per_frame > 0 ? max_heads_per_frame : 1;
    p.max_deg = mh < 3 ? 3 : mh;
    // ---- large frames (more heads than the frame-resident kernels take: > 32): fused edge-chunk + head units, every z row read
    // from HBM once. Measured on 256 six-camera ARP frames: 48 heads 1.13 ms against 3.66 ms for the gather kernel, 36 heads 0.70 / 2.18 ----
    if (((impl == 0 && (mh > kFrameOwn * kFrameWarps || tiny_batch)) || impl == 2) && max_enodes_per_frame > 0 && 3 * heads <= 32 && HD / vec <= 32 * 4 && ldz <= 128 * kRowIters) {
        p.stage_cap = kLargeStageCap;
        p.edge_units = ceil_div(max_enodes_per_frame, kLargeChunk);
        p.head_units = ceil_div(mh, kLargeHeads);
        const size_t smem_l = (size_t)large_plan(mh, HD, ldz, vec).total_floats * sizeof(float);
        const long long n_cta = (long long)n_frames * (p.edge_units + p.head_units);
        if (smem_l <= 113 * 1024 && n_cta < 2147483647LL) {                  // two CTAs per SM
            auto launch_large = [&](auto kern) -> int {
                B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l));
                B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                kern<<<(unsigned)n_cta, kAggWarps * 32, smem_l, st>>>(p, mh);
                B2_CHECK_LAUNCH();
                return B200POSE_OK;
            };
            const int n_vec_l = HD / vec, kmax = ceil_div(n_vec_l, 32);       // kernels need 32 (KMAX - 1) < n_vec <= 32 KMAX
            if (vec == 4 && kmax == 4) return launch_large(gat_aggregate_large_kernel<4, 4>);
            if (vec == 4 && kmax == 3) return launch_large(gat_aggregate_large_kernel<4, 3>);
            if (vec == 4 && kmax == 2) return launch_large(gat_aggregate_large_kernel<4, 2>);
            if (vec == 2 && kmax == 4) return launch_large(gat_aggregate_large_kernel<2, 4>);
            if (vec == 2 && kmax == 3) return launch_large(gat_aggregate_large_kernel<2, 3>);
            if (vec == 2 && kmax == 2) return launch_large(gat_aggregate_large_kernel<2, 2>);
            if (vec == 1 && kmax == 4) return launch_large(gat_aggregate_large_kernel<1, 4>);
        }
    }
    // shared memory: the frame's head rows (+1 shared edge-node row for layer 0), capped at 96 KB, plus
    // one [max_deg][heads] attention scratch per warp
    const size_t row_bytes = (size_t)ldz * sizeof(float);
    int stage_rows = (int)((96 * 1024) / row_bytes);
    const int want = max_heads_per_frame > 0 ? max_heads_per_frame + (layer0 ? 1 : 0) : 0;
    if (stage_rows > want) stage_rows = want;
    // Staging pays only while a frame's heads fit: every CTA of a frame (one per 48 destinations) re-loads the staged
    // rows, so for a 10-view x 16-person frame (160 heads, 244 CTAs) 55 staged rows would cost 97 KB of L2 reads per CTA
    // for 6 destinations per warp. Large frames gather everything through L2 instead.
    if (want > stage_rows || stage_rows > 48) stage_rows = 0;
    p.stage_rows = stage_rows;
    const size_t smem = (size_t)stage_rows * row_bytes + (size_t)kAggWarps * p.max_deg * heads * sizeof(float);
    if (smem > 200 * 1024) {
        set_error("gat_aggregate: frame too large for the shared-memory plan (%zu bytes, %d heads per frame)", smem, mh);
        return B200POSE_E_UNSUPPORTED;
    }
    int max_nodes = mh + (mh * mh) / 2;
    if (max_enodes_per_frame > 0 && mh + max_enodes_per_frame < max_nodes) max_nodes = mh + max_enodes_per_frame;
    p.chunk = 6 * kAggWarps;                                   // 48 destinations per CTA
    const int n_chunks = ceil_div(max_nodes, p.chunk);
    p.n_chunks = n_chunks;
    const int n_vec = HD / vec;
    B2_CHECK_ARG((long long)n_frames * n_chunks < 2147483647LL, "gat_aggregate: batch too large for one launch");
    dim3 grid((unsigned)(n_frames * n_chunks));
    auto launch = [&](auto kern) -> int {
        B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, kAggWarps * 32, smem, st>>>(p);
        B2_CHECK_LAUNCH();
        return B200POSE_OK;
    };
    if (n_vec > 32 * 8) { set_error("gat_aggregate: heads*dim = %d too large", HD); return B200POSE_E_UNSUPPORTED; }
    if (vec == 4) return n_vec <= 64 ? launch(gat_aggregate_kernel<4, 2>) : n_vec <= 128 ? launch(gat_aggregate_kernel<4, 4>) : launch(gat_aggregate_kernel<4, 8>);
    if (vec == 2) return n_vec <= 64 ? launch(gat_aggregate_kernel<2, 2>) : n_vec <= 128 ? launch(gat_aggregate_kernel<2, 4>) : launch(gat_aggregate_kernel<2, 8>);
    return n_vec <= 128 ? launch(gat_aggregate_kernel<1, 4>) : launch(gat_aggregate_kernel<1, 8>);
}

extern "C" __attribute__((visibility("default"))) int b200pose_gat_aggregate(int32_t n_frames, int32_t n_nodes_total, int32_t n_heads_total,
                                      const int32_t* head_off, const int32_t* node_off,
                                      const int32_t* row_ptr, const int32_t* col,
                                      const float* z, int32_t ldz, int32_t heads, int32_t dim, int32_t layer0,
                                      int32_t max_heads_per_frame, int32_t max_enodes_per_frame, float alpha, float act_slope,
                                      float* raw_f32, uint16_t* act_hi, uint16_t* act_lo, int32_t ld_planes,
                                      float* scores, int32_t impl, void* stream)
{
    return gat_aggregate_impl(n_frames, n_nodes_total, n_heads_total, head_off, node_off, row_ptr, col, z, ldz, heads, dim, layer0,
                              max_heads_per_frame, max_enodes_per_frame, alpha, act_slope, raw_f32, act_hi, act_lo, ld_planes, scores, impl,
                              stream, nullptr, 0);
}

extern "C" __attribute__((visibility("default"))) int b200pose_gat_aggregate_res(int32_t n_frames, int32_t n_nodes_total, int32_t n_heads_total,
                                          const int32_t* head_off, const int32_t* node_off,
                                          const int32_t* row_ptr, const int32_t* col,
                                          const float* z, int32_t ldz, int32_t heads, int32_t dim,
                                          int32_t max_heads_per_frame, int32_t max_enodes_per_frame, float alpha, float act_slope,
                                          const float* res, int32_t ld_res,
                                          float* raw_f32, uint16_t* act_hi, uint16_t* act_lo, int32_t ld_planes,
                                          float* scores, void* stream)
{
    B2_CHECK_ARG(res, "gat_aggregate_res: null residual");
    return gat_aggregate_impl(n_frames, n_nodes_total, n_heads_total, head_off, node_off, row_ptr, col, z, ldz, heads, dim, 0,
                              max_heads_per_frame, max_enodes_per_frame, alpha, act_slope, raw_f32, act_hi, act_lo, ld_planes, scores, 1,
                              stream, res, ld_res);
}
