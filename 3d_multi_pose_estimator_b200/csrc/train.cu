// Backward pass and optimiser step of the skeleton-matching GAT (the reference trains it with torch autograd over
// skeleton_matching/gat2.py:50-88, 137-149 in skeleton_matching/train_skeleton_matching.py:163-184: MSE loss on the edge-node
// scores, Adam). The derivative is written out by hand here; oracle/train_oracle.py is the CPU restatement of the same formulas
// and is pinned against the reference's autograd (tests/golden/make_golden_train_step.py).
//
// Per GAT layer the backward is
//   aggregation (this file):  d out[v,h,:]  ->  d ft2[u,h,:], d a1[u,h], d a2[v,h]      (edge softmax + weighted sum)
//   projections (gemm.cu):    dW2 = G2^T h2, dh2 = G2 W2, dW1 = G1^T x, dx = G1 W1      (the split-bf16 tcgen05 GEMM)
// and everything between them - activation masks, the bf16 plane splits the GEMM consumes (row-major and transposed), column
// sums for the biases and attention vectors - is the small kernels below. Nothing here uses atomics: every sum runs in a
// fixed order, so a step is reproducible run to run.
#include "common.cuh"

namespace b200pose {

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}
__device__ __forceinline__ float warp_max(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, o));
    return x;
}
// derivative of LeakyReLU as autograd applies it: 1 where the input is > 0, the slope elsewhere
__device__ __forceinline__ float dleaky(float x, float slope) { return x > 0.f ? 1.f : slope; }

// ---------------------------------------------------------------------------------------------------------------------
// Aggregation backward, destination side. One warp per (destination v, attention head h), lanes over v's in-edges.
//   e_uv = LeakyReLU(a1[u] + a2[v]),  alpha_uv = softmax_u(e_uv),  out[v] = sum_u alpha_uv ft2[u]        (gat2.py:59-66, 78-88)
//   d alpha_uv = dout[v] . ft2[u];  c_v = sum_u alpha_uv d alpha_uv;  d e_uv = alpha_uv (d alpha_uv - c_v)
//   d a2[v] = sum_u d e_uv * LeakyReLU'(a1[u] + a2[v])
// Writes stats[v, h] = (max_u e_uv, 1 / sum_u exp(e_uv - max), c_v) for the source-side pass and d a2 into dz.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) agg_bwd_dst_kernel(int n_nodes, const int* __restrict__ row_ptr, const int* __restrict__ col,
                                                         const float* __restrict__ z, int ldz, int H, int D, float alpha,
                                                         const float* __restrict__ dout, int ld_dout,
                                                         float* __restrict__ stats, float* __restrict__ dz, int ld_dz)
{
    const int lane = threadIdx.x & 31;
    const long long unit = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (unit >= (long long)n_nodes * H) return;
    const int v = (int)(unit / H), h = (int)(unit % H);
    const int HD = H * D;
    const int beg = row_ptr[v], end = row_ptr[v + 1];
    const float a2v = z[(size_t)v * ldz + HD + H + h];
    const float* dv = dout + (size_t)v * ld_dout + h * D;
    float m = -INFINITY;
    for (int e = beg + lane; e < end; e += 32) m = fmaxf(m, leaky(z[(size_t)col[e] * ldz + HD + h] + a2v, alpha));
    m = warp_max(m);
    float den = 0.f, t = 0.f, A1 = 0.f, A2 = 0.f;
    for (int e = beg + lane; e < end; e += 32) {
        const float* zu = z + (size_t)col[e] * ldz;
        const float s = zu[HD + h] + a2v;
        const float ex = expf(leaky(s, alpha) - m);
        float da = 0.f;
        for (int d = 0; d < D; ++d) da = fmaf(dv[d], zu[h * D + d], da);
        const float dl = dleaky(s, alpha);
        den += ex; t = fmaf(ex, da, t); A1 = fmaf(ex * da, dl, A1); A2 = fmaf(ex, dl, A2);
    }
    den = warp_sum(den); t = warp_sum(t); A1 = warp_sum(A1); A2 = warp_sum(A2);
    if (lane == 0) {
        const float inv = 1.f / den, c = t * inv;
        float* st = stats + ((size_t)v * H + h) * 3;
        st[0] = m; st[1] = inv; st[2] = c;
        dz[(size_t)v * ld_dz + HD + H + h] = (A1 - c * A2) * inv;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Aggregation backward, source side. One warp per (source u, head h), lanes over the head's `dim` columns. The graphs of this
// path are symmetric (graph_generator.py:627-656 adds u->v and v->u for every link, plus self-loops), so the out-edges of u go
// to exactly the nodes of u's CSR row; they are visited in row order.
//   d ft2[u] = sum_v alpha_uv dout[v] + d a1[u] attn_l + d a2[u] attn_r        (a1 = ft2 . attn_l, a2 = ft2 . attn_r, gat2.py:57-58)
//   d a1[u]  = sum_v d e_uv * LeakyReLU'(a1[u] + a2[v])
// dz[u] = [ d ft2 (heads*dim) | d a1 (heads) | d a2 (heads) ].
// ---------------------------------------------------------------------------------------------------------------------
template <int KMAX>
__global__ void __launch_bounds__(256) agg_bwd_src_kernel(int n_nodes, const int* __restrict__ row_ptr, const int* __restrict__ col,
                                                         const float* __restrict__ z, int ldz, int H, int D, float alpha,
                                                         const float* __restrict__ dout, int ld_dout,
                                                         const float* __restrict__ attn_l, const float* __restrict__ attn_r,
                                                         const float* __restrict__ stats, float* __restrict__ dz, int ld_dz)
{
    const int lane = threadIdx.x & 31;
    const long long unit = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (unit >= (long long)n_nodes * H) return;
    const int u = (int)(unit / H), h = (int)(unit % H);
    const int HD = H * D;
    const float* zu = z + (size_t)u * ldz;
    const float a1u = zu[HD + h];
    float f[KMAX], acc[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        const int d = lane + 32 * k;
        f[k] = d < D ? zu[h * D + d] : 0.f;
        acc[k] = 0.f;
    }
    float da1 = 0.f;
    const int beg = row_ptr[u], end = row_ptr[u + 1];
    for (int e = beg; e < end; ++e) {
        const int v = col[e];
        const float s = a1u + z[(size_t)v * ldz + HD + H + h];
        const float* st = stats + ((size_t)v * H + h) * 3;
        const float a = expf(leaky(s, alpha) - st[0]) * st[1];
        const float* dv = dout + (size_t)v * ld_dout + h * D;
        float g[KMAX], part = 0.f;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            const int d = lane + 32 * k;
            g[k] = d < D ? dv[d] : 0.f;
            part = fmaf(g[k], f[k], part);
        }
        const float da = warp_sum(part);
        da1 = fmaf(a * (da - st[2]), dleaky(s, alpha), da1);
#pragma unroll
        for (int k = 0; k < KMAX; ++k) acc[k] = fmaf(a, g[k], acc[k]);
    }
    float* o = dz + (size_t)u * ld_dz;
    const float da2 = o[HD + H + h];                       // written by the destination-side pass
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        const int d = lane + 32 * k;
        if (d < D) o[h * D + d] = acc[k] + da1 * attn_l[h * D + d] + da2 * attn_r[h * D + d];
    }
    if (lane == 0) o[HD + h] = da1;
}

// ---------------------------------------------------------------------------------------------------------------------
// Gradient matrix -> what the next GEMMs consume. x = g[r, c] * (mask ? LeakyReLU'(mask[r, c]) : 1); any of
//   out_f32 [R, ld_out] (may alias g), planes [R, ld_p] (hi/lo bf16, columns [C, ld_p) zero),
//   transposed planes [C, ld_t] (columns [R, round_up(R, 64)) zero): the K-major operands of the dW = G^T X products.
// mask = hi plane of the ACTIVATED tensor (LeakyReLU keeps the sign, and bf16 rounding keeps it too).
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grad_planes_kernel(const float* g, int R, int C, int ldg,
                                                         const __nv_bfloat16* __restrict__ mask_hi, int ld_mask, float slope,
                                                         float* out_f32, int ld_out,
                                                         __nv_bfloat16* __restrict__ p_hi, __nv_bfloat16* __restrict__ p_lo, int ld_p,
                                                         __nv_bfloat16* __restrict__ t_hi, __nv_bfloat16* __restrict__ t_lo, int ld_t)
{
    __shared__ float tile[32][33];
    const int r_pad = min(ld_t, (R + 63) & ~63);         // the K padding the GEMM reads: zero up to the next multiple of 64
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        float x = 0.f;
        if (r < R && c < C) {
            x = g[(size_t)r * ldg + c];
            if (mask_hi) x *= dleaky(__bfloat162float(mask_hi[(size_t)r * ld_mask + c]), slope);
            if (out_f32) out_f32[(size_t)r * ld_out + c] = x;
        }
        tile[i][tx] = x;
        if (p_hi && r < R && c < ld_p) {
            __nv_bfloat16 hi, lo;
            split_bf16(x, hi, lo);
            p_hi[(size_t)r * ld_p + c] = hi; p_lo[(size_t)r * ld_p + c] = lo;
        }
    }
    if (!t_hi) return;
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;               // transposed: row c of the output, column r
        if (c < C && r < r_pad) {
            __nv_bfloat16 hi, lo;
            split_bf16(tile[tx][i], hi, lo);
            t_hi[(size_t)c * ld_t + r] = hi; t_lo[(size_t)c * ld_t + r] = lo;
        }
    }
}

// planes [R, ld] -> transposed planes [C, ld_t], columns [R, round_up(R, 64)) zero (hi and lo are transposed separately: exact)
__global__ void __launch_bounds__(256) transpose_planes_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo,
                                                              int R, int C, int ld,
                                                              __nv_bfloat16* __restrict__ t_hi, __nv_bfloat16* __restrict__ t_lo, int ld_t)
{
    __shared__ __nv_bfloat16 th[32][34], tl[32][34];
    const int r_pad = min(ld_t, (R + 63) & ~63);
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const __nv_bfloat16 zero = __float2bfloat16_rn(0.f);
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        const bool ok = r < R && c < C;
        th[i][tx] = ok ? hi[(size_t)r * ld + c] : zero;
        tl[i][tx] = ok ? lo[(size_t)r * ld + c] : zero;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (c < C && r < r_pad) {
            t_hi[(size_t)c * ld_t + r] = th[tx][i];
            t_lo[(size_t)c * ld_t + r] = tl[tx][i];
        }
    }
}

// out[j] = sum_r x[r, j] * (w ? w[r * ld_w + j / group] : 1): bias gradients (w = null) and the attention-vector gradients
// d attn[h, d] = sum_u d a[u, h] ft2[u, h, d] (group = dim). One CTA per 32 columns, 32 warps striding the rows, partial sums
// merged in warp order.
__global__ void __launch_bounds__(1024) colsum_kernel(const float* __restrict__ x, int R, int C, int ld,
                                                     const float* __restrict__ w, int ld_w, int group, float* __restrict__ out)
{
    __shared__ float part[32][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int j = blockIdx.x * 32 + tx;
    float s = 0.f;
    if (j < C) {
        const int gcol = w ? j / group : 0;
        for (int r = ty; r < R; r += 32) {
            const float v = x[(size_t)r * ld + j];
            s = w ? fmaf(v, w[(size_t)r * ld_w + gcol], s) : s + v;
        }
    }
    part[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && j < C) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) t += part[i][tx];
        out[j] = t;
    }
}

// Every operand plane of one layer from its fp32 parameters, in one launch (after each optimiser step): W1 -> planes and
// transposed planes; [W2 ; attention folds] -> planes (+ the folded bias); W2 -> transposed planes. One CTA per 32x32 tile of
// two stacked index spaces (rows_a rows of W1, then rows_b rows of [W2 ; folds]); the transposed planes go through a
// shared-memory tile so that both layouts are written with coalesced stores. Paddings are written as zeros so the planes can
// be consumed as K padding.
// The folds: a1[n, h] = sum_d ft2[n, h, d] attn_l[h, d] = h2[n, :] . (sum_d attn_l[h, d] W2[hD + d, :]) + ... (gat2.py:55-58),
// so fc2 yields [ft2 | a1 | a2] in one GEMM. fp64 accumulation as the inference path's host-side fold.
__device__ __forceinline__ float fold_row_value(const float* __restrict__ W2, int ld_w, const float* __restrict__ attn_l,
                                                const float* __restrict__ attn_r, int H, int D, int HD, int r, int c)
{
    const int h = (r - HD) % H;
    const float* a = (r - HD) < H ? attn_l : attn_r;
    double v = 0.0;
    for (int d = 0; d < D; ++d) v += (double)a[h * D + d] * (double)W2[(size_t)(h * D + d) * ld_w + c];
    return (float)v;
}

__global__ void __launch_bounds__(256) prepare_layer_kernel(const float* __restrict__ W1, const float* __restrict__ W2, int ld_w,
                                                           const float* __restrict__ b2, const float* __restrict__ attn_l,
                                                           const float* __restrict__ attn_r, int H, int D, int din,
                                                           __nv_bfloat16* __restrict__ w1_hi, __nv_bfloat16* __restrict__ w1_lo, int ld_w1,
                                                           __nv_bfloat16* __restrict__ w1t_hi, __nv_bfloat16* __restrict__ w1t_lo, int ld_w1t,
                                                           __nv_bfloat16* __restrict__ w2_hi, __nv_bfloat16* __restrict__ w2_lo, int ld_w2,
                                                           __nv_bfloat16* __restrict__ w2t_hi, __nv_bfloat16* __restrict__ w2t_lo, int ld_w2t,
                                                           float* __restrict__ b2e, int tiles_a)
{
    __shared__ float tile[32][33];
    const int HD = H * D, n2 = HD + 2 * H;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c0 = blockIdx.x * 32;
    const bool part_a = (int)blockIdx.y < tiles_a;
    const int r0 = (part_a ? (int)blockIdx.y : (int)blockIdx.y - tiles_a) * 32;
    __nv_bfloat16 hi, lo;
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        float x = 0.f;
        if (part_a) {                                          // ---- W1 [din, din]
            if (r < din && c < din) x = W1[(size_t)r * ld_w + c];
            if (r < din && c < ld_w1) { split_bf16(x, hi, lo); w1_hi[(size_t)r * ld_w1 + c] = hi; w1_lo[(size_t)r * ld_w1 + c] = lo; }
        } else {                                               // ---- [W2 ; folds] [n2, din]
            float xe = 0.f;                                    // row r of [W2 ; folds]; x = the same restricted to the W2 rows (for W2^T)
            if (c < din) {
                if (r < HD) xe = x = W2[(size_t)r * ld_w + c];
                else if (r < n2) xe = fold_row_value(W2, ld_w, attn_l, attn_r, H, D, HD, r, c);
            }
            if (r < n2 && c < ld_w2) { split_bf16(xe, hi, lo); w2_hi[(size_t)r * ld_w2 + c] = hi; w2_lo[(size_t)r * ld_w2 + c] = lo; }
            if (c == 0 && r < n2) {
                if (r < HD) b2e[r] = b2[r];
                else {
                    const int h = (r - HD) % H;
                    const float* a = (r - HD) < H ? attn_l : attn_r;
                    double v = 0.0;
                    for (int d = 0; d < D; ++d) v += (double)a[h * D + d] * (double)b2[h * D + d];
                    b2e[r] = (float)v;
                }
            }
        }
        tile[i][tx] = x;
    }
    __syncthreads();
    __nv_bfloat16* t_hi = part_a ? w1t_hi : w2t_hi;
    __nv_bfloat16* t_lo = part_a ? w1t_lo : w2t_lo;
    const int ld_t = part_a ? ld_w1t : ld_w2t;
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;                     // transposed: row c of the output, column r
        if (c < din && r < ld_t) {
            split_bf16(tile[tx][i], hi, lo);
            t_hi[(size_t)c * ld_t + r] = hi; t_lo[(size_t)c * ld_t + r] = lo;
        }
    }
}

// The three column sums behind the aggregation backward in one pass over z and dz: d attn_l[h,d] = sum_u d a1[u,h] ft2[u,h,d],
// d attn_r likewise with d a2, d b2[j] = sum_u d ft2[u,j]. Same summation order as colsum_kernel.
__global__ void __launch_bounds__(1024) attn_bias_grad_kernel(const float* __restrict__ z, int ldz, const float* __restrict__ dz, int ld_dz,
                                                            int R, int H, int D, float* __restrict__ g_attn_l, float* __restrict__ g_attn_r,
                                                            float* __restrict__ g_b2)
{
    __shared__ float part[3][32][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int HD = H * D, j = blockIdx.x * 32 + tx;
    float sl = 0.f, sr = 0.f, sb = 0.f;
    if (j < HD) {
        const int h = j / D;
        for (int r = ty; r < R; r += 32) {
            const float f = z[(size_t)r * ldz + j];
            const float* d = dz + (size_t)r * ld_dz;
            sl = fmaf(f, d[HD + h], sl);
            sr = fmaf(f, d[HD + H + h], sr);
            sb += d[j];
        }
    }
    part[0][ty][tx] = sl; part[1][ty][tx] = sr; part[2][ty][tx] = sb;
    __syncthreads();
    if (ty < 3 && j < HD) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) t += part[ty][i][tx];
        (ty == 0 ? g_attn_l : ty == 1 ? g_attn_r : g_b2)[j] = t;
    }
}

// Residual connections in the backward (gat2.py:70-75: ret = resval + ret): dx[r, c] += sum_h src[r, h * cols + c]. heads = 1 adds
// the gradient that came back through res_fc; heads = H folds the identity branch, where the layer input was broadcast over the
// attention heads (resval = h.unsqueeze(1)), i.e. sums the output gradient over them.
__global__ void __launch_bounds__(256) residual_bwd_add_kernel(float* __restrict__ dx, int ld_dx, const float* __restrict__ src, int ld_src,
                                                              int rows, int cols, int heads)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * cols) return;
    const int r = (int)(i / cols), c = (int)(i % cols);
    float s = 0.f;
    for (int h = 0; h < heads; ++h) s += src[(size_t)r * ld_src + h * cols + c];
    dx[(size_t)r * ld_dx + c] += s;
}

// nn.MSELoss over the edge-node scores (train_skeleton_matching.py:37, 174-178) and its gradient through the final sigmoid
// (gat2.py:145): dlogit[idx[i]] = 2/M (s - y) s (1 - s). dlogit must be zeroed by the caller; idx entries are distinct
// (edge-node ids). One CTA; the loss is summed in fp64 in a fixed order.
__global__ void __launch_bounds__(1024) mse_sigmoid_kernel(const float* __restrict__ scores, const int* __restrict__ idx,
                                                          const float* __restrict__ labels, int M, float* __restrict__ loss,
                                                          float* __restrict__ dlogit)
{
    __shared__ double part[1024];
    double s = 0.0;
    for (int i = threadIdx.x; i < M; i += 1024) {
        const float p = scores[idx[i]];
        const float d = p - labels[i];
        s += (double)d * (double)d;
        if (dlogit) dlogit[idx[i]] = (2.f / (float)M) * d * p * (1.f - p);
    }
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0 && loss) *loss = (float)(part[0] / (double)M);
}

__global__ void __launch_bounds__(256) sigmoid_bwd_kernel(const float* __restrict__ scores, const float* __restrict__ dscores, int n,
                                                         float* __restrict__ dlogit)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const float p = scores[i]; dlogit[i] = dscores[i] * p * (1.f - p); }
}

// Adam with the step count on the device (so a whole optimisation step can be replayed as a CUDA graph): one thread advances
// the counter and writes step_size = lr / (1 - b1^t) and sqrt(1 - b2^t) for the element kernel that follows
__global__ void adam_scalars_kernel(int* __restrict__ step, float lr, float b1, float b2, float* __restrict__ scal)
{
    const int t = *step + 1;
    *step = t;
    scal[0] = (float)((double)lr / (1.0 - pow((double)b1, (double)t)));
    scal[1] = (float)sqrt(1.0 - pow((double)b2, (double)t));
}

// one element of the device-step Adam; shared by adam_dev_kernel and mlp_adam_planes_kernel so both round identically.
// torch.optim.Adam, single-tensor form (amsgrad off): exp_avg.lerp_(g, 1 - b1); exp_avg_sq = b2 v + (1 - b2) g g;
// denom = sqrt(v) / sqrt(1 - b2^t) + eps; theta -= lr / (1 - b1^t) * m / denom
__device__ __forceinline__ float adam_dev_element(float* __restrict__ theta, const float* __restrict__ grad, float* __restrict__ m,
                                                  float* __restrict__ v, size_t i, float b1, float b2, float eps, float wd,
                                                  float step_size, float bc2_sqrt)
{
    float g = grad[i];
    const float th = theta[i];
    if (wd != 0.f) g = fmaf(wd, th, g);
    float mi = m[i], vi = v[i];
    mi = mi + (g - mi) * (1.f - b1);
    vi = vi * b2 + (1.f - b2) * g * g;
    m[i] = mi; v[i] = vi;
    const float out = th - step_size * (mi / (sqrtf(vi) / bc2_sqrt + eps));
    theta[i] = out;
    return out;
}

__global__ void __launch_bounds__(256) adam_dev_kernel(float* __restrict__ theta, const float* __restrict__ grad, float* __restrict__ m,
                                                      float* __restrict__ v, long long n, float b1, float b2, float eps, float wd,
                                                      const float* __restrict__ scal)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    adam_dev_element(theta, grad, m, v, (size_t)i, b1, b2, eps, wd, scal[0], scal[1]);
}

// Adam over a flat parameter buffer of stacked linear layers + the split-bf16 operand planes of every updated weight, in one
// launch: per layer, the weight slot [n, ld] is walked in 32x32 tiles that update the parameters and write W planes [n, ld_w]
// and (optional) W^T planes [k, ld_wt] - the transposed tile goes through shared memory so both stores are coalesced - and the
// floats between this weight slot and the next (the bias) are updated element by element. grad == null: only the planes are
// rebuilt from theta. Plane paddings are written as zeros (the next GEMM reads them as K padding).
constexpr int kAdamPlanesMaxLayers = 16;
constexpr int kAdamTailPerBlock = 1024;
struct AdamPlanesLayer {
    long long off, tail_end;                    // weight slot at off, then floats [off + n * ld, tail_end) (the bias)
    int n, k, ld, ld_w, ld_wt, tiles_x, tiles;
    __nv_bfloat16 *w_hi, *w_lo, *wt_hi, *wt_lo;
};
struct AdamPlanesArgs {
    AdamPlanesLayer l[kAdamPlanesMaxLayers];
    int blk_begin[kAdamPlanesMaxLayers + 1];
    int n_layers;
};

__global__ void __launch_bounds__(256) mlp_adam_planes_kernel(const __grid_constant__ AdamPlanesArgs a, float* __restrict__ theta,
                                                             const float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v,
                                                             float b1, float b2, float eps, float wd, const float* __restrict__ scal)
{
    __shared__ float tile[32][33];
    int li = 0;
    while (li + 1 < a.n_layers && (int)blockIdx.x >= a.blk_begin[li + 1]) ++li;
    const AdamPlanesLayer& L = a.l[li];
    const int local = (int)blockIdx.x - a.blk_begin[li];
    const float step_size = grad ? scal[0] : 0.f, bc2_sqrt = grad ? scal[1] : 1.f;
    if (local >= L.tiles) {                                    // ---- the floats after the weight slot (bias), element-wise
        if (!grad) return;
        const long long base = L.off + (long long)L.n * L.ld + (long long)(local - L.tiles) * kAdamTailPerBlock;
        for (int t = threadIdx.x; t < kAdamTailPerBlock; t += blockDim.x)
            if (base + t < L.tail_end) adam_dev_element(theta, grad, m, v, (size_t)(base + t), b1, b2, eps, wd, step_size, bc2_sqrt);
        return;
    }
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c0 = (local % L.tiles_x) * 32, r0 = (local / L.tiles_x) * 32;
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        float x = 0.f;
        if (r < L.n && c < L.ld) {
            const size_t e = (size_t)L.off + (size_t)r * L.ld + c;
            const float th = grad ? adam_dev_element(theta, grad, m, v, e, b1, b2, eps, wd, step_size, bc2_sqrt) : theta[e];
            if (c < L.k) x = th;
        }
        if (r < L.n && c < L.ld_w) {
            __nv_bfloat16 hi, lo;
            split_bf16(x, hi, lo);
            L.w_hi[(size_t)r * L.ld_w + c] = hi; L.w_lo[(size_t)r * L.ld_w + c] = lo;
        }
        tile[i][tx] = x;
    }
    if (!L.wt_hi) return;
    __syncthreads();
    const int r_pad = min(L.ld_wt, (L.n + 63) & ~63);
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;                     // transposed: row c of W^T, column r
        if (c < L.k && r < r_pad) {
            __nv_bfloat16 hi, lo;
            split_bf16(tile[tx][i], hi, lo);
            L.wt_hi[(size_t)c * L.ld_wt + r] = hi; L.wt_lo[(size_t)c * L.ld_wt + r] = lo;
        }
    }
}

}  // namespace b200pose

using namespace b200pose;

#define B2_EXPORT extern "C" __attribute__((visibility("default")))

B2_EXPORT int b200pose_gat_aggregate_bwd(int32_t n_nodes, const int32_t* row_ptr, const int32_t* col,
                                         const float* z, int32_t ldz, int32_t heads, int32_t dim, float alpha,
                                         const float* dout, int32_t ld_dout, const float* attn_l, const float* attn_r,
                                         float* stats, float* dz, int32_t ld_dz, void* stream)
{
    B2_CHECK_ARG(row_ptr && col && z && dout && attn_l && attn_r && stats && dz, "gat_aggregate_bwd: null argument");
    B2_CHECK_ARG(heads >= 1 && dim >= 1 && dim <= 128, "gat_aggregate_bwd: heads >= 1 and 1 <= dim <= 128");
    B2_CHECK_ARG(ldz >= heads * dim + 2 * heads && ld_dz >= heads * dim + 2 * heads && ld_dout >= heads * dim, "gat_aggregate_bwd: leading dimension too small");
    if (n_nodes <= 0) return B200POSE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const long long warps = (long long)n_nodes * heads;
    const int blocks = (int)((warps + 7) / 8);
    agg_bwd_dst_kernel<<<blocks, 256, 0, st>>>(n_nodes, row_ptr, col, z, ldz, heads, dim, alpha, dout, ld_dout, stats, dz, ld_dz);
    B2_CHECK_LAUNCH();
    if (dim <= 32) agg_bwd_src_kernel<1><<<blocks, 256, 0, st>>>(n_nodes, row_ptr, col, z, ldz, heads, dim, alpha, dout, ld_dout, attn_l, attn_r, stats, dz, ld_dz);
    else if (dim <= 64) agg_bwd_src_kernel<2><<<blocks, 256, 0, st>>>(n_nodes, row_ptr, col, z, ldz, heads, dim, alpha, dout, ld_dout, attn_l, attn_r, stats, dz, ld_dz);
    else agg_bwd_src_kernel<4><<<blocks, 256, 0, st>>>(n_nodes, row_ptr, col, z, ldz, heads, dim, alpha, dout, ld_dout, attn_l, attn_r, stats, dz, ld_dz);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_grad_planes(const float* g, int32_t rows, int32_t cols, int32_t ld_g,
                                   const uint16_t* mask_hi, int32_t ld_mask, float slope,
                                   float* out_f32, int32_t ld_out,
                                   uint16_t* p_hi, uint16_t* p_lo, int32_t ld_p,
                                   uint16_t* t_hi, uint16_t* t_lo, int32_t ld_t, void* stream)
{
    B2_CHECK_ARG(g && rows >= 0 && cols >= 1 && ld_g >= cols, "grad_planes: bad input");
    B2_CHECK_ARG((p_hi == nullptr) == (p_lo == nullptr) && (t_hi == nullptr) == (t_lo == nullptr), "grad_planes: planes go together");
    B2_CHECK_ARG(out_f32 || p_hi || t_hi, "grad_planes: no output requested");
    if (mask_hi) B2_CHECK_ARG(ld_mask >= cols, "grad_planes: ld_mask < cols");
    if (out_f32) B2_CHECK_ARG(ld_out >= cols, "grad_planes: ld_out < cols");
    if (p_hi) B2_CHECK_ARG(ld_p >= cols, "grad_planes: ld_p < cols");
    if (t_hi) B2_CHECK_ARG(ld_t >= rows, "grad_planes: ld_t < rows");
    if (rows == 0 && !t_hi) return B200POSE_OK;
    const int r_pad = ((rows + 63) / 64) * 64 < ld_t ? ((rows + 63) / 64) * 64 : ld_t;
    const int gx = ceil_div(p_hi ? ld_p : cols, 32), gy = ceil_div(t_hi ? (r_pad > rows ? r_pad : rows) : rows, 32);
    if (gx == 0 || gy == 0) return B200POSE_OK;
    grad_planes_kernel<<<dim3(gx, gy), 256, 0, (cudaStream_t)stream>>>(g, rows, cols, ld_g, reinterpret_cast<const __nv_bfloat16*>(mask_hi), ld_mask, slope,
        out_f32, ld_out, reinterpret_cast<__nv_bfloat16*>(p_hi), reinterpret_cast<__nv_bfloat16*>(p_lo), ld_p,
        reinterpret_cast<__nv_bfloat16*>(t_hi), reinterpret_cast<__nv_bfloat16*>(t_lo), ld_t);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_transpose_planes(const uint16_t* hi, const uint16_t* lo, int32_t rows, int32_t cols, int32_t ld,
                                        uint16_t* t_hi, uint16_t* t_lo, int32_t ld_t, void* stream)
{
    B2_CHECK_ARG(hi && lo && t_hi && t_lo && rows >= 0 && cols >= 1 && ld >= cols && ld_t >= rows, "transpose_planes: bad argument");
    const int r_pad = ((rows + 63) / 64) * 64 < ld_t ? ((rows + 63) / 64) * 64 : ld_t;
    const int gx = ceil_div(cols, 32), gy = ceil_div(r_pad, 32);
    if (gy == 0) return B200POSE_OK;
    transpose_planes_kernel<<<dim3(gx, gy), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(hi), reinterpret_cast<const __nv_bfloat16*>(lo),
        rows, cols, ld, reinterpret_cast<__nv_bfloat16*>(t_hi), reinterpret_cast<__nv_bfloat16*>(t_lo), ld_t);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_colsum(const float* x, int32_t rows, int32_t cols, int32_t ld, const float* w, int32_t ld_w, int32_t group,
                              float* out, void* stream)
{
    B2_CHECK_ARG(x && out && rows >= 0 && cols >= 1 && ld >= cols, "colsum: bad argument");
    if (w) B2_CHECK_ARG(group >= 1 && ld_w >= ceil_div(cols, group), "colsum: bad weight layout");
    colsum_kernel<<<ceil_div(cols, 32), 1024, 0, (cudaStream_t)stream>>>(x, rows, cols, ld, w, ld_w, group, out);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_mse_sigmoid(const float* scores, int32_t n_nodes, const int32_t* idx, const float* labels, int32_t m,
                                   float* loss, float* dlogit, void* stream)
{
    B2_CHECK_ARG(scores && idx && labels && m >= 1 && n_nodes >= 1, "mse_sigmoid: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (dlogit) B2_CHECK_CUDA(cudaMemsetAsync(dlogit, 0, sizeof(float) * (size_t)n_nodes, st));
    mse_sigmoid_kernel<<<1, 1024, 0, st>>>(scores, idx, labels, m, loss, dlogit);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_sigmoid_bwd(const float* scores, const float* dscores, int32_t n, float* dlogit, void* stream)
{
    B2_CHECK_ARG(scores && dscores && dlogit && n >= 0, "sigmoid_bwd: bad argument");
    if (n == 0) return B200POSE_OK;
    sigmoid_bwd_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(scores, dscores, n, dlogit);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_adam_step_dev(float* theta, const float* grad, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                                     float eps, float weight_decay, int32_t* step_dev, float* scalars_dev, void* stream)
{
    B2_CHECK_ARG(theta && grad && m && v && n >= 0 && step_dev && scalars_dev, "adam_step_dev: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    adam_scalars_kernel<<<1, 1, 0, st>>>(step_dev, lr, beta1, beta2, scalars_dev);
    B2_CHECK_LAUNCH();
    if (n == 0) return B200POSE_OK;
    adam_dev_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(theta, grad, m, v, (long long)n, beta1, beta2, eps, weight_decay, scalars_dev);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_mlp_adam_planes(float* theta, const float* grad, float* m, float* v, int64_t n_total,
                                       const b200pose_mlp_layer* layers, int32_t n_layers, float lr, float beta1, float beta2,
                                       float eps, float weight_decay, int32_t* step_dev, float* scalars_dev, void* stream)
{
    B2_CHECK_ARG(theta && layers && n_layers >= 1 && n_layers <= kAdamPlanesMaxLayers && n_total >= 0,
                 "mlp_adam_planes: bad argument (1 <= n_layers <= %d)", kAdamPlanesMaxLayers);
    if (grad) B2_CHECK_ARG(m && v && step_dev && scalars_dev, "mlp_adam_planes: an optimiser step needs m, v, step_dev and scalars_dev");
    AdamPlanesArgs a;
    a.n_layers = n_layers;
    a.blk_begin[0] = 0;
    long long blocks = 0;
    for (int i = 0; i < n_layers; ++i) {
        const b200pose_mlp_layer& s = layers[i];
        B2_CHECK_ARG(s.w_hi && s.w_lo && (s.wt_hi == nullptr) == (s.wt_lo == nullptr), "mlp_adam_planes: layer %d: null W planes", i);
        B2_CHECK_ARG(s.n >= 1 && s.k >= 1 && s.ld >= s.k && s.ld_w % 64 == 0 && s.ld_w >= s.ld,
                     "mlp_adam_planes: layer %d: need n, k >= 1, ld >= k, ld_w a multiple of 64 >= ld", i);
        if (s.wt_hi) B2_CHECK_ARG(s.ld_wt % 64 == 0 && s.ld_wt >= s.n, "mlp_adam_planes: layer %d: ld_wt must be a multiple of 64 >= n", i);
        const long long end = s.offset + (long long)s.n * s.ld;
        const long long next = i + 1 < n_layers ? layers[i + 1].offset : n_total;
        B2_CHECK_ARG((i > 0 || s.offset == 0) && s.offset >= 0 && end <= next && next <= n_total,
                     "mlp_adam_planes: layer %d: weight slots must be in increasing order inside [0, n_total), the first at 0", i);
        AdamPlanesLayer& d = a.l[i];
        d.off = s.offset; d.tail_end = next;
        d.n = s.n; d.k = s.k; d.ld = s.ld; d.ld_w = s.ld_w; d.ld_wt = s.wt_hi ? s.ld_wt : 0;
        const int rows = s.wt_hi ? ((s.n + 63) / 64) * 64 : s.n;
        d.tiles_x = ceil_div(s.ld_w, 32);
        d.tiles = d.tiles_x * ceil_div(rows, 32);
        d.w_hi = reinterpret_cast<__nv_bfloat16*>(s.w_hi); d.w_lo = reinterpret_cast<__nv_bfloat16*>(s.w_lo);
        d.wt_hi = reinterpret_cast<__nv_bfloat16*>(s.wt_hi); d.wt_lo = reinterpret_cast<__nv_bfloat16*>(s.wt_lo);
        blocks += d.tiles + (grad ? (next - end + kAdamTailPerBlock - 1) / kAdamTailPerBlock : 0);
        B2_CHECK_ARG(blocks < (1LL << 31), "mlp_adam_planes: too many tiles");
        a.blk_begin[i + 1] = (int)blocks;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (grad) {
        adam_scalars_kernel<<<1, 1, 0, st>>>(step_dev, lr, beta1, beta2, scalars_dev);
        B2_CHECK_LAUNCH();
    }
    mlp_adam_planes_kernel<<<(int)blocks, 256, 0, st>>>(a, theta, grad, m, v, beta1, beta2, eps, weight_decay, scalars_dev);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_gat_prepare_layer(const float* w1, const float* w2, int32_t ld_w, const float* b2, const float* attn_l,
                                         const float* attn_r, int32_t heads, int32_t dim, int32_t din,
                                         uint16_t* w1_hi, uint16_t* w1_lo, int32_t ld_w1, uint16_t* w1t_hi, uint16_t* w1t_lo, int32_t ld_w1t,
                                         uint16_t* w2_hi, uint16_t* w2_lo, int32_t ld_w2, uint16_t* w2t_hi, uint16_t* w2t_lo, int32_t ld_w2t,
                                         float* b2e, void* stream)
{
    B2_CHECK_ARG(w1 && w2 && b2 && attn_l && attn_r && w1_hi && w1_lo && w1t_hi && w1t_lo && w2_hi && w2_lo && w2t_hi && w2t_lo && b2e,
                 "gat_prepare_layer: null argument");
    const int hd = heads * dim, n2 = hd + 2 * heads, kp = ((din + 63) / 64) * 64, hp = ((hd + 63) / 64) * 64;
    B2_CHECK_ARG(heads >= 1 && dim >= 1 && din >= 1 && ld_w >= din, "gat_prepare_layer: bad shape");
    B2_CHECK_ARG(ld_w1 == kp && ld_w2 == kp && ld_w1t >= kp && ld_w2t >= hp, "gat_prepare_layer: plane leading dimensions must be round_up(din, 64) "
                 "(W1, [W2; folds]), >= round_up(din, 64) (W1^T) and >= round_up(heads*dim, 64) (W2^T)");
    const int rows_a = ld_w1t > kp ? ld_w1t : kp;             // din rows of W1 + the K padding of W1^T
    const int rows_b = (n2 > ld_w2t ? n2 : ld_w2t);           // rows of [W2 ; folds], and the K padding of W2^T
    const int tiles_a = ceil_div(rows_a, 32), tiles_b = ceil_div(rows_b, 32);
    (void)hp;
    prepare_layer_kernel<<<dim3(kp / 32, tiles_a + tiles_b), 256, 0, (cudaStream_t)stream>>>(w1, w2, ld_w, b2, attn_l, attn_r, heads, dim, din,
        reinterpret_cast<__nv_bfloat16*>(w1_hi), reinterpret_cast<__nv_bfloat16*>(w1_lo), ld_w1,
        reinterpret_cast<__nv_bfloat16*>(w1t_hi), reinterpret_cast<__nv_bfloat16*>(w1t_lo), ld_w1t,
        reinterpret_cast<__nv_bfloat16*>(w2_hi), reinterpret_cast<__nv_bfloat16*>(w2_lo), ld_w2,
        reinterpret_cast<__nv_bfloat16*>(w2t_hi), reinterpret_cast<__nv_bfloat16*>(w2t_lo), ld_w2t, b2e, tiles_a);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_gat_attn_bias_grad(const float* z, int32_t ldz, const float* dz, int32_t ld_dz, int32_t rows, int32_t heads, int32_t dim,
                                          float* g_attn_l, float* g_attn_r, float* g_b2, void* stream)
{
    B2_CHECK_ARG(z && dz && g_attn_l && g_attn_r && g_b2 && rows >= 0 && heads >= 1 && dim >= 1, "gat_attn_bias_grad: bad argument");
    B2_CHECK_ARG(ldz >= heads * dim && ld_dz >= heads * dim + 2 * heads, "gat_attn_bias_grad: leading dimension too small");
    attn_bias_grad_kernel<<<ceil_div(heads * dim, 32), 1024, 0, (cudaStream_t)stream>>>(z, ldz, dz, ld_dz, rows, heads, dim, g_attn_l, g_attn_r, g_b2);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

B2_EXPORT int b200pose_residual_bwd_add(float* dx, int32_t ld_dx, const float* src, int32_t ld_src, int32_t rows, int32_t cols, int32_t heads,
                                        void* stream)
{
    B2_CHECK_ARG(dx && src && rows >= 0 && cols >= 1 && heads >= 1 && ld_dx >= cols && ld_src >= heads * cols, "residual_bwd_add: bad argument");
    if (rows == 0) return B200POSE_OK;
    const long long total = (long long)rows * cols;
    residual_bwd_add_kernel<<<(int)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dx, ld_dx, src, ld_src, rows, cols, heads);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}
