// Dense projections out = act(A * W^T + bias) on the 5th-generation tensor cores (tcgen05 + TMEM),
// operands staged by TMA, 3-term split-bf16 (hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM).
//
// Replaces the nn.Linear calls of the reference's GAT (skeleton_matching/gat2.py:53,55, with the
// attention dots of :57-58 folded in as extra output columns) and pose MLP (utils/mlp.py:8-28).
// Plain bf16 or TF32 inputs miss the 1e-4 score / 0.5 mm joint tolerances (SURVEY.md 7-1), so every
// fp32 operand is carried as two bf16 planes and each k-block issues three UMMA groups.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>

namespace b200pose {

constexpr int kBM = 128;          // UMMA M (cta_group::1)
constexpr int kBK = 64;           // one 128-byte swizzle atom of bf16 along K
constexpr int kUmmaK = 16;
constexpr int kGemmThreads = 192;
constexpr int kMaxStages = 8;

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        if (clock64() - t0 > 4000000000LL) __trap();      // ~2 s: turn a pipeline bug into an error, not a hang
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int x, int y, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(bar) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {   // arrives on the mbarrier when all prior MMAs are done
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128B-swizzled shared-memory matrix descriptor (sm_100 "version 1"):
//   start address >> 4 | LBO (unused for swizzled K-major, 1) | SBO = 1024 B (8 rows x 128 B) | SWIZZLE_128B
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

__device__ __forceinline__ uint32_t tmem_cols_for(int bn) {
    uint32_t c = 32;
    while ((int)c < bn) c <<= 1;
    return c;
}

// ------------------------------------------------------------------------------------------------
// product kernel v2: persistent, double-buffered TMEM accumulators, TMA-store epilogue
//
//   grid = min(#tiles, #SMs); every CTA walks tiles t = blockIdx.x, += gridDim.x (n fastest, so the CTAs
//   of one wave share A tiles through L2). The three roles run decoupled across tiles:
//     warp 0 : TMA producer - keeps `stages` k-blocks in flight, runs ahead into the next tile while
//              the epilogue of the previous one drains
//     warp 1 : MMA issuer   - accumulator (tile & 1) of two TMEM buffers
//     warps 2..5 : epilogue - TMEM -> registers -> (bias, LeakyReLU, scale, re-split) -> 128B-swizzled
//              shared staging -> cp.async.bulk.tensor store; frees the accumulator as soon as its last
//              TMEM load retired
//   Output tiles are made of 64-column panels (bf16 planes: one 128-byte row per panel; fp32: two 32-column
//   boxes), W is fetched in 64-row boxes, so a tile can be 64..256 columns wide at run time.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

struct GemmParams2 {
    int M, N, num_kb;
    int k_last;                              // 16-wide k steps of the last k-block that hold data (the rest is K padding: zeros)
    int tiles_m, tiles_n, panels_total;      // 64-column output panels; tiles_m counts (128 * NCTA)-row tiles
    int group_n;                             // consecutive n-tiles of one m-tile a CTA (pair) processes per visit
    int stages, stage_bn;                    // pipeline depth, widest tile (smem / TMEM sizing)
    const float* bias; float slope, out_scale;
    int has_f32, has_planes;
    const int* m_dev;                        // when set: the number of valid rows lives on the device (M is then the capacity the maps were made for)
    // fused second projection (b200pose_linear_fused2): out2[row, t] = sum_c act(out1)[row, c] * fuse_w[t, c] + fuse_b[t], t < fuse_n <= 4,
    // evaluated in the epilogue registers of a single n-tile; nothing of out1 is stored
    const float* fuse_w; const float* fuse_b; float* fuse_out; int fuse_n, fuse_ldw, fuse_ldo;
};

struct TileInfo { int m0, n0, bn, n_eff; };   // n_eff: the tile's valid width rounded up to the MMA granule (16) - what is actually multiplied
// Tile walk of one CTA (or CTA pair). Work is dealt out in "visits": visit s covers group_n consecutive
// n-tiles of one m-tile, and worker c takes visits c, c + workers, ... With group_n == tiles_n (tall GEMMs:
// many m-tiles) a worker sweeps every n-tile of an m-tile back to back, so the A tile is fetched from HBM once
// and re-read from L2 microseconds later; with group_n == 1 (wide GEMMs: few m-tiles) the walk is the plain
// n-fastest order.
template <int NCTA>
struct TileWalk {
    int visit, j, groups_per_m, total_visits;
    __device__ __forceinline__ TileWalk(const GemmParams2& p, int tiles_m) {
        groups_per_m = (p.tiles_n + p.group_n - 1) / p.group_n;
        total_visits = tiles_m * groups_per_m;
        visit = blockIdx.x / NCTA; j = 0;
    }
    __device__ __forceinline__ bool valid() const { return visit < total_visits; }
    __device__ __forceinline__ int tile(const GemmParams2& p) const {
        const int mb = visit / groups_per_m, g = visit - mb * groups_per_m;
        return mb * p.tiles_n + g * p.group_n + j;
    }
    __device__ __forceinline__ void next(const GemmParams2& p) {
        const int g = visit % groups_per_m;
        ++j;
        if (j >= p.group_n || g * p.group_n + j >= p.tiles_n) { j = 0; visit += gridDim.x / NCTA; }
    }
};
template <int NCTA>
__device__ __forceinline__ TileInfo tile_info(const GemmParams2& p, int tile) {
    const int nb = tile % p.tiles_n, mb = tile / p.tiles_n;
    const int base = p.panels_total / p.tiles_n, rem = p.panels_total % p.tiles_n;
    TileInfo t;
    t.m0 = mb * kBM * NCTA;
    t.n0 = 64 * (nb * base + min(nb, rem));
    t.bn = 64 * (base + (nb < rem ? 1 : 0));
    // the last n-tile of a projection whose width is not a multiple of 64 (400, 420, 336, 160, 150 ...): columns past
    // round_up(N, 16) are K-padding zeros times anything - not issued (N = 400: 144 instead of 192 columns, -11 % MMA work)
    t.n_eff = min(t.bn, ((p.N - t.n0 + 15) >> 4) << 4);
    return t;
}

// ---- CTA-pair (cta_group::2) primitives ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {   // same smem offset in CTA `rank` of the cluster
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int x, int y, uint32_t bar_cluster) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(bar_cluster) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {   // arrives on the barrier at this offset in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
template <int NCTA> __device__ __forceinline__ void tmem_alloc_n(uint32_t slot_smem, uint32_t ncols) {
    if constexpr (NCTA == 1) {
        tmem_alloc(slot_smem, ncols);
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int NCTA> __device__ __forceinline__ void tmem_dealloc_n(uint32_t taddr, uint32_t ncols) {
    if constexpr (NCTA == 1) tmem_dealloc(taddr, ncols);
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128*NCTA, N=bn
template <int NCTA> __device__ __forceinline__ uint32_t make_idesc_n(int bn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)((kBM * NCTA) >> 4) << 24);
}

// NCTA == 1: one CTA per SM computes 128 x bn tiles.
// NCTA == 2: the two CTAs of a cluster (one TPC) compute 256 x bn tiles with tcgen05.mma.cta_group::2: each CTA
//   loads its own 128 rows of A and HALF of the W tile (bn/2 rows), the leader CTA issues the MMAs, which read both
//   CTAs' shared memory and write both CTAs' TMEM; each CTA runs the epilogue of its own 128 rows. Per flop this
//   halves the W bytes every SM pulls through the L2->SM fabric, which is what bounds the 128 x 256 single-CTA
//   tiles of the tall GAT projections (profiles/r01_v2_ncu_summary.md).
template <int NCTA>
__global__ void __launch_bounds__(kGemmThreads, 1) gemm_split_tc2_kernel(
    const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
    const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
    const __grid_constant__ CUtensorMap map_w2_hi, const __grid_constant__ CUtensorMap map_w2_lo,
    const __grid_constant__ CUtensorMap map_o_f32, const __grid_constant__ CUtensorMap map_o_hi,
    const __grid_constant__ CUtensorMap map_o_lo, const GemmParams2 p)
{
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    __shared__ __align__(8) uint64_t bar_full[kMaxStages];
    __shared__ __align__(8) uint64_t bar_empty[kMaxStages];
    __shared__ __align__(8) uint64_t bar_acc_full[2];
    __shared__ __align__(8) uint64_t bar_acc_empty[2];
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // rows to compute: the host's count, or - launched for a capacity - the count a previous kernel left on the device
    const int M_rows = p.m_dev ? min(p.M, __ldg(p.m_dev)) : p.M;
    const int tiles_m = p.m_dev ? (M_rows + kBM * NCTA - 1) / (kBM * NCTA) : p.tiles_m;
    const uint32_t rank = (NCTA == 2) ? cluster_ctarank() : 0u;
    const bool leader = rank == 0;
    const uint32_t a_bytes = kBM * kBK * 2;                                  // 16 KB per plane (this CTA's 128 rows)
    const uint32_t b_rows_stage = (uint32_t)p.stage_bn / NCTA;               // W rows this CTA holds per stage
    const uint32_t b_bytes = b_rows_stage * kBK * 2;
    const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;
    const uint32_t tiles_base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    const uint32_t staging_base = tiles_base + (uint32_t)p.stages * stage_bytes;   // 1024-aligned
    const uint32_t acc_cols = tmem_cols_for(p.stage_bn);
    const uint32_t ncols = 2 * acc_cols;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&bar_acc_full[a]), 1); mbar_init(smem_u32(&bar_acc_empty[a]), 4 * NCTA); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_w_hi); prefetch_tmap(&map_w_lo);
        prefetch_tmap(&map_w2_hi); prefetch_tmap(&map_w2_lo);
        if (p.has_f32) prefetch_tmap(&map_o_f32);
        if (p.has_planes) { prefetch_tmap(&map_o_hi); prefetch_tmap(&map_o_lo); }
    }
    if (warp == 1) tmem_alloc_n<NCTA>(smem_u32(&tmem_slot), ncols);
    tcgen05_fence_before();
    if constexpr (NCTA == 2) cluster_sync_all(); else __syncthreads();       // barriers of BOTH CTAs are initialised past this point
    tcgen05_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        // ================= TMA producer (every CTA loads its own operand halves) =================
        if (lane == 0) {
            int it = 0;
            for (TileWalk<NCTA> w(p, tiles_m); w.valid(); w.next(p)) {
                const TileInfo t = tile_info<NCTA>(p, w.tile(p));
                const int b_rows = t.bn / NCTA;                               // rows of the box this CTA loads per stage
                // this CTA's share of the W tile starts at its half of the columns that are multiplied (n_eff), not of the box
                const int m_cta = t.m0 + (int)rank * kBM, n_cta = t.n0 + (int)rank * (t.n_eff / NCTA);
                const uint32_t tx = NCTA * (2 * a_bytes + 2 * (uint32_t)b_rows * kBK * 2);   // bytes landing for the whole pair
                for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (uint32_t)(it / p.stages) & 1u;
                    mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1u);
                    const uint32_t full = smem_u32(&bar_full[s]);
                    const uint32_t base = tiles_base + (uint32_t)s * stage_bytes;
                    // one box per operand plane: the W maps are encoded with exactly this CTA's share of a wide (map_w_*)
                    // or a narrow (map_w2_*) tile as box height, so a k-block costs four TMA instructions
                    const CUtensorMap* mwh = (t.bn == p.stage_bn) ? &map_w_hi : &map_w2_hi;
                    const CUtensorMap* mwl = (t.bn == p.stage_bn) ? &map_w_lo : &map_w2_lo;
                    if constexpr (NCTA == 1) {
                        mbar_expect_tx(full, tx);
                        tma_load_2d(base, &map_a_hi, kb * kBK, m_cta, full);
                        tma_load_2d(base + a_bytes, &map_a_lo, kb * kBK, m_cta, full);
                        tma_load_2d(base + 2 * a_bytes, mwh, kb * kBK, n_cta, full);
                        tma_load_2d(base + 2 * a_bytes + b_bytes, mwl, kb * kBK, n_cta, full);
                    } else {
                        if (leader) mbar_expect_tx(full, tx);                 // the leader's barrier counts both CTAs' bytes
                        const uint32_t full0 = mapa_shared(full, 0);
                        tma_load_2d_pair(base, &map_a_hi, kb * kBK, m_cta, full0);
                        tma_load_2d_pair(base + a_bytes, &map_a_lo, kb * kBK, m_cta, full0);
                        tma_load_2d_pair(base + 2 * a_bytes, mwh, kb * kBK, n_cta, full0);
                        tma_load_2d_pair(base + 2 * a_bytes + b_bytes, mwl, kb * kBK, n_cta, full0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA only when paired) =================
        if (lane == 0 && leader) {
            int it = 0, i = 0;
            for (TileWalk<NCTA> w(p, tiles_m); w.valid(); w.next(p), ++i) {
                const TileInfo t = tile_info<NCTA>(p, w.tile(p));
                const uint32_t idesc = make_idesc_n<NCTA>(t.n_eff);
                const int a = i & 1;
                mbar_wait(smem_u32(&bar_acc_empty[a]), ((uint32_t)(i >> 1) & 1u) ^ 1u);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)a * acc_cols;
                for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (uint32_t)(it / p.stages) & 1u;
                    mbar_wait(smem_u32(&bar_full[s]), ph);
                    tcgen05_fence_after();
                    const uint32_t base = tiles_base + (uint32_t)s * stage_bytes;
                    const uint32_t sa_hi = base, sa_lo = base + a_bytes, sb_hi = base + 2 * a_bytes, sb_lo = base + 2 * a_bytes + b_bytes;
                    // k steps that are entirely K padding (zero planes) are not issued: 3 of the 28 steps of a K = 400
                    // projection - the operands an MMA reads from shared memory are the resource this kernel is bound by
                    const int nk4 = kb == p.num_kb - 1 ? p.k_last : kBK / kUmmaK;
#pragma unroll
                    for (int k4 = 0; k4 < kBK / kUmmaK; ++k4) {              // hi*hi, lo*hi, hi*lo per 16-wide k step
                        if (k4 >= nk4) break;
                        const uint32_t off = k4 * kUmmaK * 2;
                        const uint64_t dah = make_sw128_desc(sa_hi + off), dal = make_sw128_desc(sa_lo + off);
                        const uint64_t dbh = make_sw128_desc(sb_hi + off), dbl = make_sw128_desc(sb_lo + off);
                        const uint32_t first = (kb == 0 && k4 == 0) ? 0u : 1u;
                        if constexpr (NCTA == 1) {
                            umma_bf16(tmem_d, dah, dbh, idesc, first);
                            umma_bf16(tmem_d, dal, dbh, idesc, 1u);
                            umma_bf16(tmem_d, dah, dbl, idesc, 1u);
                        } else {
                            umma_bf16_pair(tmem_d, dah, dbh, idesc, first);
                            umma_bf16_pair(tmem_d, dal, dbh, idesc, 1u);
                            umma_bf16_pair(tmem_d, dah, dbl, idesc, 1u);
                        }
                    }
                    if constexpr (NCTA == 1) umma_commit(smem_u32(&bar_empty[s]));
                    else umma_commit_pair(smem_u32(&bar_empty[s]));           // frees the slot in both CTAs
                }
                if constexpr (NCTA == 1) umma_commit(smem_u32(&bar_acc_full[a]));
                else umma_commit_pair(smem_u32(&bar_acc_full[a]));
            }
        }
    } else {
        // ================= epilogue (each CTA drains its own 128 accumulator rows) =================
        const int q = warp & 3;                                   // TMEM lane quarter of this warp
        const uint32_t stage_f32 = staging_base + (uint32_t)(warp - 2) * (uint32_t)((p.has_f32 ? 8192 : 0) + (p.has_planes ? 8192 : 0));
        const uint32_t stage_hi = stage_f32 + (p.has_f32 ? 8192u : 0u);
        const uint32_t stage_lo = stage_hi + 4096u;
        const uint32_t sw = (uint32_t)(lane & 7);
        const uint32_t row_off = (uint32_t)lane * 128u;
        int i = 0;
        bool stores_pending = false;
        const bool slope_le1 = p.slope >= 0.f && p.slope <= 1.f;
        const bool bias_vec = p.bias != nullptr && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
        for (TileWalk<NCTA> w(p, tiles_m); w.valid(); w.next(p), ++i) {
            const TileInfo t = tile_info<NCTA>(p, w.tile(p));
            const int a = i & 1;
            mbar_wait(smem_u32(&bar_acc_full[a]), (uint32_t)(i >> 1) & 1u);
            tcgen05_fence_after();
            const uint32_t tmem_t = tmem_base + (uint32_t)a * acc_cols + ((uint32_t)(q * 32) << 16);
            const int npanels = t.bn / 64;
            float facc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int j = 0; j < npanels; ++j) {
                const int col0 = t.n0 + 64 * j;
                uint32_t r0[32], r1[32];
                tmem_ld_32x32(tmem_t + (uint32_t)(64 * j), r0);
                tmem_ld_32x32(tmem_t + (uint32_t)(64 * j + 32), r1);
                if (j == npanels - 1) {                           // accumulator drained: hand it back to the MMA warp
                    tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if constexpr (NCTA == 1) mbar_arrive(smem_u32(&bar_acc_empty[a]));
                        else mbar_arrive_cluster(mapa_shared(smem_u32(&bar_acc_empty[a]), 0));
                    }
                }
                float v[64];
                // full panels with a 16-byte aligned bias: every lane reads the panel's 64 bias values with 16 broadcast
                // vector loads (one L1 transaction each) instead of 128 shuffles - the epilogue warps share their
                // schedulers with the TMA and MMA issuing threads, so every instruction less is tensor-pipe time
                if (slope_le1 && bias_vec && col0 + 64 <= p.N) {
                    const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
                    // LeakyReLU(y) * s = max(y * s, y * slope * s) for s > 0 and slope <= 1; with s == 1 (every projection but the
                    // last MLP layer) one multiply disappears
                    const float s1 = p.out_scale, s2 = p.slope * p.out_scale;
                    if (s1 == 1.f) {
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const float4 ba = __ldg(b4 + c), bb = __ldg(b4 + 8 + c);
                            const float ya[4] = {__uint_as_float(r0[4 * c]) + ba.x, __uint_as_float(r0[4 * c + 1]) + ba.y,
                                                 __uint_as_float(r0[4 * c + 2]) + ba.z, __uint_as_float(r0[4 * c + 3]) + ba.w};
                            const float yb[4] = {__uint_as_float(r1[4 * c]) + bb.x, __uint_as_float(r1[4 * c + 1]) + bb.y,
                                                 __uint_as_float(r1[4 * c + 2]) + bb.z, __uint_as_float(r1[4 * c + 3]) + bb.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                v[4 * c + e] = fmaxf(ya[e], ya[e] * s2);
                                v[32 + 4 * c + e] = fmaxf(yb[e], yb[e] * s2);
                            }
                        }
                    } else if (s1 > 0.f) {
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const float4 ba = __ldg(b4 + c), bb = __ldg(b4 + 8 + c);
                            const float ya[4] = {__uint_as_float(r0[4 * c]) + ba.x, __uint_as_float(r0[4 * c + 1]) + ba.y,
                                                 __uint_as_float(r0[4 * c + 2]) + ba.z, __uint_as_float(r0[4 * c + 3]) + ba.w};
                            const float yb[4] = {__uint_as_float(r1[4 * c]) + bb.x, __uint_as_float(r1[4 * c + 1]) + bb.y,
                                                 __uint_as_float(r1[4 * c + 2]) + bb.z, __uint_as_float(r1[4 * c + 3]) + bb.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                v[4 * c + e] = fmaxf(ya[e] * s1, ya[e] * s2);
                                v[32 + 4 * c + e] = fmaxf(yb[e] * s1, yb[e] * s2);
                            }
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const float4 ba = __ldg(b4 + c), bb = __ldg(b4 + 8 + c);
                            const float ya[4] = {__uint_as_float(r0[4 * c]) + ba.x, __uint_as_float(r0[4 * c + 1]) + ba.y,
                                                 __uint_as_float(r0[4 * c + 2]) + ba.z, __uint_as_float(r0[4 * c + 3]) + ba.w};
                            const float yb[4] = {__uint_as_float(r1[4 * c]) + bb.x, __uint_as_float(r1[4 * c + 1]) + bb.y,
                                                 __uint_as_float(r1[4 * c + 2]) + bb.z, __uint_as_float(r1[4 * c + 3]) + bb.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                v[4 * c + e] = leaky_le1(ya[e], p.slope) * s1;
                                v[32 + 4 * c + e] = leaky_le1(yb[e], p.slope) * s1;
                            }
                        }
                    }
                } else {
                // bias of the panel: lane l holds columns col0+l and col0+32+l
                float b0 = 0.f, b1 = 0.f;
                if (p.bias) {
                    if (col0 + lane < p.N) b0 = __ldg(p.bias + col0 + lane);
                    if (col0 + 32 + lane < p.N) b1 = __ldg(p.bias + col0 + 32 + lane);
                }
                if (slope_le1) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const float bb0 = __shfl_sync(0xffffffffu, b0, c), bb1 = __shfl_sync(0xffffffffu, b1, c);
                        v[c] = (col0 + c < p.N) ? leaky_le1(__uint_as_float(r0[c]) + bb0, p.slope) * p.out_scale : 0.f;
                        v[32 + c] = (col0 + 32 + c < p.N) ? leaky_le1(__uint_as_float(r1[c]) + bb1, p.slope) * p.out_scale : 0.f;
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const float bb0 = __shfl_sync(0xffffffffu, b0, c), bb1 = __shfl_sync(0xffffffffu, b1, c);
                        v[c] = (col0 + c < p.N) ? leaky(__uint_as_float(r0[c]) + bb0, p.slope) * p.out_scale : 0.f;
                        v[32 + c] = (col0 + 32 + c < p.N) ? leaky(__uint_as_float(r1[c]) + bb1, p.slope) * p.out_scale : 0.f;
                    }
                }
                }
                if (p.fuse_n > 0) {
                    // second projection on the activated row in registers (this thread owns row m0 + rank*128 + q*32 + lane): the
                    // weight rows are read as broadcast float4 loads, all lanes the same address
#pragma unroll
                    for (int tt = 0; tt < 4; ++tt) {
                        if (tt >= p.fuse_n) break;
                        const float4* w4 = reinterpret_cast<const float4*>(p.fuse_w + (size_t)tt * p.fuse_ldw + col0);
                        float sacc = facc[tt];
#pragma unroll
                        for (int c = 0; c < 16; ++c) {
                            const float4 w = __ldg(w4 + c);
                            sacc = fmaf(v[4 * c], w.x, sacc); sacc = fmaf(v[4 * c + 1], w.y, sacc);
                            sacc = fmaf(v[4 * c + 2], w.z, sacc); sacc = fmaf(v[4 * c + 3], w.w, sacc);
                        }
                        facc[tt] = sacc;
                    }
                    if (j == npanels - 1) {
                        const int row = t.m0 + (int)rank * kBM + q * 32 + lane;
                        if (row < M_rows) {
                            for (int tt = 0; tt < p.fuse_n; ++tt) p.fuse_out[(size_t)row * p.fuse_ldo + tt] = facc[tt] + __ldg(p.fuse_b + tt);
                        }
                    }
                    continue;
                }
                if (stores_pending) {                             // staging buffers are about to be overwritten
                    if (lane == 0) bulk_wait_read0();
                    __syncwarp();
                }
                if (p.has_f32) {
#pragma unroll
                    for (int half = 0; half < 2; ++half)
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const uint32_t addr = stage_f32 + (uint32_t)half * 4096u + row_off + (((uint32_t)c ^ sw) << 4);
                            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v[half * 32 + 4 * c]),
                                         "f"(v[half * 32 + 4 * c + 1]), "f"(v[half * 32 + 4 * c + 2]), "f"(v[half * 32 + 4 * c + 3]) : "memory");
                        }
                }
                if (p.has_planes) {
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        uint32_t h[4], l[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) split_pack2(v[8 * c + 2 * u], v[8 * c + 2 * u + 1], h[u], l[u]);
                        const uint32_t off = row_off + (((uint32_t)c ^ sw) << 4);
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stage_hi + off), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stage_lo + off), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
                    }
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    const int row0 = t.m0 + (int)rank * kBM + q * 32;
                    if (row0 < M_rows) {
                        if (p.has_f32) {
                            if (col0 < p.N) tma_store_2d(&map_o_f32, stage_f32, col0, row0);
                            if (col0 + 32 < p.N) tma_store_2d(&map_o_f32, stage_f32 + 4096u, col0 + 32, row0);
                        }
                        if (p.has_planes) {
                            tma_store_2d(&map_o_hi, stage_hi, col0, row0);
                            tma_store_2d(&map_o_lo, stage_lo, col0, row0);
                        }
                    }
                    bulk_commit();
                }
                stores_pending = true;
            }
        }
        if (lane == 0) bulk_wait0();
    }
    tcgen05_fence_before();
    if constexpr (NCTA == 2) cluster_sync_all(); else __syncthreads();       // the peer still arrives on the leader's barriers until here
    if (warp == 1) tmem_dealloc_n<NCTA>(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------------
// Small-M kernel (m <= 8 rows: the pose MLP of a single frame). With a handful of rows the projection is a
// weight-streaming problem - the MLP holds 116 MB of hi/lo weights - and the tensor-core kernel would read them
// through the 12-48 CTAs its tiling yields. Here every warp owns output columns: it streams the hi/lo weight
// rows of a column with 16-byte loads (each weight read exactly once, all SMs pulling), keeps the A rows as fp32
// in shared memory, and reduces across lanes. Evaluates (a_hi + a_lo) . (w_hi + w_lo) in fp32, i.e. the same
// product as the 3-term tensor-core path plus the (negligible) lo*lo term.
// ------------------------------------------------------------------------------------------------
constexpr int kSmallM = 16;            // rows the weight-streaming kernel takes (8 accumulators per lane below 9 rows, 16 above)
constexpr int kSmallWarps = 16;

// Few rows (a live frame has a handful of persons): the layer is a stream of its weights - 116 MB of hi/lo planes for the
// pose MLP - against which a tensor-core tile would be 98 % padding. A is staged once per CTA as fp32 (hi + lo, exact:
// the planes are the split of an fp32 value) with 16-byte loads; every warp then streams whole weight rows (one output
// column each) with 16-byte loads, 8 in flight per lane, and the 32 lanes' partial dot products meet in a shuffle tree.
template <int MMAX>
__global__ void __launch_bounds__(kSmallWarps * 32) gemm_small_m_kernel(
    const __nv_bfloat16* __restrict__ a_hi, const __nv_bfloat16* __restrict__ a_lo, int lda,
    const __nv_bfloat16* __restrict__ w_hi, const __nv_bfloat16* __restrict__ w_lo, int ldw,
    const float* __restrict__ bias, int M, int N, int kpad, float slope, float out_scale,
    float* __restrict__ out_f32, int ld_out, __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, int ld_planes)
{
    extern __shared__ __align__(16) float As[];              // [M][kpad]
    {
        const int vec_per_row = kpad >> 3;                    // kpad is a multiple of 64, lda of 8
        for (int i = threadIdx.x; i < M * vec_per_row; i += blockDim.x) {
            const int m = i / vec_per_row, k8 = i - m * vec_per_row;
            const uint4 h = __ldg(reinterpret_cast<const uint4*>(a_hi + (size_t)m * lda) + k8);
            const uint4 l = __ldg(reinterpret_cast<const uint4*>(a_lo + (size_t)m * lda) + k8);
            const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
            float v[8];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                v[2 * e] = __uint_as_float(hw[e] << 16) + __uint_as_float(lw[e] << 16);
                v[2 * e + 1] = __uint_as_float(hw[e] & 0xffff0000u) + __uint_as_float(lw[e] & 0xffff0000u);
            }
            float4* d = reinterpret_cast<float4*>(As + (size_t)m * kpad + 8 * k8);
            d[0] = make_float4(v[0], v[1], v[2], v[3]);
            d[1] = make_float4(v[4], v[5], v[6], v[7]);
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_cols = out_hi ? ld_planes : N;               // plane padding columns are written as zeros
    for (int n = blockIdx.x * kSmallWarps + warp; n < n_cols; n += gridDim.x * kSmallWarps) {
        float acc[MMAX];
#pragma unroll
        for (int m = 0; m < MMAX; ++m) acc[m] = 0.f;
        if (n < N) {
            const uint4* wh = reinterpret_cast<const uint4*>(w_hi + (size_t)n * ldw);
            const uint4* wl = reinterpret_cast<const uint4*>(w_lo + (size_t)n * ldw);
#pragma unroll 4
            for (int k0 = lane * 8; k0 < kpad; k0 += 256) {
                const uint4 h = __ldg(wh + (k0 >> 3)), l = __ldg(wl + (k0 >> 3));
                const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
                float wv[8];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    wv[2 * e] = __uint_as_float(hw[e] << 16) + __uint_as_float(lw[e] << 16);
                    wv[2 * e + 1] = __uint_as_float(hw[e] & 0xffff0000u) + __uint_as_float(lw[e] & 0xffff0000u);
                }
#pragma unroll
                for (int m = 0; m < MMAX; ++m) {
                    if (m < M) {
                        const float4 x0 = *reinterpret_cast<const float4*>(As + (size_t)m * kpad + k0);
                        const float4 x1 = *reinterpret_cast<const float4*>(As + (size_t)m * kpad + k0 + 4);
                        acc[m] = fmaf(x0.x, wv[0], acc[m]); acc[m] = fmaf(x0.y, wv[1], acc[m]);
                        acc[m] = fmaf(x0.z, wv[2], acc[m]); acc[m] = fmaf(x0.w, wv[3], acc[m]);
                        acc[m] = fmaf(x1.x, wv[4], acc[m]); acc[m] = fmaf(x1.y, wv[5], acc[m]);
                        acc[m] = fmaf(x1.z, wv[6], acc[m]); acc[m] = fmaf(x1.w, wv[7], acc[m]);
                    }
                }
            }
        }
#pragma unroll
        for (int m = 0; m < MMAX; ++m)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], o);
        if (lane < M) {
            float v = 0.f;
#pragma unroll
            for (int m = 0; m < MMAX; ++m) if (m == lane) v = acc[m];
            if (n < N) v = leaky(v + (bias ? __ldg(bias + n) : 0.f), slope) * out_scale; else v = 0.f;
            if (out_f32 && n < N) out_f32[(size_t)lane * ld_out + n] = v;
            if (out_hi) {
                __nv_bfloat16 hh, ll;
                split_bf16(v, hh, ll);
                out_hi[(size_t)lane * ld_planes + n] = hh;
                out_lo[(size_t)lane * ld_planes + n] = ll;
            }
        }
    }
}

// The same layer when it is a pure weight stream (at most 8 rows, K <= 4096): the k range is split over the lanes of the
// whole CTA - lane (warp, lane) owns the 8 consecutive k values at (32 warp + lane) * 8 and keeps A[0..M) x those 8 in
// registers for the life of the CTA - and the CTA walks blocks of C = 32 / MMAX output columns. Per block a lane issues the
// 2 C 16-byte weight loads of its k slice back to back (nothing depends on shared memory, so they are all in flight
// together: 96 KB per CTA for K = 3072), forms its C x MMAX partial dot products, and the warp reduces all 32 of them at
// once with a 31-shuffle transposing butterfly (lane l ends up with the warp total of partial l) instead of 5 shuffles per
// value; one shared-memory hop adds the warps. A is never staged, and the weights are touched exactly once.
template <int MMAX>
__global__ void __launch_bounds__(512, 1) gemm_stream_kernel(
    const __nv_bfloat16* __restrict__ a_hi, const __nv_bfloat16* __restrict__ a_lo, int lda,
    const __nv_bfloat16* __restrict__ w_hi, const __nv_bfloat16* __restrict__ w_lo, int ldw,
    const float* __restrict__ bias, int M, int N, int kpad, float slope, float out_scale,
    float* __restrict__ out_f32, int ld_out, __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, int ld_planes)
{
    constexpr int C = 32 / MMAX;
    __shared__ float part[2][16][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int k0 = (warp * 32 + lane) * 8;
    const bool active = k0 < kpad;
    auto unpack = [](const uint4& h, const uint4& l, float (&v)[8]) {
        const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            v[2 * e] = __uint_as_float(hw[e] << 16) + __uint_as_float(lw[e] << 16);
            v[2 * e + 1] = __uint_as_float(hw[e] & 0xffff0000u) + __uint_as_float(lw[e] & 0xffff0000u);
        }
    };
    float a[MMAX][8];
#pragma unroll
    for (int m = 0; m < MMAX; ++m) {
#pragma unroll
        for (int j = 0; j < 8; ++j) a[m][j] = 0.f;
        if (m < M && active)
            unpack(__ldg(reinterpret_cast<const uint4*>(a_hi + (size_t)m * lda + k0)),
                   __ldg(reinterpret_cast<const uint4*>(a_lo + (size_t)m * lda + k0)), a[m]);
    }
    const int n_cols = out_hi ? ld_planes : N;               // plane padding columns are written as zeros
    const int n_blocks = (n_cols + C - 1) / C;
    int it = 0;
    for (int cb = blockIdx.x; cb < n_blocks; cb += gridDim.x, ++it) {
        const int n0 = cb * C;
        uint4 wh[C], wl[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            wh[c] = make_uint4(0u, 0u, 0u, 0u); wl[c] = wh[c];
            if (active && n0 + c < N) {
                wh[c] = __ldg(reinterpret_cast<const uint4*>(w_hi + (size_t)(n0 + c) * ldw + k0));
                wl[c] = __ldg(reinterpret_cast<const uint4*>(w_lo + (size_t)(n0 + c) * ldw + k0));
            }
        }
        float v[32];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float w[8];
            unpack(wh[c], wl[c], w);
#pragma unroll
            for (int m = 0; m < MMAX; ++m) {
                float s = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) s = fmaf(a[m][j], w[j], s);
                v[c * MMAX + m] = s;
            }
        }
        // transposing butterfly: after the step with offset o a lane keeps the half of its values whose index has bit o
        // equal to its own lane bit, summed with its partner's copy; lane l ends with the warp total of value l
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < o; ++i) {
                const float keep = upper ? v[i + o] : v[i];
                const float send = upper ? v[i] : v[i + o];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
        }
        part[it & 1][warp][lane] = v[0];
        __syncthreads();
        if (warp == 0) {
            float t = 0.f;
            for (int w = 0; w < n_warps; ++w) t += part[it & 1][w][lane];
            const int n = n0 + lane / MMAX, m = lane % MMAX;
            if (m < M && n < n_cols) {
                float y = 0.f;
                if (n < N) y = leaky(t + (bias ? __ldg(bias + n) : 0.f), slope) * out_scale;
                if (out_f32 && n < N) out_f32[(size_t)m * ld_out + n] = y;
                if (out_hi) {
                    __nv_bfloat16 hh, ll;
                    split_bf16(y, hh, ll);
                    out_hi[(size_t)m * ld_planes + n] = hh;
                    out_lo[(size_t)m * ld_planes + n] = ll;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
    }
    return fn;
}

static int make_map_ex(CUtensorMap* map, CUtensorMapDataType dt, int elt, const void* base, int rows, int cols, int ld,
                       int box_cols, int box_rows) {
    auto fn = get_encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return B200POSE_E_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * elt};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %d cols %d ld %d box %dx%d)", (int)r, rows, cols, ld, box_cols, box_rows);
        return B200POSE_E_CUDA;
    }
    return B200POSE_OK;
}
static int make_map(CUtensorMap* map, const void* base, int rows, int kpad, int ld, int box_rows) {
    return make_map_ex(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, kpad, ld, kBK, box_rows);
}

static int num_sms() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

}  // namespace b200pose

using namespace b200pose;


struct FuseArgs { const float* w; const float* b; float* out; int n, ldw, ldo; };

static int linear_impl(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                       const uint16_t* w_hi, const uint16_t* w_lo, int32_t ldw,
                       const float* bias, int32_t m, const int32_t* m_dev, int32_t n, int32_t k, float slope, float out_scale,
                       float* out_f32, int32_t ld_out, uint16_t* out_hi, uint16_t* out_lo, int32_t ld_planes,
                       int32_t impl, void* stream, const FuseArgs* fuse = nullptr)
{
    B2_CHECK_ARG(impl == 0 || impl == 4 || impl == 5 || impl == 7, "linear: impl must be 0 (dispatch), 4 (persistent, single CTAs), "
                 "5 (persistent, CTA pairs) or 7 (few-row kernels when m <= 16)");
    B2_CHECK_ARG(a_hi && a_lo && w_hi && w_lo, "linear: null operand");
    if (fuse) {
        B2_CHECK_ARG(impl == 0 && !m_dev, "linear_fused2: impl must be 0");
        B2_CHECK_ARG(fuse->w && fuse->b && fuse->out && fuse->n >= 1 && fuse->n <= 4, "linear_fused2: 1..4 fused output columns");
        B2_CHECK_ARG(n <= 256, "linear_fused2: the first projection must fit one n-tile (n <= 256)");
        B2_CHECK_ARG(fuse->ldw % 4 == 0 && fuse->ldw >= ((n + 63) / 64) * 64 && ((uintptr_t)fuse->w % 16 == 0), "linear_fused2: fused weight rows must be 16-byte aligned and padded to a multiple of 64 columns");
        B2_CHECK_ARG(fuse->ldo >= fuse->n, "linear_fused2: ld_out2 < n2");
        B2_CHECK_ARG(!out_f32 && !out_hi, "linear_fused2: the first projection is not stored");
    }
    if (m_dev) B2_CHECK_ARG(impl == 0 || impl == 4 || impl == 5, "linear_n: only the persistent kernels read the row count from the device");
    B2_CHECK_ARG(m >= 0 && n >= 1 && k >= 1, "linear: bad shape m=%d n=%d k=%d", m, n, k);
    const int kpad = ceil_div(k, kBK) * kBK;
    B2_CHECK_ARG(lda % 64 == 0 && ldw % 64 == 0 && lda >= kpad && ldw >= kpad, "linear: lda/ldw must be multiples of 64 >= round_up(k,64)");
    B2_CHECK_ARG(out_f32 || out_hi || fuse, "linear: no output requested");
    B2_CHECK_ARG((out_hi == nullptr) == (out_lo == nullptr), "linear: planes go together");
    if (out_f32) B2_CHECK_ARG(ld_out >= n, "linear: ld_out < n");
    if (out_hi) B2_CHECK_ARG(ld_planes % 64 == 0 && ld_planes >= n, "linear: ld_planes must be a multiple of 64 >= n");
    B2_CHECK_ARG(((uintptr_t)a_hi % 16 == 0) && ((uintptr_t)a_lo % 16 == 0) && ((uintptr_t)w_hi % 16 == 0) && ((uintptr_t)w_lo % 16 == 0),
                 "linear: operands must be 16-byte aligned");
    if (m == 0) return B200POSE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    // the few-row kernels take the planes as bf16 pointers
    const __nv_bfloat16* ah = reinterpret_cast<const __nv_bfloat16*>(a_hi);
    const __nv_bfloat16* al = reinterpret_cast<const __nv_bfloat16*>(a_lo);
    const __nv_bfloat16* wh = reinterpret_cast<const __nv_bfloat16*>(w_hi);
    const __nv_bfloat16* wl = reinterpret_cast<const __nv_bfloat16*>(w_lo);
    __nv_bfloat16* oh = reinterpret_cast<__nv_bfloat16*>(out_hi);
    __nv_bfloat16* ol = reinterpret_cast<__nv_bfloat16*>(out_lo);
    if (!m_dev && !fuse && (impl == 0 || impl == 7) && m <= 8 && kpad <= 4096 && lda % 8 == 0 && ldw % 8 == 0) {
        // weight stream with A in registers: k split over the CTA's lanes, blocks of 32 / MMAX columns
        const int warps = ceil_div(kpad, 256);
        const int cols = out_hi ? ld_planes : n;
        const int per_sm = warps >= 12 ? 1 : warps >= 6 ? 2 : 4;              // ~96 KB of weight loads in flight per SM
        auto launch_stream = [&](auto kern, int c_per_block) -> int {
            int ctas = ceil_div(cols, c_per_block);
            if (ctas > num_sms() * per_sm) ctas = num_sms() * per_sm;
            kern<<<ctas, warps * 32, 0, st>>>(ah, al, lda, wh, wl, ldw, bias, m, n, kpad, slope, out_scale,
                                              out_f32, ld_out, oh, ol, ld_planes);
            B2_CHECK_LAUNCH();
            return B200POSE_OK;
        };
        return m <= 4 ? launch_stream(gemm_stream_kernel<4>, 8) : launch_stream(gemm_stream_kernel<8>, 4);
    }
    if (!m_dev && !fuse && (impl == 0 || impl == 7) && m <= kSmallM && (size_t)m * kpad * sizeof(float) <= 200 * 1024 && lda % 8 == 0 && ldw % 8 == 0) {
        // weight-streaming small-M kernel: as many CTAs as fit at once (the A staging is per CTA), every warp takes columns
        const size_t smem = (size_t)m * kpad * sizeof(float);
        const int cols = out_hi ? ld_planes : n;
        int ctas = ceil_div(cols, kSmallWarps);
        const int cap = num_sms() * (smem <= 100 * 1024 ? 2 : 1);
        if (ctas > cap) ctas = cap;
        auto launch_small = [&](auto kern) -> int {
            B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<ctas, kSmallWarps * 32, smem, st>>>(ah, al, lda, wh, wl, ldw, bias, m, n, kpad, slope, out_scale,
                                                       out_f32, ld_out, oh, ol, ld_planes);
            B2_CHECK_LAUNCH();
            return B200POSE_OK;
        };
        return m <= 8 ? launch_small(gemm_small_m_kernel<8>) : launch_small(gemm_small_m_kernel<16>);
    }
    // ---- persistent kernel ----
    if (out_f32) B2_CHECK_ARG(ld_out % 4 == 0 && ((uintptr_t)out_f32 % 16 == 0), "linear: out_f32 needs ld_out %% 4 == 0 and 16-byte alignment (TMA store)");
    if (out_hi) B2_CHECK_ARG(((uintptr_t)out_hi % 16 == 0) && ((uintptr_t)out_lo % 16 == 0), "linear: output planes must be 16-byte aligned");
    // CTA pairs (cta_group::2, 256-row tiles) as soon as there is more than one pair tile of rows: per flop a pair pulls
    // 1.5x fewer bytes through the L2->SM fabric, which bounds both the tall GAT projections and the MLP (every m-tile
    // re-reads the whole weight matrix from L2)
    const int ncta = (impl == 5) ? 2 : (impl == 4) ? 1 : (m > 4 * kBM ? 2 : 1);
    GemmParams2 q;
    q.M = m; q.N = n; q.num_kb = kpad / kBK; q.k_last = ceil_div(k - (kpad / kBK - 1) * kBK, kUmmaK); q.bias = bias; q.slope = slope; q.out_scale = out_scale;
    q.has_f32 = out_f32 ? 1 : 0; q.has_planes = out_hi ? 1 : 0; q.m_dev = m_dev;
    q.fuse_n = 0; q.fuse_w = nullptr; q.fuse_b = nullptr; q.fuse_out = nullptr; q.fuse_ldw = 0; q.fuse_ldo = 0;
    if (fuse) { q.fuse_n = fuse->n; q.fuse_w = fuse->w; q.fuse_b = fuse->b; q.fuse_out = fuse->out; q.fuse_ldw = fuse->ldw; q.fuse_ldo = fuse->ldo; }
    q.panels_total = ceil_div(n, 64);                         // 64-column panels; planes panels also zero columns [n, 64*panels)
    const size_t staging = 4 * (size_t)((q.has_f32 ? 8192 : 0) + (q.has_planes ? 8192 : 0));
    CUtensorMap ma_hi, ma_lo, mw_hi, mw_lo, mw2_hi, mw2_lo, mo_f32, mo_hi, mo_lo;
    int rc;
    if ((rc = make_map(&ma_hi, a_hi, m, kpad, lda, kBM))) return rc;
    if ((rc = make_map(&ma_lo, a_lo, m, kpad, lda, kBM))) return rc;
    mo_f32 = ma_hi; mo_hi = ma_hi; mo_lo = ma_hi;                              // placeholders when unused
    if (out_f32 && (rc = make_map_ex(&mo_f32, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out_f32, m, n, ld_out, 32, 32))) return rc;
    if (out_hi) {
        if ((rc = make_map_ex(&mo_hi, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, out_hi, m, ld_planes, ld_planes, 64, 32))) return rc;
        if ((rc = make_map_ex(&mo_lo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, out_lo, m, ld_planes, ld_planes, 64, 32))) return rc;
    }
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    q.tiles_n = ceil_div(q.panels_total, 4);
    q.tiles_m = ceil_div(m, kBM * ncta);
    // a handful of m-tiles (single-frame calls: ~180 graph nodes): one 64-column panel per tile, so that the k-loops of
    // an output row run side by side on many SMs instead of back to back on one - latency, not throughput, matters here
    if (impl == 0 && ncta == 1 && !fuse && q.tiles_m * q.tiles_n * 8 < num_sms()) q.tiles_n = q.panels_total;
    q.stage_bn = 64 * ceil_div(q.panels_total, q.tiles_n);
    const size_t stage2 = 2 * (size_t)kBM * kBK * 2 + 2 * (size_t)(q.stage_bn / ncta) * kBK * 2;
    int stages = (int)((227 * 1024 - 2048 - staging) / stage2);
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 1) { set_error("linear: tile does not fit in shared memory"); return B200POSE_E_UNSUPPORTED; }
    q.stages = stages;
    const size_t smem = (size_t)stages * stage2 + staging + 1024;
    // n-tiles are `base` or `base + 1` panels wide (tile_info): one W map per width, box height = one CTA's share
    const int panels_narrow = q.panels_total / q.tiles_n;
    const int bn_narrow = 64 * (panels_narrow < 1 ? 1 : panels_narrow);
    if ((rc = make_map(&mw_hi, w_hi, n, kpad, ldw, q.stage_bn / ncta))) return rc;
    if ((rc = make_map(&mw_lo, w_lo, n, kpad, ldw, q.stage_bn / ncta))) return rc;
    if ((rc = make_map(&mw2_hi, w_hi, n, kpad, ldw, bn_narrow / ncta))) return rc;
    if ((rc = make_map(&mw2_lo, w_lo, n, kpad, ldw, bn_narrow / ncta))) return rc;
    // tall GEMMs (GAT projections: thousands of m-tiles, 1-2 n-tiles): sweep the n-tiles of an m-tile inside one worker
    const int workers_max = num_sms() / ncta;
    q.group_n = (q.tiles_m >= 2 * workers_max) ? q.tiles_n : 1;
    const int total_visits = q.tiles_m * ceil_div(q.tiles_n, q.group_n);
    const int workers = total_visits < workers_max ? total_visits : workers_max;
    if (ncta == 1) {
        B2_CHECK_CUDA(cudaFuncSetAttribute(gemm_split_tc2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gemm_split_tc2_kernel<1><<<workers, kGemmThreads, smem, st>>>(ma_hi, ma_lo, mw_hi, mw_lo, mw2_hi, mw2_lo, mo_f32, mo_hi, mo_lo, q);
        B2_CHECK_LAUNCH();
    } else {
        B2_CHECK_CUDA(cudaFuncSetAttribute(gemm_split_tc2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * workers); cfg.blockDim = dim3(kGemmThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cfg.attrs = attr; cfg.numAttrs = 1;
        B2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_split_tc2_kernel<2>, ma_hi, ma_lo, mw_hi, mw_lo, mw2_hi, mw2_lo, mo_f32, mo_hi, mo_lo, q));
    }
    return B200POSE_OK;
}

extern "C" __attribute__((visibility("default"))) int b200pose_linear(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                               const uint16_t* w_hi, const uint16_t* w_lo, int32_t ldw,
                               const float* bias, int32_t m, int32_t n, int32_t k, float slope, float out_scale,
                               float* out_f32, int32_t ld_out, uint16_t* out_hi, uint16_t* out_lo, int32_t ld_planes,
                               int32_t impl, void* stream)
{
    return linear_impl(a_hi, a_lo, lda, w_hi, w_lo, ldw, bias, m, nullptr, n, k, slope, out_scale, out_f32, ld_out, out_hi, out_lo, ld_planes, impl, stream);
}

extern "C" __attribute__((visibility("default"))) int b200pose_linear_n(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                                 const uint16_t* w_hi, const uint16_t* w_lo, int32_t ldw,
                                 const float* bias, int32_t m_capacity, const int32_t* m_dev, int32_t n, int32_t k, float slope, float out_scale,
                                 float* out_f32, int32_t ld_out, uint16_t* out_hi, uint16_t* out_lo, int32_t ld_planes,
                                 int32_t impl, void* stream)
{
    B2_CHECK_ARG(m_dev, "linear_n: null row-count pointer");
    return linear_impl(a_hi, a_lo, lda, w_hi, w_lo, ldw, bias, m_capacity, m_dev, n, k, slope, out_scale, out_f32, ld_out, out_hi, out_lo, ld_planes, impl, stream);
}

extern "C" __attribute__((visibility("default"))) int b200pose_linear_fused2(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                                      const uint16_t* w1_hi, const uint16_t* w1_lo, int32_t ldw1, const float* bias1,
                                      int32_t m, int32_t n1, int32_t k, float slope1,
                                      const float* w2_f32, int32_t ldw2, const float* bias2, int32_t n2,
                                      float* out2_f32, int32_t ld_out2, void* stream)
{
    FuseArgs f;
    f.w = w2_f32; f.b = bias2; f.out = out2_f32; f.n = n2; f.ldw = ldw2; f.ldo = ld_out2;
    return linear_impl(a_hi, a_lo, lda, w1_hi, w1_lo, ldw1, bias1, m, nullptr, n1, k, slope1, 1.0f, nullptr, 0, nullptr, nullptr, 0, 0, stream, &f);
}
