// Tensor-core path of the blend-shape contraction (the only GEMM-shaped work of the fit):
//
//   k_blend_fwd_tc : v_posed tile [128 frames x 192 coords] = pf @ Bm on tcgen05 (kind::tf32,
//                    3xTF32 split: hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM), operands
//                    staged by TMA (swizzled, K-major) through a 4-stage mbarrier pipeline,
//                    persistent CTAs with two TMEM accumulators (MMA of tile i+1 overlaps the
//                    read-out of tile i), accumulator read back with tcgen05.ld and written as
//                    row-contiguous v_posed.  Skinning is NOT done here: it gathers 192 B of joint
//                    transforms per vertex and frame, which bound a fused epilogue at ~37 us per
//                    tile whatever the GEMM depth (L2 gather); the fit's per-frame kernel skins its
//                    live vertices from shared memory instead (bf_frame.cuh) and the all-vertex
//                    operator uses k_skin_rows (bf_skin.cuh, transforms resident in shared memory).
//   k_blend_bwd_tc : dpf tile [128 frames x <=256 k] = dvp @ Bm^T, same machinery, reduction over
//                    the vertex coordinates.
//
// Warp roles: warp 0 = TMA producer (one lane), warp 1 = TMEM allocator + MMA issuer (one lane),
// warps 2.. = epilogue (TMEM lane quarter = warp_idx % 4).
//
// Why 3xTF32: single TF32 (10-bit mantissa) leaves ~5e-4 relative error on the blend-shape
// offsets, i.e. ~1e-5 of the vertex magnitude -- at the north-star tolerance (1e-5 relative on
// vertices) and, more importantly, too coarse for the 1e-4 per-iteration loss parity through 100
// Adam steps.  The split keeps the error at ~2^-21 per product (measured: see DESIGN.md).
#pragma once
#include <cuda.h>
#include <stdlib.h>
#include "bf_common.cuh"

#define TC_BM 128          // frames per tile (UMMA M)
#ifndef TC_BK
#define TC_BK 16           // fp32 elements per K chunk = one swizzle row (16 -> SWIZZLE_64B, 32 -> SWIZZLE_128B)
#endif
#define TC_ROWB (TC_BK * 4)   // bytes per operand row of one K chunk
#define TC_BN1 192         // coords per tile in the forward (64 vertices)
#ifndef TC_STAGES
#define TC_STAGES (TC_BK == 16 ? 4 : 2)   // the same 160 KB of operand staging, but up to three chunks in flight instead of one
#endif

namespace tc {

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major swizzled operand tile: rows of TC_ROWB bytes (= the swizzle span), 8-row groups 8 * TC_ROWB apart (SBO), LBO unused (=1)
__device__ __forceinline__ uint64_t make_desc(const void* smem_tile) {
    const uint32_t a = smem_u32(smem_tile);
    uint64_t d = 0;
    d |= (uint64_t)((a >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * TC_ROWB) >> 4) << 32;
    d |= (uint64_t)1 << 46;          // descriptor version 1 (Blackwell)
    d |= (uint64_t)(TC_BK == 32 ? 2 : 4) << 61;          // layout type: SWIZZLE_128B = 2, SWIZZLE_64B = 4
    return d;
}
__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared main loop: warp 0 lane 0 streams K chunks with TMA, warp 1 lane 0 issues the MMAs.
// Stage layout: A_hi | A_lo | B_hi | B_lo, each a [rows x TC_ROWB] swizzled tile.
struct Pipe {
    uint8_t* stage_base;
    uint64_t* full;
    uint64_t* empty;
    uint64_t* tmem_full;      // one barrier (backward GEMM) or two (double-buffered forward)
    uint32_t a_bytes, b_bytes;
    __device__ __forceinline__ uint32_t stage_bytes() const { return 2 * a_bytes + 2 * b_bytes; }
    __device__ __forceinline__ uint8_t* stage(int s) const { return stage_base + (size_t)s * stage_bytes(); }
};

// blk_mask != ~0u (needs TC_BK == 16): the reduction runs only over the 16-vertex blocks (3 chunks of 16 coordinates each)
// whose bit is set -- the other columns of the A operand are exactly zero for every row of this tile
template <int NS>
__device__ __forceinline__ void producer(const Pipe& p, const CUtensorMap* mA_hi, const CUtensorMap* mA_lo,
                                         const CUtensorMap* mB_hi, const CUtensorMap* mB_lo, int num_k, int rowA, int rowB,
                                         int kc_begin = 0, uint32_t blk_mask = 0xFFFFFFFFu, int pipe0 = 0) {
    for (int kc = 0; kc < num_k; ++kc) {
        const int s = (pipe0 + kc) % NS;                    // pipe0: chunks already sent through the pipeline by an earlier run
        const uint32_t ph = ((pipe0 + kc) / NS) & 1;
        mbar_wait(&p.empty[s], ph ^ 1);
        mbar_expect_tx(&p.full[s], p.stage_bytes());
        uint8_t* st = p.stage(s);
        const int kk = kc_begin + kc;                       // masked: index into the tile's list of (set block, chunk) pairs
        const int chunk = blk_mask == 0xFFFFFFFFu ? kk : 3 * (int)__fns(blk_mask, 0, kk / 3 + 1) + kk % 3;
        const int c0 = chunk * TC_BK;
        tma_load_2d(st, mA_hi, &p.full[s], c0, rowA);
        tma_load_2d(st + p.a_bytes, mA_lo, &p.full[s], c0, rowA);
        tma_load_2d(st + 2 * p.a_bytes, mB_hi, &p.full[s], c0, rowB);
        tma_load_2d(st + 2 * p.a_bytes + p.b_bytes, mB_lo, &p.full[s], c0, rowB);
    }
}

template <int NS>
__device__ __forceinline__ void mma_issuer(const Pipe& p, int num_k, uint32_t tmem_d, uint32_t idesc, int pipe0 = 0,
                                           bool last = true) {
    for (int kc = 0; kc < num_k; ++kc) {
        const int s = (pipe0 + kc) % NS;
        const uint32_t ph = ((pipe0 + kc) / NS) & 1;
        mbar_wait(&p.full[s], ph);
        tc_fence_after();
        uint8_t* st = p.stage(s);
        const uint64_t a_hi = make_desc(st), a_lo = make_desc(st + p.a_bytes);
        const uint64_t b_hi = make_desc(st + 2 * p.a_bytes), b_lo = make_desc(st + 2 * p.a_bytes + p.b_bytes);
#pragma unroll
        for (int k = 0; k < TC_BK / 8; ++k) {            // UMMA K = 8 tf32 = 32 B -> +2 in the 16-byte address field
            const uint64_t o = (uint64_t)(2 * k);
            umma_tf32(tmem_d, a_hi + o, b_hi + o, idesc, (kc | k) ? 1u : 0u);
            umma_tf32(tmem_d, a_lo + o, b_hi + o, idesc, 1u);
            umma_tf32(tmem_d, a_hi + o, b_lo + o, idesc, 1u);
        }
        umma_commit(&p.empty[s]);                        // frees the smem slot when these MMAs have read it
    }
    if (last) umma_commit(p.tmem_full);                  // accumulator(s) complete
}

}  // namespace tc

// Persistent: one CTA per SM walks the (frame tile, vertex tile) list.  Two TMEM accumulators: the MMA warp fills
// buffer (i+1)&1 while the eight epilogue warps drain buffer i&1.  Epilogue warps 2..9: TMEM lane quarter
// q = warp % 4 (lane = frame row of the tile), vertex half h = (warp - 2) / 4 of the 64-vertex tile, two passes of
// 16 vertices (48 accumulator columns), transposed through a per-warp shared tile so that the global stores are
// row-contiguous (192 B per frame row).
#define TC_BAND 64         // frame tiles per band of the tile order
// Tile order: bands of TC_BAND frame tiles; inside a band the frame tile runs fastest, then the vertex tile.  The CTAs
// that run together then share a few model-matrix tiles (each read from DRAM once per band and re-used from L2 by the
// whole band) while the band's pose-feature rows (<= 64 x 128 frames x Kp x 8 B = 33 MB at Kp = 512) stay L2-resident.
// (Vertex-tile-fastest order streamed the whole 128 MB SMPL-X model matrix once per frame tile: 4 GB of DRAM reads
// for a 10,000-frame all-vertex forward.)
__device__ __forceinline__ void tc_tile_coords(int t, int tm, int tn, int& fm, int& vn) {
    const int per_band = TC_BAND * tn;
    const int band = t / per_band, rem = t - band * per_band;
    const int bs = min(TC_BAND, tm - band * TC_BAND);
    vn = rem / bs;
    fm = band * TC_BAND + (rem - vn * bs);
}
#define TC_EPI_WARPS 8
#define TC_ST_LD 33        // row stride (floats) of the per-warp [48 coords][32 frames] staging tile
#define TC_ST_FLOATS (48 * TC_ST_LD)

namespace tc {
// 48 consecutive accumulator columns of this warp's 32 lanes -> registers (one wait for the three loads)
__device__ __forceinline__ void tmem_ld48(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%48];\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%49];\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47}, [%50];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]),
          "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]),
          "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47])
        : "r"(taddr), "r"(taddr + 16u), "r"(taddr + 32u)
        : "memory");
}

// staging tile [48 coords][32 frames] -> rows of `dst` (row stride ld floats), `ncols` valid coords, `nrows` valid frames.
// 2 rows x 48 coords = 96 elements = 3 warp-wide stores per step; a lane's three (row-of-the-pair, coord) slots are fixed,
// so a full tile is walked with pointer increments only.
__device__ __forceinline__ void store_rows48(const float* st, float* __restrict__ dst, size_t ld, int ncols, int nrows, int lane) {
    if (nrows == 32 && ncols == 48) {
        const int hi1 = lane >= 16, c1 = lane + 32 - 48 * hi1;
        const size_t g0 = (size_t)lane, g1 = (size_t)hi1 * ld + c1, g2 = ld + lane + 16;
        const float* s0 = st + lane * TC_ST_LD;
        const float* s1 = st + c1 * TC_ST_LD + hi1;
        const float* s2 = st + (lane + 16) * TC_ST_LD + 1;
#pragma unroll 8
        for (int rp = 0; rp < 16; ++rp, dst += 2 * ld) {
            dst[g0] = s0[2 * rp]; dst[g1] = s1[2 * rp]; dst[g2] = s2[2 * rp];
        }
        return;
    }
#pragma unroll 4
    for (int rp = 0; rp < 16; ++rp) {
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int idx = lane + 32 * s, hi = idx >= 48;
            const int fr = 2 * rp + hi, c = idx - 48 * hi;
            if (fr < nrows && c < ncols) dst[(size_t)fr * ld + c] = st[c * TC_ST_LD + fr];
        }
    }
}
}  // namespace tc

__global__ void __launch_bounds__(64 + 32 * TC_EPI_WARPS, 1)
k_blend_fwd_tc(const __grid_constant__ CUtensorMap mA_hi, const __grid_constant__ CUtensorMap mA_lo,
               const __grid_constant__ CUtensorMap mB_hi, const __grid_constant__ CUtensorMap mB_lo,
               int n_verts, int Kp, float* __restrict__ vposed, int B, int ld_v, int n_tiles_m, int n_tiles_n, int n_tiles) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    tc::Pipe p;
    p.a_bytes = TC_BM * TC_ROWB;
    p.b_bytes = TC_BN1 * TC_ROWB;
    p.stage_base = base;
    float* St = reinterpret_cast<float*>(base + TC_STAGES * p.stage_bytes());
    uint64_t* bars = reinterpret_cast<uint64_t*>(St + TC_EPI_WARPS * TC_ST_FLOATS);
    p.full = bars; p.empty = bars + TC_STAGES; p.tmem_full = bars + 2 * TC_STAGES;      // tmem_full[2]
    uint64_t* tmem_empty = bars + 2 * TC_STAGES + 2;                                   // tmem_empty[2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k = Kp / TC_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { tc::mbar_init(&p.full[s], 1); tc::mbar_init(&p.empty[s], 1); }
        for (int s = 0; s < 2; ++s) { tc::mbar_init(&p.tmem_full[s], 1); tc::mbar_init(&tmem_empty[s], TC_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int it = 0;                                              // running K-chunk counter across tiles
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                int fm, vn;
                tc_tile_coords(t, n_tiles_m, n_tiles_n, fm, vn);
                const int b0 = fm * TC_BM, n0 = vn * TC_BN1;
                for (int kc = 0; kc < num_k; ++kc, ++it) {
                    const int s = it % TC_STAGES;
                    const uint32_t ph = (it / TC_STAGES) & 1;
                    tc::mbar_wait(&p.empty[s], ph ^ 1);
                    tc::mbar_expect_tx(&p.full[s], p.stage_bytes());
                    uint8_t* st = p.stage(s);
                    tc::tma_load_2d(st, &mA_hi, &p.full[s], kc * TC_BK, b0);
                    tc::tma_load_2d(st + p.a_bytes, &mA_lo, &p.full[s], kc * TC_BK, b0);
                    tc::tma_load_2d(st + 2 * p.a_bytes, &mB_hi, &p.full[s], kc * TC_BK, n0);
                    tc::tma_load_2d(st + 2 * p.a_bytes + p.b_bytes, &mB_lo, &p.full[s], kc * TC_BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = tc::make_idesc_tf32(TC_BM, TC_BN1);
            int it = 0, i = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
                const int buf = i & 1;
                tc::mbar_wait(&tmem_empty[buf], ((i >> 1) & 1) ^ 1);          // epilogue has drained this accumulator
                tc::tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(buf * TC_BN1);
                for (int kc = 0; kc < num_k; ++kc, ++it) {
                    const int s = it % TC_STAGES;
                    const uint32_t ph = (it / TC_STAGES) & 1;
                    tc::mbar_wait(&p.full[s], ph);
                    tc::tc_fence_after();
                    uint8_t* st = p.stage(s);
                    const uint64_t a_hi = tc::make_desc(st), a_lo = tc::make_desc(st + p.a_bytes);
                    const uint64_t b_hi = tc::make_desc(st + 2 * p.a_bytes), b_lo = tc::make_desc(st + 2 * p.a_bytes + p.b_bytes);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k) {
                        const uint64_t o = (uint64_t)(2 * k);
                        tc::umma_tf32(tmem_d, a_hi + o, b_hi + o, idesc, (kc | k) ? 1u : 0u);
                        tc::umma_tf32(tmem_d, a_lo + o, b_hi + o, idesc, 1u);
                        tc::umma_tf32(tmem_d, a_hi + o, b_lo + o, idesc, 1u);
                    }
                    tc::umma_commit(&p.empty[s]);
                }
                tc::umma_commit(&p.tmem_full[buf]);
            }
        }
    } else {
        const int q = warp & 3;                               // TMEM lane quarter this warp may read
        const int h = (warp - 2) >> 2;                        // which 32 vertices of the 64-vertex tile
        float* st = St + (warp - 2) * TC_ST_FLOATS;
        int i = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
            const int buf = i & 1;
            int fm, vn;
            tc_tile_coords(t, n_tiles_m, n_tiles_n, fm, vn);
            const int b0 = fm * TC_BM + 32 * q, n0 = vn * TC_BN1;
            const int nrows = min(32, B - b0);
            tc::mbar_wait(&p.tmem_full[buf], (i >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t tmem_d = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * TC_BN1 + h * 96);
#pragma unroll 1
            for (int pass = 0; pass < 2; ++pass) {
                uint32_t r[48];
                tc::tmem_ld48(tmem_d + (uint32_t)(pass * 48), r);
                if (pass == 1) {                              // accumulator half fully read: hand it back to the MMA warp
                    tc::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(&tmem_empty[buf])) : "memory");
                }
                const int vbase = n0 / 3 + h * 32 + pass * 16;
                if (vbase >= n_verts || nrows <= 0) continue; // warp-uniform: pad vertices / pad frames of the last tiles
#pragma unroll
                for (int c = 0; c < 48; ++c) st[c * TC_ST_LD + lane] = __uint_as_float(r[c]);
                __syncwarp();
                tc::store_rows48(st, vposed + (size_t)b0 * ld_v + 3 * vbase, (size_t)ld_v, 3 * min(16, n_verts - vbase), nrows, lane);
                __syncwarp();
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
}

// Block-masked forward blend of the active set: per 128-frame tile only the 16-vertex blocks (48 coordinates) named by the
// tile's mask are computed (BfFrames.blk_mask: OR over the tile's frames of the blocks their contour row needs; with the
// frames of a batch sorted by row that is ~16 of 30 blocks).  A "virtual" N tile gathers up to four such blocks: the B operand
// stage is assembled from four 48-row TMA boxes taken at the blocks' rows of the blend matrix (the 64-byte swizzle repeats
// every 8 rows = 512 B, so boxes placed 48 rows apart form the same layout as one 192-row box), the MMA runs with
// N = 48 x blocks, and the epilogue stores each 48-column group at its block's own column offset of v_posed.  Columns of
// blocks outside the mask are not written -- no frame of the tile reads them.
// Slot order: virtual tile index major, frame tile minor -- every frame tile has at least three virtual tiles (the static
// blocks), so consecutive slots are almost all real and the static round-robin over the CTAs stays balanced.
#define TC_BLK_ROWS 48
#define BW_SPLIT_BLOCK 8
#define TC_MAX_VT 8
__global__ void __launch_bounds__(64 + 32 * TC_EPI_WARPS, 1)
k_blend_fwd_tc_blk(const __grid_constant__ CUtensorMap mA_hi, const __grid_constant__ CUtensorMap mA_lo,
                   const __grid_constant__ CUtensorMap mB_hi, const __grid_constant__ CUtensorMap mB_lo,
                   const __grid_constant__ CUtensorMap mB4_hi, const __grid_constant__ CUtensorMap mB4_lo,
                   int n_verts, int Kp, float* __restrict__ vposed, int B, int ld_v, int n_tiles_m,
                   const uint32_t* __restrict__ blk_mask, int n_blocks) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    tc::Pipe p;
    p.a_bytes = TC_BM * TC_ROWB;
    p.b_bytes = TC_BN1 * TC_ROWB;
    p.stage_base = base;
    float* St = reinterpret_cast<float*>(base + TC_STAGES * p.stage_bytes());
    uint64_t* bars = reinterpret_cast<uint64_t*>(St + TC_EPI_WARPS * TC_ST_FLOATS);
    p.full = bars; p.empty = bars + TC_STAGES; p.tmem_full = bars + 2 * TC_STAGES;
    uint64_t* tmem_empty = bars + 2 * TC_STAGES + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k = Kp / TC_BK;
    const int n_slots = n_tiles_m * TC_MAX_VT;
    const uint32_t valid = n_blocks < 32 ? (1u << n_blocks) - 1u : 0xFFFFFFFFu;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { tc::mbar_init(&p.full[s], 1); tc::mbar_init(&p.empty[s], 1); }
        for (int s = 0; s < 2; ++s) { tc::mbar_init(&p.tmem_full[s], 1); tc::mbar_init(&tmem_empty[s], TC_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int it = 0;
            for (int t = blockIdx.x; t < n_slots; t += gridDim.x) {
                const int vt = t / n_tiles_m, fm = t - vt * n_tiles_m;
                const uint32_t mask = __ldg(blk_mask + fm) & valid;
                const int nb = min(4, __popc(mask) - 4 * vt);
                if (nb <= 0) continue;
                int rows[4];
                for (int j = 0; j < nb; ++j) rows[j] = TC_BLK_ROWS * (int)__fns(mask, 0, 4 * vt + j + 1);
                // four consecutive blocks (the static part of the set): one 192-row box instead of four 48-row ones.  (Boxes of
                // two and three blocks for shorter runs were measured and lost: 72 -> 83 us per 10,000 frames.)
                const bool run4 = nb == 4 && rows[3] == rows[0] + 3 * TC_BLK_ROWS;
                const int b0 = fm * TC_BM;
                const uint32_t bytes = 2 * p.a_bytes + 2u * (uint32_t)nb * TC_BLK_ROWS * TC_ROWB;
                for (int kc = 0; kc < num_k; ++kc, ++it) {
                    const int s = it % TC_STAGES;
                    const uint32_t ph = (it / TC_STAGES) & 1;
                    tc::mbar_wait(&p.empty[s], ph ^ 1);
                    tc::mbar_expect_tx(&p.full[s], bytes);
                    uint8_t* st = p.stage(s);
                    tc::tma_load_2d(st, &mA_hi, &p.full[s], kc * TC_BK, b0);
                    tc::tma_load_2d(st + p.a_bytes, &mA_lo, &p.full[s], kc * TC_BK, b0);
                    if (run4) {
                        tc::tma_load_2d(st + 2 * p.a_bytes, &mB4_hi, &p.full[s], kc * TC_BK, rows[0]);
                        tc::tma_load_2d(st + 2 * p.a_bytes + p.b_bytes, &mB4_lo, &p.full[s], kc * TC_BK, rows[0]);
                    } else {
                        for (int j = 0; j < nb; ++j) {
                            tc::tma_load_2d(st + 2 * p.a_bytes + j * TC_BLK_ROWS * TC_ROWB, &mB_hi, &p.full[s], kc * TC_BK, rows[j]);
                            tc::tma_load_2d(st + 2 * p.a_bytes + p.b_bytes + j * TC_BLK_ROWS * TC_ROWB, &mB_lo, &p.full[s], kc * TC_BK, rows[j]);
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int it = 0, i = 0;
            for (int t = blockIdx.x; t < n_slots; t += gridDim.x) {
                const int vt = t / n_tiles_m, fm = t - vt * n_tiles_m;
                const uint32_t mask = __ldg(blk_mask + fm) & valid;
                const int nb = min(4, __popc(mask) - 4 * vt);
                if (nb <= 0) continue;
                const uint32_t idesc = tc::make_idesc_tf32(TC_BM, TC_BLK_ROWS * nb);
                const int buf = i & 1;
                tc::mbar_wait(&tmem_empty[buf], ((i >> 1) & 1) ^ 1);
                tc::tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(buf * TC_BN1);
                for (int kc = 0; kc < num_k; ++kc, ++it) {
                    const int s = it % TC_STAGES;
                    const uint32_t ph = (it / TC_STAGES) & 1;
                    tc::mbar_wait(&p.full[s], ph);
                    tc::tc_fence_after();
                    uint8_t* st = p.stage(s);
                    const uint64_t a_hi = tc::make_desc(st), a_lo = tc::make_desc(st + p.a_bytes);
                    const uint64_t b_hi = tc::make_desc(st + 2 * p.a_bytes), b_lo = tc::make_desc(st + 2 * p.a_bytes + p.b_bytes);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k) {
                        const uint64_t o = (uint64_t)(2 * k);
                        tc::umma_tf32(tmem_d, a_hi + o, b_hi + o, idesc, (kc | k) ? 1u : 0u);
                        tc::umma_tf32(tmem_d, a_lo + o, b_hi + o, idesc, 1u);
                        tc::umma_tf32(tmem_d, a_hi + o, b_lo + o, idesc, 1u);
                    }
                    tc::umma_commit(&p.empty[s]);
                }
                tc::umma_commit(&p.tmem_full[buf]);
                ++i;
            }
        }
    } else {
        const int q = warp & 3;
        const int h = (warp - 2) >> 2;
        float* st = St + (warp - 2) * TC_ST_FLOATS;
        int i = 0;
        for (int t = blockIdx.x; t < n_slots; t += gridDim.x) {
            const int vt = t / n_tiles_m, fm = t - vt * n_tiles_m;
            const uint32_t mask = __ldg(blk_mask + fm) & valid;
            const int nb = min(4, __popc(mask) - 4 * vt);
            if (nb <= 0) continue;                              // warp-uniform, and the same decision in all three roles
            const int buf = i & 1;
            const int b0 = fm * TC_BM + 32 * q;
            const int nrows = min(32, B - b0);
            tc::mbar_wait(&p.tmem_full[buf], (i >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t tmem_d = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * TC_BN1 + h * 96);
#pragma unroll 1
            for (int pass = 0; pass < 2; ++pass) {
                const int j = 2 * h + pass;                     // which of the tile's (up to) four blocks
                uint32_t r[48];
                if (j < nb) tc::tmem_ld48(tmem_d + (uint32_t)(pass * 48), r);
                if (pass == 1) {
                    tc::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(&tmem_empty[buf])) : "memory");
                }
                if (j >= nb || nrows <= 0) continue;
                const int vbase = 16 * (int)__fns(mask, 0, 4 * vt + j + 1);
                if (vbase >= n_verts) continue;
#pragma unroll
                for (int c = 0; c < 48; ++c) st[c * TC_ST_LD + lane] = __uint_as_float(r[c]);
                __syncwarp();
                tc::store_rows48(st, vposed + (size_t)b0 * ld_v + 3 * vbase, (size_t)ld_v, 3 * min(16, n_verts - vbase), nrows, lane);
                __syncwarp();
            }
            ++i;
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
}

// dpf[b, k0 + c] = sum_n dvp[b, n] Bm[k0 + c, n]; BN = columns of this CTA (multiple of 16, <= 256); NS = pipeline stages
// (4: one CTA per SM; 2 with BN <= 128: 67 KB and 128 TMEM columns per CTA, so three CTAs share an SM and a grid a little
// larger than the SM count does not leave a nearly empty second wave)
template <int NS>
__global__ void __launch_bounds__(192, 1) k_blend_bwd_tc(const __grid_constant__ CUtensorMap mA_hi,
                                                         const __grid_constant__ CUtensorMap mA_lo,
                                                         const __grid_constant__ CUtensorMap mB_hi,
                                                         const __grid_constant__ CUtensorMap mB_lo,
                                                         int BN, int num_k_total, int cps, int Kp,
                                                         float* __restrict__ out, size_t split_stride, int B,
                                                         const uint32_t* __restrict__ blk_mask, int fuse_halves) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    tc::Pipe p;
    p.a_bytes = TC_BM * TC_ROWB;
    p.b_bytes = (uint32_t)BN * TC_ROWB;
    p.stage_base = base;
    uint64_t* bars = reinterpret_cast<uint64_t*>(base + NS * p.stage_bytes());
    p.full = bars; p.empty = bars + NS; p.tmem_full = bars + 2 * NS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NS + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b0 = blockIdx.y * TC_BM;
    const int k0 = blockIdx.x * BN;
    const int acc_cols = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    const int tmem_cols = fuse_halves ? 2 * acc_cols : acc_cols;
    // split-K: this CTA reduces K chunks [kc_begin, kc_begin + num_k) and writes its own partial
    // (the tensor-core accumulator truncates, so long reductions are cut and summed in fp32 RN)
    int kc_begin = blockIdx.z * cps;
    uint32_t mask = 0xFFFFFFFFu, mask2 = 0u;
    int num_k;
    if (blk_mask) {
        // masked reduction: 3 chunks per set block.  With gridDim.z == 2 the reduction is cut at a FIXED block (BW_SPLIT_BLOCK:
        // the first eight blocks are static, i.e. always set; the rest holds three static and the ~5 contour blocks of a tile),
        // run z reduces its side of the cut and the consumer adds the two partial sums in a fixed order.  The cut does not
        // depend on the mask, so an element's summation order -- and the result -- is the same for every batch and frame order.
        mask = blk_mask[blockIdx.y];
        const int nblk = num_k_total / 3;
        if (nblk < 32) mask &= (1u << nblk) - 1u;
        if (gridDim.z == 2 || fuse_halves) {
            const uint32_t low = (1u << min(BW_SPLIT_BLOCK, nblk / 2)) - 1u;
            mask2 = mask & ~low;
            mask = gridDim.z == 2 ? (blockIdx.z == 0 ? (mask & low) : mask2) : (mask & low);
            if (mask == 0xFFFFFFFFu) mask = 0xFFFFFFFEu;   // cannot happen (a half never has 32 blocks); keeps the masked path
        }
    }
    // fuse_halves: the same two half-reductions, run one after the other by ONE CTA into two TMEM accumulators that the
    // epilogue adds -- the arithmetic of the two-CTA form (acc0 + acc1 in fp32, then the consumer's sum) without the second
    // output buffer; the launcher picks it for large batches, where the grid fills the SMs anyway
    int num_k2 = 0;
    if (blk_mask && (gridDim.z == 2 || fuse_halves || mask != 0xFFFFFFFFu)) {
        kc_begin = 0;
        num_k = 3 * __popc(mask);
        if (fuse_halves) num_k2 = 3 * __popc(mask2);
    } else {
        mask = 0xFFFFFFFFu;
        num_k = min(cps, num_k_total - kc_begin);
    }
    float* dpf = out + (size_t)blockIdx.z * split_stride;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) { tc::mbar_init(&p.full[s], 1); tc::mbar_init(&p.empty[s], 1); }
        tc::mbar_init(p.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(tmem_slot)), "r"(tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            if (num_k > 0) tc::producer<NS>(p, &mA_hi, &mA_lo, &mB_hi, &mB_lo, num_k, b0, k0, kc_begin, mask);
            if (num_k2 > 0) tc::producer<NS>(p, &mA_hi, &mA_lo, &mB_hi, &mB_lo, num_k2, b0, k0, 0, mask2, num_k);
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = tc::make_idesc_tf32(TC_BM, BN);
            if (num_k > 0) tc::mma_issuer<NS>(p, num_k, tmem_d, idesc, 0, num_k2 == 0);
            if (num_k2 > 0) tc::mma_issuer<NS>(p, num_k2, tmem_d + (uint32_t)acc_cols, idesc, num_k, true);
        }
    } else {
        if (num_k + num_k2 > 0) {
            tc::mbar_wait(p.tmem_full, 0);
            tc::tc_fence_after();
        }
        const int q = warp & 3;
        const int b = b0 + 32 * q + lane;
        for (int c = 0; c < BN; c += 32) {
            uint32_t r[32];
            if (num_k > 0) tc::tmem_ld32(tmem_d + ((uint32_t)(32 * q) << 16) + (uint32_t)c, r);
            else {
#pragma unroll
                for (int i = 0; i < 32; ++i) r[i] = 0u;                        // empty mask: the gradient rows are zero
            }
            if (fuse_halves) {
                uint32_t r2[32];
                if (num_k2 > 0) tc::tmem_ld32(tmem_d + ((uint32_t)(32 * q) << 16) + (uint32_t)(acc_cols + c), r2);
                else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) r2[i] = 0u;
                }
#pragma unroll
                for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(r2[i]));
            }
            if (b < B) {
                float4* o = reinterpret_cast<float4*>(dpf + (size_t)b * Kp + k0 + c);
                const int nv = (BN - c >= 32) ? 8 : (BN - c) / 4;
                for (int i = 0; i < nv; ++i)
                    o[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]),
                                       __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(tmem_cols));
    }
}

// dst[i] = sum_z ws[z][i], fixed order (deterministic); n is a multiple of 4 (Kp % 16 == 0)
__global__ void __launch_bounds__(256) k_sum_partials(const float* __restrict__ ws, float* __restrict__ dst, size_t n, int S) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n) return;
    float4 a = *reinterpret_cast<const float4*>(ws + i);
    for (int z = 1; z < S; ++z) {
        const float4 b = *reinterpret_cast<const float4*>(ws + (size_t)z * n + i);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    *reinterpret_cast<float4*>(dst + i) = a;
}

// ---------------------------------------------------------------------------------------------
// host side
typedef CUresult (*bf_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static bf_encode_tiled_fn bf_get_encode() {
    static bf_encode_tiled_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<bf_encode_tiled_fn>(ptr);
    }
    return fn;
}

// Tensor maps describe (address, shape, box) only, so one encoded for a buffer stays valid for as long as the same view of
// the same address is used: the per-iteration launches of a fit re-use them from this table instead of calling the
// driver twelve times per iteration (the operands of a session never move).
struct BfMapKey { const void* base; uint64_t rows, cols, ld; uint32_t box_rows; int dev; };
struct BfMapEntry { BfMapKey k; CUtensorMap map; };
#define BF_MAP_CACHE 512
static BfMapEntry g_map_cache[BF_MAP_CACHE];
static int g_map_used = 0;

static int bf_make_map_uncached(CUtensorMap* m, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows);
// [rows, cols] fp32 row-major with leading dimension ld (elements); box = TC_BK cols (one swizzle row) x box_rows
static int bf_make_map(CUtensorMap* m, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    const int dev = bf_cur_dev();
    std::lock_guard<std::mutex> lk(g_bf_mu);
    for (int i = 0; i < g_map_used; ++i) {
        const BfMapKey& k = g_map_cache[i].k;
        if (k.base == base && k.rows == rows && k.cols == cols && k.ld == ld && k.box_rows == box_rows && k.dev == dev) {
            *m = g_map_cache[i].map;
            return BF_OK;
        }
    }
    const int rc = bf_make_map_uncached(m, base, rows, cols, ld, box_rows);
    if (rc) return rc;
    if (g_map_used == BF_MAP_CACHE) g_map_used = 0;            // full: start over (entries are only a cache)
    g_map_cache[g_map_used].k = BfMapKey{base, rows, cols, ld, box_rows, dev};
    g_map_cache[g_map_used].map = *m;
    ++g_map_used;
    return BF_OK;
}
static int bf_make_map_uncached(CUtensorMap* m, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    bf_encode_tiled_fn enc = bf_get_encode();
    if (!enc) { bf_set_error("cuTensorMapEncodeTiled not available from the driver"); return BF_ECUDA; }
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * sizeof(float)};
    cuuint32_t box[2] = {TC_BK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, TC_BK == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { bf_set_error("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu", (int)r,
                                          (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld); return BF_ECUDA; }
    return BF_OK;
}

// BODYFIT_BLKMASK=0: the GEMMs touch every block of the active set (A/B timing, debugging)
static inline bool bf_blk_mask_on() {
    static int env = -1;
    if (env < 0) { const char* e = getenv("BODYFIT_BLKMASK"); env = e ? atoi(e) : 1; }
    return env != 0;
}
static inline bool bf_tc_ready_fwd(const BfVSet* vs, const BfFrames* f) {
    return (f->flags & BF_F_TC) && vs->Bt_hi && vs->Bt_lo && f->pf_hi && f->pf_lo;
}
static inline bool bf_tc_ready_bwd(const BfVSet* vs, const BfFrames* f) {
    return (f->flags & BF_F_TC) && vs->Bm_hi && vs->Bm_lo && f->dvp_hi && f->dvp_lo;
}

// dst[B, ld_dst] (first 3 * n_verts columns) = A[B, Kp] @ Bt[ldn, Kp]^T on the tensor cores, operands pre-split for 3xTF32.
// Used for the blend shapes (A = pose features, Bt = blend matrix) and for the GMM prior (A = [pose | 1], Bt = precisions).
static int bf_gemm_forward_tc(const float* a_hi_p, const float* a_lo_p, const float* bt_hi_p, const float* bt_lo_p, int B, int Kp,
                              int ldn, int n_verts, float* dst, int ld_dst, cudaStream_t s) {
    CUtensorMap a_hi, a_lo, b_hi, b_lo;
    int rc;
    if (Kp % TC_BK != 0 || ldn % 3 != 0) { bf_set_error("bf_gemm_forward_tc: Kp=%d / ldn=%d not tileable", Kp, ldn); return BF_EINVAL; }
    if ((rc = bf_make_map(&a_hi, a_hi_p, B, Kp, Kp, TC_BM))) return rc;
    if ((rc = bf_make_map(&a_lo, a_lo_p, B, Kp, Kp, TC_BM))) return rc;
    if ((rc = bf_make_map(&b_hi, bt_hi_p, ldn, Kp, Kp, TC_BN1))) return rc;
    if ((rc = bf_make_map(&b_lo, bt_lo_p, ldn, Kp, Kp, TC_BN1))) return rc;
    const size_t smem = 1024 + TC_STAGES * (2 * TC_BM * TC_ROWB + 2 * TC_BN1 * TC_ROWB) + TC_EPI_WARPS * TC_ST_FLOATS * 4 + 128;
    static size_t attr[BF_MAXDEV] = {0};
    if ((rc = bf_ensure_smem(k_blend_fwd_tc, smem, attr, "k_blend_fwd_tc"))) return rc;
    const int num_sms = bf_num_sms();
    const int tn = (ldn + TC_BN1 - 1) / TC_BN1, tm = (B + TC_BM - 1) / TC_BM;
    const int tiles = tn * tm;
    const int grid = tiles < num_sms ? tiles : num_sms;          // persistent: one CTA per SM
    k_blend_fwd_tc<<<grid, 64 + 32 * TC_EPI_WARPS, smem, s>>>(a_hi, a_lo, b_hi, b_lo, n_verts, Kp, dst, B, ld_dst, tm, tn, tiles);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// block-masked forward of the active set (k_blend_fwd_tc_blk); returns 1 when not applicable
static int bf_gemm_forward_tc_blk(const float* a_hi_p, const float* a_lo_p, const float* bt_hi_p, const float* bt_lo_p, int B, int Kp,
                                  int ldn, int n_verts, float* dst, int ld_dst, const uint32_t* blk_mask, cudaStream_t s) {
    const int n_blocks = (ldn / 3 + 15) / 16;
    if (TC_BK != 16 || Kp % TC_BK != 0 || ldn % (3 * 16) != 0 || n_blocks > 32 || n_blocks > 4 * TC_MAX_VT) return 1;
    CUtensorMap a_hi, a_lo, b_hi, b_lo;
    int rc;
    if ((rc = bf_make_map(&a_hi, a_hi_p, B, Kp, Kp, TC_BM))) return rc;
    if ((rc = bf_make_map(&a_lo, a_lo_p, B, Kp, Kp, TC_BM))) return rc;
    if ((rc = bf_make_map(&b_hi, bt_hi_p, ldn, Kp, Kp, TC_BLK_ROWS))) return rc;
    if ((rc = bf_make_map(&b_lo, bt_lo_p, ldn, Kp, Kp, TC_BLK_ROWS))) return rc;
    CUtensorMap b4_hi, b4_lo;
    if ((rc = bf_make_map(&b4_hi, bt_hi_p, ldn, Kp, Kp, TC_BN1))) return rc;
    if ((rc = bf_make_map(&b4_lo, bt_lo_p, ldn, Kp, Kp, TC_BN1))) return rc;
    const size_t smem = 1024 + TC_STAGES * (2 * TC_BM * TC_ROWB + 2 * TC_BN1 * TC_ROWB) + TC_EPI_WARPS * TC_ST_FLOATS * 4 + 128;
    static size_t attr[BF_MAXDEV] = {0};
    if ((rc = bf_ensure_smem(k_blend_fwd_tc_blk, smem, attr, "k_blend_fwd_tc_blk"))) return rc;
    const int num_sms = bf_num_sms();
    const int tm = (B + TC_BM - 1) / TC_BM;
    // at most ceil(n_blocks / 4) virtual tiles per frame tile are real; one CTA per SM, fewer when there is less work
    const int real_max = tm * ((n_blocks + 3) / 4);
    const int grid = real_max < num_sms ? real_max : num_sms;
    k_blend_fwd_tc_blk<<<grid, 64 + 32 * TC_EPI_WARPS, smem, s>>>(a_hi, a_lo, b_hi, b_lo, b4_hi, b4_lo, n_verts, Kp, dst, B, ld_dst, tm, blk_mask, n_blocks);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// v_posed[B, ld_v] = pf @ Bm (dst = f->vposed, or any [B, ld_v] buffer)
static int bf_gemm_forward_tc2(const float* a_hi_p, const float* a_lo_p, const float* bt_hi_p, const float* bt_lo_p, int B, int Kp,
                               int ldn, int n_verts, float* dst, int ld_dst, cudaStream_t s);      // bf_blend_tc2.cuh
static int bf_blend_forward_tc(const BfModel* m, const BfVSet* vs, const BfFrames* f, float* dst, cudaStream_t s) {
    if (bf_blk_mask_on() && f->blk_mask && vs->lv_blk && vs == &m->act) {
        const int rcb = bf_gemm_forward_tc_blk(f->pf_hi, f->pf_lo, vs->Bt_hi, vs->Bt_lo, f->B, m->Kp, vs->ldn, vs->n, dst, f->ld_v,
                                               f->blk_mask + (size_t)(f->iter & 1) * ((f->B + 127) / 128), s);
        if (rcb != 1) return rcb;
    }
    const int rc2 = bf_gemm_forward_tc2(f->pf_hi, f->pf_lo, vs->Bt_hi, vs->Bt_lo, f->B, m->Kp, vs->ldn, vs->n, dst, f->ld_v, s);
    if (rc2 != 1) return rc2;                              // CTA-pair kernel ran (or failed loudly); 1 = not applicable
    return bf_gemm_forward_tc(f->pf_hi, f->pf_lo, vs->Bt_hi, vs->Bt_lo, f->B, m->Kp, vs->ldn, vs->n, dst, f->ld_v, s);
}

// Column tile of the backward GEMM: the widest multiple of 16 (the MMA's N granule) up to 256 that divides Kp.  The kernel
// streams its operands from L2 and every column tile re-reads the whole dvp row block, so the widest tile wins even when it
// leaves a partial last wave: measured on 10,000 frames x Kp 512, 64 / 128 / 256 columns = 0.134 / 0.123 / 0.109 ms (158 CTAs
// on 148 SMs).  Kp = round16(P + NS + 1) is 224 or 240 for SMPL and 512 or 496 for SMPL-X (496 = 16 x 31: NS <= 9, 16-column
// tiles).  Kp is a multiple of 16 (check_model), so a tile always exists.
static int bf_bwd_col_tile(int Kp) {
    for (int bn = Kp < 256 ? Kp : 256; bn > 16; bn -= 16)
        if (Kp % bn == 0) return bn;
    return 16;
}

// The masked backward GEMM always reduces a tile in two halves cut at a fixed block (BW_SPLIT_BLOCK) and adds the two
// partial sums.  Two forms of the same arithmetic: two CTAs per tile writing dpf and dpf2 (summed by k_pose_bwd), chosen
// when even the doubled grid is at most one wave -- the batch is small and bound by the latency of one CTA's K loop -- and
// one CTA per tile with two TMEM accumulators added in its epilogue otherwise (no second buffer to write and re-read).
static bool bf_bwd_two_cta(const BfModel* m, const BfFrames* f) {
    if (!f->dpf2 || !f->blk_mask || !bf_blk_mask_on()) return false;
    const int BN = bf_bwd_col_tile(m->Kp);
    const int mt = (f->B + TC_BM - 1) / TC_BM;
    return (m->Kp / BN) * mt * 2 <= bf_num_sms();
}

static int bf_blend_backward_tc(const BfModel* m, const BfVSet* vs, const BfFrames* f, cudaStream_t s) {
    CUtensorMap a_hi, a_lo, b_hi, b_lo;
    int rc;
    const int num_sms = bf_num_sms();
    int BN = bf_bwd_col_tile(m->Kp);                     // the tile bf_bwd_two_cta assumes (narrowed below for small batches)
    if (m->Kp % BN != 0 || BN % 16 != 0) { bf_set_error("Kp=%d not tileable by %d", m->Kp, BN); return BF_EINVAL; }
    // Small batches (a shard of a strong-scaled sequence: 1,250 frames x Kp 512 = 20 tiles of 256 columns on 148 SMs): narrower
    // column tiles until the grid covers at least half of the SMs.  Every output element still accumulates its K products
    // in the same order, so the result does not depend on the tile width (bit-identical across batch sizes, tested).
    if (vs->ldn / TC_BK <= 2048 / TC_BK) {                 // single accumulation run only (the all-vertex backward is split-K)
        const int mt = (f->B + TC_BM - 1) / TC_BM;
        const int halves = bf_bwd_two_cta(m, f) ? 2 : 1;
        while (BN > 64 && (m->Kp / BN) * mt * halves * 2 < num_sms && m->Kp % (BN / 2) == 0 && (BN / 2) % 16 == 0) BN /= 2;
    }
    {
        static int forced = -1;                           // BODYFIT_BWD_BN=64|128|256: tile-width experiments
        if (forced < 0) { const char* e = getenv("BODYFIT_BWD_BN"); forced = e ? atoi(e) : 0; }
        if (forced > 0 && forced <= m->Kp && m->Kp % forced == 0 && forced % 16 == 0 && forced <= 256) BN = forced;
    }
    if ((rc = bf_make_map(&a_hi, f->dvp_hi, f->B, vs->ldn, vs->ldn, TC_BM))) return rc;
    if ((rc = bf_make_map(&a_lo, f->dvp_lo, f->B, vs->ldn, vs->ldn, TC_BM))) return rc;
    if ((rc = bf_make_map(&b_hi, vs->Bm_hi, m->Kp, vs->ldn, vs->ldn, BN))) return rc;
    if ((rc = bf_make_map(&b_lo, vs->Bm_lo, m->Kp, vs->ldn, vs->ldn, BN))) return rc;
    // pipeline depth: TC_STAGES with one CTA per SM, or 2 stages with narrow tiles so that three CTAs share an SM
    int NS = TC_STAGES;
    {
        static int st_env = -1;                           // BODYFIT_BWD_STAGES=2|4: experiments
        if (st_env < 0) { const char* e = getenv("BODYFIT_BWD_STAGES"); st_env = e ? atoi(e) : 0; }
        if (st_env == 2) NS = 2;                        // measured: slower in the full fit at either width (DESIGN.md section 4)
        // narrow tiles (small batches, see above): a CTA's K loop is bound by the round trip of a stage (commit -> TMA ->
        // MMA, ~1.8 us; measured 0.45 us per chunk with 4 stages whatever the tile width), so the freed shared memory buys a
        // deeper pipeline: 8 stages of 16 + 2 x 4 KB
        else if (BN <= 64 && TC_BK == 16 && st_env != 4) NS = 8;
    }
    const size_t smem = 1024 + NS * (2 * TC_BM * TC_ROWB + 2 * (size_t)BN * TC_ROWB) + 64;
    static size_t attr[2][BF_MAXDEV] = {{0}};
    static size_t attr8[BF_MAXDEV] = {0};
    if ((rc = NS == 2 ? bf_ensure_smem(k_blend_bwd_tc<2>, smem, attr[1], "k_blend_bwd_tc<2>")
            : NS == 8 ? bf_ensure_smem(k_blend_bwd_tc<8>, smem, attr8, "k_blend_bwd_tc<8>")
                      : bf_ensure_smem(k_blend_bwd_tc<TC_STAGES>, smem, attr[0], "k_blend_bwd_tc"))) return rc;
    const int num_k = vs->ldn / TC_BK;
    const size_t stride = (size_t)f->B * m->Kp;
    // split-K: at most 2048 coordinates per tensor-core accumulation run (accuracy, see above); when the (frame tile x
    // column tile) grid alone leaves SMs idle -- the all-vertex backward of a ~1000-frame batch has 8 tiles and a 20k-long
    // reduction -- the reduction is cut further, into as many runs as fill the SMs once (workspace permitting)
    int cps = 2048 / TC_BK;
    int S = (num_k + cps - 1) / cps;
    if (S > 1 && (!f->ws || (size_t)f->ws_floats < (size_t)S * stride)) return 1;   // caller falls back to the FFMA kernel
    {
        const int tiles = (m->Kp / BN) * ((f->B + TC_BM - 1) / TC_BM);
        int S_fill = num_sms / tiles;
        if (S_fill > num_k) S_fill = num_k;
        // Off by default: the GEMM alone gets faster (SMPL x 1024 frames: 100 -> 77 us) but the all-vertex backward as a whole
        // slower (327 -> 341 us) -- its 144 large-shared-memory CTAs crowd out the dA gather kernel that runs next to it on the
        // side stream, which is the longer of the two; and a batch-size dependent split would make results depend on the
        // batch size in the last bit.  BODYFIT_BWD_FILL=1 enables it.
        static int fill_env = -1;
        if (fill_env < 0) { const char* e = getenv("BODYFIT_BWD_FILL"); fill_env = e ? atoi(e) : 0; }
        if (!fill_env) S_fill = 0;
        if (S_fill > S && f->ws && (size_t)f->ws_floats >= (size_t)S_fill * stride) {
            cps = (num_k + S_fill - 1) / S_fill;
            S = (num_k + cps - 1) / cps;
        }
    }
    dim3 grid(m->Kp / BN, (f->B + TC_BM - 1) / TC_BM, S);
    // block mask of the active set (BfFrames.blk_mask, buffer of this iteration's parity): single-run reductions only
    const uint32_t* mask = (bf_blk_mask_on() && f->blk_mask && vs->lv_blk && S == 1 && TC_BK == 16 && vs->n_pad <= 512 && num_k % 3 == 0)
                               ? f->blk_mask + (size_t)(f->iter & 1) * ((f->B + 127) / 128) : nullptr;
    // two half-reductions per tile (bf_bwd_two_cta above): by two CTAs into dpf / dpf2, or fused in one CTA
    float* out0 = S > 1 ? f->ws : f->dpf;
    size_t out_stride = stride;
    int fuse = 0;
    if (mask && bf_bwd_two_cta(m, f)) { grid.z = 2; out0 = f->dpf; out_stride = (size_t)(f->dpf2 - f->dpf); }
    else if (mask) fuse = 1;
    if (NS == 2) k_blend_bwd_tc<2><<<grid, 192, smem, s>>>(a_hi, a_lo, b_hi, b_lo, BN, num_k, cps, m->Kp, out0, out_stride, f->B, mask, fuse);
    else if (NS == 8) k_blend_bwd_tc<8><<<grid, 192, smem, s>>>(a_hi, a_lo, b_hi, b_lo, BN, num_k, cps, m->Kp, out0, out_stride, f->B, mask, fuse);
    else k_blend_bwd_tc<TC_STAGES><<<grid, 192, smem, s>>>(a_hi, a_lo, b_hi, b_lo, BN, num_k, cps, m->Kp, out0, out_stride, f->B, mask, fuse);
    BF_LAUNCH_CHECK();
    if (S > 1) {
        const size_t n = stride;
        k_sum_partials<<<(unsigned)((n / 4 + 255) / 256), 256, 0, s>>>(f->ws, f->dpf, n, S);
        BF_LAUNCH_CHECK();
    }
    return BF_OK;
}
