// genrec_b200 - Blackwell-native GEMM: TMA (cp.async.bulk.tensor, 128B swizzle) -> shared memory -> tcgen05.mma
// (single-thread issue, fp32 accumulators in TMEM, double-buffered) -> tcgen05.ld epilogue with fused element-wise work.
//
//   C[M,N] (+)= opA(A) * opB(B)          bf16 operands, fp32 accumulate
//     A_MN = 0 : A stored [M][K] (K contiguous)        A_MN = 1 : A stored [K][M] (M contiguous)
//     B_MN = 0 : B stored [N][K] (K contiguous)        B_MN = 1 : B stored [K][N] (N contiguous)
//   Both majors map straight onto UMMA shared-memory descriptors (K-major / MN-major canonical SWIZZLE_128B layouts),
//   so no operand is ever transposed in memory.
//
// Persistent kernel, one CTA per SM, 320 threads:
//   warp 0    : TMA producer (one elected lane)      - ring of TC_STAGES x (A 16 KB + B 16 KB)
//   warp 1    : TMEM allocator + MMA issuer (one lane): 4 x tcgen05.mma (K = 16 each) per 64-wide k-block
//   warps 2-9 : epilogue; warp w owns TMEM lanes 32*(w%4)..+31 = 32 rows of the 128 x 128 tile and, by (w-2)/4, one
//               64-column half of it (two warps per TMEM sub-partition so the element-wise work has 8 warps to run on)
// Work item = (m tile, n tile, k split).  Split-K partial sums go out through an atomic epilogue.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace grb {

constexpr int TC_EPI_WARPS = 8;    // 2 per TMEM sub-partition: each converts 4 / (TC_EPI_WARPS / 4) 32-column chunks of the tile
constexpr int TC_EPI_CPW = 4 / (TC_EPI_WARPS / 4);   // chunks per warp (16 warps measured slower here: register spills)
static_assert(TC_EPI_CPW == 2, "a warp's 2 x 32 columns are one 64-column bf16 store box");
constexpr int TC_BM = 128, TC_BN = 128, TC_BK = 64, TC_STAGES = 3, TC_THREADS = 64 + 32 * TC_EPI_WARPS;  // TMA, MMA, epilogue warps
constexpr int TC_TILE_BYTES = TC_BM * TC_BK * 2;  // 16 KB per operand per stage
constexpr int TC_STAGE_OUT_BYTES = 64 * 1024;   // epilogue staging: 2 x bf16 [128x128] or 1 x fp32 [128x128], 128B-swizzled boxes
constexpr int TC_SMEM_BYTES = 2 * TC_STAGES * TC_TILE_BYTES + 2 * TC_STAGE_OUT_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int TC_TMEM_COLS = 2 * TC_BN;           // two accumulators

// ------------------------------------------------------------------------------------------------ PTX wrappers
GRB_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
GRB_DEVINL void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
GRB_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
GRB_DEVINL void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
GRB_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
GRB_DEVINL void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// shared -> global tile store (bulk async group); rows/cols outside the tensor map's extents are clipped by the hardware
GRB_DEVINL void tma_store_2d(const CUtensorMap* tmap, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
GRB_DEVINL void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
GRB_DEVINL void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
GRB_DEVINL void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
GRB_DEVINL void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
GRB_DEVINL void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_EPI_WARPS) : "memory"); }   // the epilogue warps only
GRB_DEVINL void tma_prefetch_desc(const CUtensorMap* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
GRB_DEVINL void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
GRB_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
GRB_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
GRB_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc]
GRB_DEVINL void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once every tcgen05.mma issued so far by this thread has completed
GRB_DEVINL void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
GRB_DEVINL void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,"
        "%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor, SWIZZLE_128B, sm_100 (version = 1).  Tile base must be 1024-byte aligned; `byte_off`
// selects the k-slice inside it.   K-major : rows of 128 B (64 bf16 along K), 8-row groups SBO = 1024 B apart.
//                                  MN-major: k-rows of 128 B (64 bf16 along MN), 8-k groups SBO = 1024 B apart, the next
//                                            64-wide MN block LBO bytes away.
GRB_DEVINL uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;  // SWIZZLE_128B
    return d;
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> f32
GRB_DEVINL constexpr uint32_t umma_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

struct TcGemmShape {
    int M, N, K;
    int num_m, num_n, splits;
    int kblocks_total, kblocks_per_split;
};

// Epilogue concept:
//   static constexpr int kOut;   0: the functor stores by itself (atomics / odd strides)      signature (row, col0, v, nvalid)
//                                1: one bf16 output tile   2: two bf16 output tiles   3: one fp32 output tile
//                                   -> signature (row, col0, v /*in: acc, out: primary*/, w /*out: secondary*/, nvalid); the kernel
//                                      stages the tile in shared memory (128B swizzle) and writes it with TMA stores (tmC0 / tmC1).
//   void prepare();
template <int A_MN, int B_MN, class Epi>
__global__ void __launch_bounds__(TC_THREADS, 1)
    tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC0,
                   const __grid_constant__ CUtensorMap tmC1, TcGemmShape sh, Epi epi) {
    extern __shared__ unsigned char tc_smem_raw[];
    // 1024-byte aligned operand ring, then barriers
    unsigned char* base = tc_smem_raw + ((1024u - (smem_u32(tc_smem_raw) & 1023u)) & 1023u)   /* offset from the __shared__ array: keeps the shared address space (LDS / STS) */;
    unsigned char* sA = base;
    unsigned char* sB = base + TC_STAGES * TC_TILE_BYTES;
    unsigned char* sOut0 = base + 2 * TC_STAGES * TC_TILE_BYTES;  // 2 x 64 KB staging (double-buffered), 1024-aligned
    uint64_t* bars = reinterpret_cast<uint64_t*>(sOut0 + 2 * TC_STAGE_OUT_BYTES);
    uint64_t* full_bar = bars;                       // [TC_STAGES]  TMA -> MMA
    uint64_t* empty_bar = bars + TC_STAGES;          // [TC_STAGES]  MMA -> TMA
    uint64_t* tfull_bar = bars + 2 * TC_STAGES;      // [2]          MMA -> epilogue
    uint64_t* tempty_bar = bars + 2 * TC_STAGES + 2; // [2]          epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_STAGES + 4);
    uint64_t* zfull_bar = bars + 2 * TC_STAGES + 5;  // [2]          TMA -> epilogue (auxiliary operand tile, Epi::kAux)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    epi.prepare();

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < TC_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], TC_EPI_WARPS);  // one arrive per epilogue warp
            mbar_init(&zfull_bar[a], 1);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TC_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();  // prologue above overlaps the previous kernel's tail

    const int num_work = sh.num_m * sh.num_n * sh.splits;

    if (warp == 0) {
        // ===================================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
                const int split = w % sh.splits;
                const int tile = w / sh.splits;
                const int m0 = (tile / sh.num_n) * TC_BM, n0 = (tile % sh.num_n) * TC_BN;
                const int kb0 = split * sh.kblocks_per_split;
                const int kb1 = min(sh.kblocks_total, kb0 + sh.kblocks_per_split);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_expect_tx(&full_bar[stage], 2 * TC_TILE_BYTES);
                    unsigned char* a_dst = sA + stage * TC_TILE_BYTES;
                    unsigned char* b_dst = sB + stage * TC_TILE_BYTES;
                    const int k0 = kb * TC_BK;
                    if (A_MN == 0) {
                        tma_load_2d(a_dst, &tmA, k0, m0, &full_bar[stage]);            // box {64 k, 128 rows}
                    } else {
                        tma_load_2d(a_dst, &tmA, m0, k0, &full_bar[stage]);            // box {64 m, 64 k-rows}
                        tma_load_2d(a_dst + TC_TILE_BYTES / 2, &tmA, m0 + 64, k0, &full_bar[stage]);
                    }
                    if (B_MN == 0) {
                        tma_load_2d(b_dst, &tmB, k0, n0, &full_bar[stage]);
                    } else {
                        tma_load_2d(b_dst, &tmB, n0, k0, &full_bar[stage]);
                        tma_load_2d(b_dst + TC_TILE_BYTES / 2, &tmB, n0 + 64, k0, &full_bar[stage]);
                    }
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
                if constexpr (Epi::kAux) {
                    // auxiliary element-wise operand of this tile -> the unused half of the tile's staging buffer, as soon as
                    // the epilogue that last used that buffer (two tiles ago) has drained it
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                    unsigned char* z_dst = sOut0 + acc * TC_STAGE_OUT_BYTES + 32768;
                    mbar_expect_tx(&zfull_bar[acc], 32768);
                    tma_load_2d(z_dst, &tmC1, n0, m0, &zfull_bar[acc]);                  // box {64 cols, 128 rows}
                    tma_load_2d(z_dst + 16384, &tmC1, n0 + 64, m0, &zfull_bar[acc]);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================================== MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc(TC_BM, TC_BN, A_MN, B_MN);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
                const int split = w % sh.splits;
                const int kb0 = split * sh.kblocks_per_split;
                const int kb1 = min(sh.kblocks_total, kb0 + sh.kblocks_per_split);
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * TC_BN;
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(sA + stage * TC_TILE_BYTES);
                    const uint32_t b_addr = smem_u32(sB + stage * TC_TILE_BYTES);
#pragma unroll
                    for (int k = 0; k < TC_BK / 16; ++k) {
                        // K-major: +32 B per 16-wide k-slice inside the 128 B swizzle row ; MN-major: +16 k-rows = 2048 B
                        const uint64_t ad = A_MN == 0 ? umma_desc(a_addr + k * 32, 16, 1024) : umma_desc(a_addr + k * 2048, TC_TILE_BYTES / 2, 1024);
                        const uint64_t bd = B_MN == 0 ? umma_desc(b_addr + k * 32, 16, 1024) : umma_desc(b_addr + k * 2048, TC_TILE_BYTES / 2, 1024);
                        umma_bf16(d_tmem, ad, bd, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                    }
                    umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tfull_bar[acc]);        // accumulator complete
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================================================================== epilogue (warps 2..9)
        const int sub = warp & 3;         // TMEM sub-partition this warp may access: lanes 32*sub .. 32*sub+31
        const int cq = (warp - 2) >> 2;     // which 32-column chunk of the tile this warp converts
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
            const int tile = w / sh.splits;
            const int m0 = (tile / sh.num_n) * TC_BM, n0 = (tile % sh.num_n) * TC_BN;
            const int r = sub * 32 + lane;  // row inside the tile == TMEM lane
            const int row = m0 + r;
            // operands of the fused element-wise work that do not depend on the MMA (residual rows, saved pre-activations)
            // are fetched BEFORE waiting for the accumulator, so their latency hides behind the tensor-core work
            float pre[Epi::kPre ? TC_EPI_CPW : 1][Epi::kPre ? 32 : 1];
            if constexpr (Epi::kPre) {
#pragma unroll
                for (int ci = 0; ci < TC_EPI_CPW; ++ci) {
                    const int col0 = n0 + (cq * TC_EPI_CPW + ci) * 32;
                    const int nvalid = min(32, sh.N - col0);
                    if (row < sh.M && nvalid > 0) epi.preload(row, col0, nvalid, pre[ci]);
                }
            }
            if constexpr (Epi::kOut != 0) {
                if (lane == 0) tma_store_wait_read1();   // this warp's store from two tiles ago has finished reading its staging piece
                __syncwarp();
            }
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            unsigned char* sOut = sOut0 + acc * TC_STAGE_OUT_BYTES;  // staging buffer alternates with the accumulator
            if constexpr (Epi::kAux) mbar_wait(&zfull_bar[acc], acc_phase);
#pragma unroll
            for (int ci = 0; ci < TC_EPI_CPW; ++ci) {
                const int c = cq * TC_EPI_CPW + ci;
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(acc * TC_BN + c * 32), v);
                const int col0 = n0 + c * 32;
                const int nvalid = min(32, sh.N - col0);
                if constexpr (Epi::kOut == 0) {
                    if (row < sh.M && nvalid > 0) epi(row, col0, v, nvalid);
                } else {
                    float w[32];
                    if constexpr (Epi::kAux) {
                        // this thread's 32 bf16 of the auxiliary tile (same 128B-swizzled box layout as the bf16 staging tile)
                        float zz[32];
                        const unsigned char* zsrc = sOut + 32768 + (c >> 1) * 16384 + r * 128;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint4 u = *reinterpret_cast<const uint4*>(zsrc + ((((c & 1) * 4 + j) ^ (r & 7)) << 4));
                            const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
                            zz[8 * j] = f0.x; zz[8 * j + 1] = f0.y; zz[8 * j + 2] = f1.x; zz[8 * j + 3] = f1.y;
                            zz[8 * j + 4] = f2.x; zz[8 * j + 5] = f2.y; zz[8 * j + 6] = f3.x; zz[8 * j + 7] = f3.y;
                        }
                        if (row < sh.M && nvalid > 0) epi(row, col0, v, w, nvalid, zz);
                    } else if constexpr (Epi::kPre) {
                        if (row < sh.M && nvalid > 0) epi(row, col0, v, w, nvalid, pre[ci]);
                    } else {
                        if (row < sh.M && nvalid > 0) epi(row, col0, v, w, nvalid);
                    }
                    if constexpr (Epi::kOut == 3) {
                        // fp32: box c = [128 rows][32 cols] = 128 B rows, 16-byte chunk j stored at (j ^ (r & 7))
                        unsigned char* dst = sOut + c * 16384 + r * 128;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            *reinterpret_cast<float4*>(dst + ((j ^ (r & 7)) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    } else {
                        // bf16: box h = [128 rows][64 cols]; this 32-column chunk covers 16-byte chunks (c&1)*4 .. +3 of box c>>1
                        unsigned char* dst = sOut + (c >> 1) * 16384 + r * 128;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            uint4 u;
                            u.x = pack_bf16(v[8 * j], v[8 * j + 1]); u.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
                            u.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]); u.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
                            *reinterpret_cast<uint4*>(dst + ((((c & 1) * 4 + j) ^ (r & 7)) << 4)) = u;
                        }
                        if constexpr (Epi::kOut == 2) {
                            unsigned char* dst1 = dst + 32768;
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                uint4 u;
                                u.x = pack_bf16(w[8 * j], w[8 * j + 1]); u.y = pack_bf16(w[8 * j + 2], w[8 * j + 3]);
                                u.z = pack_bf16(w[8 * j + 4], w[8 * j + 5]); u.w = pack_bf16(w[8 * j + 6], w[8 * j + 7]);
                                *reinterpret_cast<uint4*>(dst1 + ((((c & 1) * 4 + j) ^ (r & 7)) << 4)) = u;
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);   // accumulator drained: the MMA warp may start the next-but-one tile
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            if constexpr (Epi::kOut != 0) {
                // Every epilogue warp owns rows 32*sub .. +31 of the 64-column (bf16) / 2 x 32-column (fp32) slab cq of the staging
                // tile - a contiguous, swizzle-aligned 4 KB piece of each 128-row box - and stores it with its OWN bulk store (tensor-map
                // box = 32 rows): no CTA-wide barrier per tile, the warps drift apart freely.  Buffer reuse is guarded per warp by
                // `wait_group.read 1` at the top of the tile (the piece written two tiles ago has been read).
                fence_proxy_async();   // generic-proxy smem writes -> visible to the TMA (async proxy)
                __syncwarp();
                if (lane == 0 && m0 + sub * 32 < sh.M) {
                    if constexpr (Epi::kOut == 3) {
#pragma unroll
                        for (int ci = 0; ci < TC_EPI_CPW; ++ci) {
                            const int c = cq * TC_EPI_CPW + ci;
                            if (n0 + c * 32 < sh.N) tma_store_2d(&tmC0, sOut + c * 16384 + sub * 4096, n0 + c * 32, m0 + sub * 32);
                        }
                    } else {
                        if (n0 + cq * 64 < sh.N) {
                            tma_store_2d(&tmC0, sOut + cq * 16384 + sub * 4096, n0 + cq * 64, m0 + sub * 32);
                            if constexpr (Epi::kOut == 2) tma_store_2d(&tmC1, sOut + 32768 + cq * 16384 + sub * 4096, n0 + cq * 64, m0 + sub * 32);
                        }
                    }
                }
                if (lane == 0) tma_store_commit();
            }
        }
        if (Epi::kOut != 0 && lane == 0) tma_store_wait_read();  // smem must outlive this warp's last bulk stores
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TC_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------ row-chunk epilogues
GRB_DEVINL void store_bf16x32(bf16* dst, const float (&v)[32], int nvalid) {
    if (nvalid == 32 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            uint4 u;
            u.x = pack_bf16(v[8 * i], v[8 * i + 1]);
            u.y = pack_bf16(v[8 * i + 2], v[8 * i + 3]);
            u.z = pack_bf16(v[8 * i + 4], v[8 * i + 5]);
            u.w = pack_bf16(v[8 * i + 6], v[8 * i + 7]);
            reinterpret_cast<uint4*>(dst)[i] = u;
        }
    } else {
        for (int i = 0; i < nvalid; ++i) dst[i] = __float2bfloat16(v[i]);
    }
}
GRB_DEVINL void store_f32x32(float* dst, const float (&v)[32], int nvalid) {
    if (nvalid == 32 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) reinterpret_cast<float4*>(dst)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else {
        for (int i = 0; i < nvalid; ++i) dst[i] = v[i];
    }
}
GRB_DEVINL void load_bf16x32(const bf16* src, float (&v)[32], int nvalid) {
    if (nvalid == 32 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            uint4 u = reinterpret_cast<const uint4*>(src)[i];
            float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
            v[8 * i] = a.x; v[8 * i + 1] = a.y; v[8 * i + 2] = b.x; v[8 * i + 3] = b.y;
            v[8 * i + 4] = c.x; v[8 * i + 5] = c.y; v[8 * i + 6] = d.x; v[8 * i + 7] = d.y;
        }
    } else {
        for (int i = 0; i < 32; ++i) v[i] = i < nvalid ? __bfloat162float(src[i]) : 0.f;
    }
}
GRB_DEVINL void load_f32x32(const float* src, float (&v)[32], int nvalid) {
    if (nvalid == 32 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 f = reinterpret_cast<const float4*>(src)[i];
            v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
        }
    } else {
        for (int i = 0; i < 32; ++i) v[i] = i < nvalid ? src[i] : 0.f;
    }
}

// z = acc + bias -> bf16 ; act = dropout(ACT(z_rounded)) -> bf16      ACT 0: none (act_out unused), 1: silu, 2: relu
template <int ACT>
struct TcEpiBiasAct {
    static constexpr int kOut = ACT == 0 ? 1 : 2;   // tmC0 = z, tmC1 = act
    static constexpr bool kPre = false;
    static constexpr bool kAux = false;
    const float* bias;
    int ld;
    Dropout drop;
    GRB_DEVINL void prepare() { drop.resolve(); }
    GRB_DEVINL void operator()(int row, int col0, float (&v)[32], float (&w)[32], int nvalid) const {
        float bb[32];
        load_f32x32(bias + col0, bb, nvalid);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            float zz = v[i] + bb[i];
            v[i] = zz;
            if (ACT != 0) {
                float zr = bf16_round(zz);
                w[i] = ACT == 1 ? siluf(zr) : fmaxf(zr, 0.f);
            }
        }
        if (ACT != 0) {
#pragma unroll
            for (int i = 0; i < 32; i += 2) drop.apply2p(w[i], w[i + 1], row, (col0 >> 1) + (i >> 1));
        }
    }
};
// y = res + dropout(acc + bias) (* row_scale) -> fp32
struct TcEpiBiasResidual {
    static constexpr int kOut = 3;
    static constexpr bool kPre = true;
    static constexpr bool kAux = false;
    const float* bias;
    const float* res;
    const float* row_scale;
    int ld;
    Dropout drop;
    GRB_DEVINL void prepare() { drop.resolve(); }
    GRB_DEVINL void preload(int row, int col0, int nvalid, float (&r)[32]) const { load_f32x32(res + (size_t)row * ld + col0, r, nvalid); }
    GRB_DEVINL void operator()(int row, int col0, float (&v)[32], float (&)[32], int nvalid, const float (&r)[32]) const {
        const float s = row_scale ? row_scale[row] : 1.f;
        float bb[32];
        load_f32x32(bias + col0, bb, nvalid);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            float y0 = v[i] + bb[i], y1 = v[i + 1] + bb[i + 1];
            drop.apply2p(y0, y1, row, (col0 >> 1) + (i >> 1));
            v[i] = (r[i] + y0) * s;
            v[i + 1] = (r[i + 1] + y1) * s;
        }
    }
};
// g = dropmask(acc) * ACT'(z) -> bf16
template <int ACT>
struct TcEpiDAct {
    static constexpr int kOut = 1;
    static constexpr bool kPre = false;
    static constexpr bool kAux = true;   // the saved pre-activation tile z[128 x 128] arrives by TMA (tensor map in the kernel's tmC1 slot)
    const bf16* z;
    int ld;
    Dropout drop;
    GRB_DEVINL void prepare() { drop.resolve(); }
    GRB_DEVINL void operator()(int row, int col0, float (&v)[32], float (&)[32], int nvalid, const float (&zz)[32]) const {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            drop.apply2p(v[i], v[i + 1], row, (col0 >> 1) + (i >> 1));
            v[i] *= ACT == 1 ? dsiluf(zz[i]) : (zz[i] > 0.f ? 1.f : 0.f);
            v[i + 1] *= ACT == 1 ? dsiluf(zz[i + 1]) : (zz[i + 1] > 0.f ? 1.f : 0.f);
        }
    }
};
// out = scale * acc (+ res) -> fp32
struct TcEpiF32 {
    static constexpr int kOut = 3;
    static constexpr bool kPre = true;
    static constexpr bool kAux = false;
    const float* res;
    int ld;
    float scale;
    GRB_DEVINL void prepare() {}
    GRB_DEVINL void preload(int row, int col0, int nvalid, float (&y)[32]) const {
        if (res) load_f32x32(res + (size_t)row * ld + col0, y, nvalid);
    }
    GRB_DEVINL void operator()(int row, int col0, float (&v)[32], float (&)[32], int nvalid, const float (&y)[32]) const {
        if (res) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = y[i] + v[i] * scale;
        } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] *= scale;
        }
    }
};
// exp(x) to ~1 ulp with FMA-pipe arithmetic only (the library is compiled with --use_fast_math, which would turn expf into the
// 2^-21-accurate ex2.approx path): Cody-Waite reduction x = n ln2 + r, |r| <= ln2 / 2, degree-6 polynomial, scale by 2^n.
GRB_DEVINL float exp_accurate(float x) {
    x = fminf(fmaxf(x, -87.f), 88.f);
    const float n = rintf(x * 1.44269504088896341f);
    float r = __fmaf_rn(n, -0.693145751953125f, x);            // ln2 high part (exact product for |n| < 2^10)
    r = __fmaf_rn(n, -1.42860682030941723e-6f, r);             // ln2 low part
    float p = 1.f / 720.f;
    p = __fmaf_rn(p, r, 1.f / 120.f);
    p = __fmaf_rn(p, r, 1.f / 24.f);
    p = __fmaf_rn(p, r, 1.f / 6.f);
    p = __fmaf_rn(p, r, 0.5f);
    p = __fmaf_rn(p, r, 1.f);
    p = __fmaf_rn(p, r, 1.f);
    return p * __int_as_float(((int)n + 127) << 23);
}
// out = ACT(res + acc + bias) + res2 -> fp32 : second pass of the split-bf16 GEMM (res = the sum of the five small cross terms;
// bias [N] and res2 [M, ld] nullable: the linear layers and the residual connection of the fp32-exact HSTU block)
template <int ACT>
struct TcEpiActResF32 {
    static constexpr int kOut = 3;
    static constexpr bool kPre = true;
    static constexpr bool kAux = false;
    const float* res;
    int ld;
    const float* bias;
    const float* res2;
    GRB_DEVINL void prepare() {}
    GRB_DEVINL void preload(int row, int col0, int nvalid, float (&y)[32]) const { load_f32x32(res + (size_t)row * ld + col0, y, nvalid); }
    GRB_DEVINL void operator()(int row, int col0, float (&v)[32], float (&)[32], int nvalid, const float (&y)[32]) const {
        float bb[32], rr[32];
        if (bias) load_f32x32(bias + col0, bb, nvalid);
        if (res2) load_f32x32(res2 + (size_t)row * ld + col0, rr, nvalid);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            float z = v[i] + y[i];
            if (bias) z += bb[i];
            z = ACT == 1 ? __fdiv_rn(z, 1.f + exp_accurate(-z)) : z;
            v[i] = res2 ? z + rr[i] : z;
        }
    }
};
// out += scale * acc (split-K partial sums, weight gradients)
struct TcEpiAtomicF32 {
    static constexpr int kOut = 0;
    static constexpr bool kPre = false;
    static constexpr bool kAux = false;
    float* out;
    int ld;
    float scale;
    GRB_DEVINL void prepare() {}
    GRB_DEVINL void operator()(int row, int col0, const float (&v)[32], int nvalid) const {
        float* dst = out + (size_t)row * ld + col0;
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if (i < nvalid) atomicAdd(dst + i, v[i] * scale);
    }
};
// plain fp32 store, arbitrary leading dimension
struct TcEpiF32Plain {
    static constexpr int kOut = 0;
    static constexpr bool kPre = false;
    static constexpr bool kAux = false;
    float* out;
    int ld;
    GRB_DEVINL void prepare() {}
    GRB_DEVINL void operator()(int row, int col0, const float (&v)[32], int nvalid) const {
        store_f32x32(out + (size_t)row * ld + col0, v, nvalid);
    }
};

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_tmapEncodeTiled tmap_encoder() {
    static PFN_tmapEncodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
    }
    return fn;
}

// 2-D row-major tensor [rows][cols] with leading dimension ld (elements); box = {box_cols (inner, 128 bytes), box_rows}
inline bool make_tmap(CUtensorMap* m, const void* base, bool fp32, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols, uint32_t box_rows) {
    PFN_tmapEncodeTiled enc = tmap_encoder();
    if (!enc) return false;
    const uint64_t esz = fp32 ? 4 : 2;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || ((ld * esz) & 15)) return false;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * esz};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    return enc(m, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
inline bool make_tmap_bf16(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols, uint32_t box_rows) {
    return make_tmap(m, base, false, rows, cols, ld, box_cols, box_rows);
}

// A: A_MN == 0 -> [M][K] ld=lda ; A_MN == 1 -> [K][M] ld=lda.   Same for B with N.
// out0 / out1: output tensors [M][N] with leading dimension ldo (bf16 for kOut 1/2, fp32 for kOut 3); unused for kOut 0.
template <int A_MN, int B_MN, class Epi>
inline cudaError_t launch_tc_gemm(const bf16* A, const bf16* B, int M, int N, int K, int lda, int ldb, int splits, const Epi& epi,
                                  void* out0, void* out1, int ldo, int num_sms, cudaStream_t st) {
    CUtensorMap tmA, tmB, tmC0, tmC1;
    bool ok = A_MN == 0 ? make_tmap_bf16(&tmA, A, M, K, lda, TC_BK, TC_BM) : make_tmap_bf16(&tmA, A, K, M, lda, 64, TC_BK);
    ok = ok && (B_MN == 0 ? make_tmap_bf16(&tmB, B, N, K, ldb, TC_BK, TC_BN) : make_tmap_bf16(&tmB, B, K, N, ldb, 64, TC_BK));
    if (Epi::kOut == 0) {
        tmC0 = tmA; tmC1 = tmA;
    } else if (Epi::kOut == 3) {
        ok = ok && make_tmap(&tmC0, out0, true, M, N, ldo, 32, 32);     // store boxes: 32 rows, one per epilogue warp
        tmC1 = tmC0;
    } else {
        ok = ok && make_tmap(&tmC0, out0, false, M, N, ldo, 64, 32);
        if (Epi::kOut == 2) ok = ok && make_tmap(&tmC1, out1, false, M, N, ldo, 64, 32);
        else tmC1 = tmC0;
    }
    if constexpr (Epi::kAux) {
        static_assert(Epi::kOut == 1, "the auxiliary tile lives in the half of the staging buffer a single bf16 output leaves free");
        ok = ok && make_tmap(&tmC1, epi.z, false, M, N, epi.ld, 64, TC_BM);
    }
    if (!ok) return cudaErrorInvalidValue;
    TcGemmShape sh;
    sh.M = M; sh.N = N; sh.K = K;
    sh.num_m = (M + TC_BM - 1) / TC_BM;
    sh.num_n = (N + TC_BN - 1) / TC_BN;
    sh.kblocks_total = (K + TC_BK - 1) / TC_BK;
    if (splits < 1) splits = 1;
    if (splits > sh.kblocks_total) splits = sh.kblocks_total;
    sh.kblocks_per_split = (sh.kblocks_total + splits - 1) / splits;
    sh.splits = (sh.kblocks_total + sh.kblocks_per_split - 1) / sh.kblocks_per_split;
    auto kern = tc_gemm_kernel<A_MN, B_MN, Epi>;
    static bool attr_set_dev[64] = {false};
    int attr_dev = 0;
    cudaGetDevice(&attr_dev);
    bool& attr_set = attr_set_dev[attr_dev & 63];   // the attribute is per device
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    int work = sh.num_m * sh.num_n * sh.splits;
    int grid = work < num_sms ? work : num_sms;
    launch_k(kern, grid, TC_THREADS, TC_SMEM_BYTES, st, tmA, tmB, tmC0, tmC1, sh, epi);
    return cudaGetLastError();
}

}  // namespace grb
