// bd_gemm.cu -- strict band depth as an int8 violation Gram on the 5th-gen tensor cores.
//
// North-star formulation of K2 (SURVEY 8a row a3): for query curve q
//     M[c][k] in {0,1},  k = (time, below|above):  M[c][t,0] = [X[t,c] < X[t,q]],  M[c][t,1] = [X[t,c] > X[t,q]]
//     V = M M^T  (int8 x int8 -> int32),   pair (c1 < c2) contains q at all T points  <=>  V[c1,c2] == 0
// which replaces the strict branch of _r2_containment (_containment.py:68-80) over all pairs
// (_functional.py:238-253) by a dense contraction with K = 2T.
//
// Kernels
//   bd_mask8_kernel : fp64 compares -> int8 operand tiles written to HBM ALREADY in the UMMA
//                     canonical K-major / no-swizzle ("interleaved") shared-memory layout:
//                     tile(row block, k stage) = [8 k-chunks][128 rows][16 bytes], 16 KB contiguous,
//                     one stage = 64 time points = 64 "below" bytes | 64 "above" bytes per row.
//   bd_gram_kernel  : warp-specialised, persistent over the upper-triangular tile pairs of one query:
//                       warp 0   producer: 1-D TMA bulk copies (cp.async.bulk, 2 x 16 KB per stage,
//                                mbarrier complete_tx) -- tiles are contiguous, so no tensor map
//                       warp 1   TMEM allocator + single-thread tcgen05.mma.cta_group::1.kind::i8
//                                (M = N = 128, K = 32 per instruction, accumulator 128 lanes x 128
//                                columns of TMEM), tcgen05.commit to free smem stages / publish the tile
//                       warps 2-5 epilogue: tcgen05.ld 32x32b.x32 -> count zero entries of the strict
//                                upper triangle (c1 < c2, both != q, both < n)
// Selection: SD_OPT_BD_IMPL.  SD_BD_AUTO keeps the bit-mask kernel (bd_bits.cu), which retires ~99 % of
// pairs after one 32-bit AND; the dense Gram does 2*(2T)*C(n-1,2) int8 ops per query regardless of the
// data.  Measured comparison: profiles/README.md.
#include "common.cuh"

namespace sd {

constexpr int GM_TILE = 128;                        // rows per operand tile; UMMA M = N = 128
constexpr int GM_TSTEP = 64;                        // time points per k stage
constexpr int GM_KSTAGE = 2 * GM_TSTEP;             // K bytes per stage
constexpr int GM_TILE_BYTES = GM_TILE * GM_KSTAGE;  // 16 KB
constexpr int GM_STAGES = 3;                        // 3 x 32 KB of shared memory -> 2 CTAs per SM
constexpr int GM_THREADS = 192;
constexpr u32 GM_TMEM_COLS = 256;                   // two 128-column accumulators: MMA of tile i+1 overlaps epilogue of tile i
constexpr u32 GM_CHUNK_PLANE = GM_TILE * 16;        // bytes of one k-chunk plane: 128 rows x 16 B = 2048

// ---------------------------------------------------------------------------------------------
// operand generation
// ---------------------------------------------------------------------------------------------
// grid (row blocks, 2 * k stages, ceil(queries / GM_MQ)), 128 threads = 128 rows.  One CTA builds half a
// stage (32 time points -> 2 "below" + 2 "above" 16-byte chunks per row) for GM_MQ queries, so X is read
// once per GM_MQ queries.
constexpr int GM_MQ = 4;

__global__ void __launch_bounds__(GM_TILE) bd_mask8_kernel(const double *__restrict__ X, const i64 T, const i64 n,
                                                           const i64 ld, const i64 *__restrict__ qidx, const int nqb,
                                                           const int NB, const int KS, uint8_t *__restrict__ M8,
                                                           int *__restrict__ status) {
    __shared__ double sq[32][GM_MQ];
    const int rb = blockIdx.x, ks = blockIdx.y >> 1, half = blockIdx.y & 1, q0 = blockIdx.z * GM_MQ;
    const i64 t0 = (i64)ks * GM_TSTEP + half * 32;
    {
        const int tt = threadIdx.x / GM_MQ, qq = threadIdx.x % GM_MQ;  // 128 threads = 32 x 4
        const i64 t = t0 + tt;
        sq[tt][qq] = (t < T && q0 + qq < nqb) ? X[t * ld + qidx[q0 + qq]] : 0.0;
    }
    __syncthreads();
    const i64 c = (i64)rb * GM_TILE + threadIdx.x;
    u32 below[GM_MQ][8], above[GM_MQ][8];  // 32 bytes each per query
#pragma unroll
    for (int qq = 0; qq < GM_MQ; ++qq)
#pragma unroll
        for (int w = 0; w < 8; ++w) below[qq][w] = above[qq][w] = 0u;
    bool bad = false;
    if (c < n) {
#pragma unroll
        for (int tt = 0; tt < 32; ++tt) {
            const i64 t = t0 + tt;
            if (t < T) {
                const double x = X[t * ld + c];
                bad |= !isfinite(x);
#pragma unroll
                for (int qq = 0; qq < GM_MQ; ++qq) {
                    const double xq = sq[tt][qq];
                    below[qq][tt >> 2] |= (u32)(x < xq) << ((tt & 3) * 8);
                    above[qq][tt >> 2] |= (u32)(x > xq) << ((tt & 3) * 8);
                }
            }
        }
    }
    if (bad) atomicOr(status, ST_NONFINITE);
#pragma unroll
    for (int qq = 0; qq < GM_MQ; ++qq) {
        if (q0 + qq >= nqb) break;
        uint8_t *tile = M8 + (((i64)(q0 + qq) * NB + rb) * KS + ks) * GM_TILE_BYTES;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
            *reinterpret_cast<uint4 *>(tile + (size_t)(2 * half + ch) * GM_CHUNK_PLANE + threadIdx.x * 16) =
                make_uint4(below[qq][4 * ch], below[qq][4 * ch + 1], below[qq][4 * ch + 2], below[qq][4 * ch + 3]);
            *reinterpret_cast<uint4 *>(tile + (size_t)(4 + 2 * half + ch) * GM_CHUNK_PLANE + threadIdx.x * 16) =
                make_uint4(above[qq][4 * ch], above[qq][4 * ch + 1], above[qq][4 * ch + 2], above[qq][4 * ch + 3]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(u64 *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
    const u32 addr = smem_u32(bar);
    u32 done = 0;
    while (!done) {
        asm volatile(
            "{\n\t"
            ".reg .pred P1;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
            "selp.b32 %0, 1, 0, P1;\n\t"
            "}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, u32 bytes, u64 *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(u64 *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], int8 operands, int32 accumulate
__device__ __forceinline__ void tc_mma_i8(u32 tmem_d, u64 desc_a, u64 desc_b, u32 idesc, u32 accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void tc_ld_32x32(u32 taddr, u32 (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE ("interleaved" canonical layout, in 16-byte
// units ((8,n),2):((1,SBO),LBO)): core matrix = 8 rows x 16 B contiguous (128 B); SBO = distance
// between 8-row groups = 128 B; LBO = distance between the two 16-byte k halves = one chunk plane.
__device__ __forceinline__ u64 umma_desc(u32 saddr) {
    u64 d = 0;
    d |= (u64)((saddr >> 4) & 0x3fffu);                 // start address  [0,14)
    d |= (u64)((GM_CHUNK_PLANE >> 4) & 0x3fffu) << 16;  // leading byte offset [16,30)
    d |= (u64)((128u >> 4) & 0x3fffu) << 32;            // stride byte offset  [32,46)
    d |= (u64)1 << 46;                                  // descriptor version 1 (sm_100)
    return d;                                           // base_offset 0, lbo_mode 0, layout_type 0 (no swizzle)
}

// instruction descriptor for kind::i8: D = S32, A = B = unsigned 8-bit, both K-major, N = 128, M = 128
constexpr u32 GM_IDESC = (2u << 4) | (0u << 7) | (0u << 10) | ((u32)(GM_TILE >> 3) << 17) | ((u32)(GM_TILE >> 4) << 24);

// tile pair p of the upper triangle incl. diagonal: p = J(J+1)/2 + I, I <= J
__device__ __forceinline__ void unrank_tile_pair(const int p, int &I, int &J) {
    J = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
    while (J * (J + 1) / 2 > p) --J;
    while ((J + 1) * (J + 2) / 2 <= p) ++J;
    I = p - J * (J + 1) / 2;
}

// grid (ctas per query, queries); every role walks the same list of tile pairs
__global__ void __launch_bounds__(GM_THREADS, 2) bd_gram_kernel(const uint8_t *__restrict__ M8, const int NB,
                                                                 const int KS, const i64 n,
                                                                 const i64 *__restrict__ qidx,
                                                                 i64 *__restrict__ out) {
    extern __shared__ __align__(1024) uint8_t gm_smem[];  // GM_STAGES x (A tile | B tile)
    __shared__ __align__(8) u64 full_bar[GM_STAGES];
    __shared__ __align__(8) u64 empty_bar[GM_STAGES];
    __shared__ __align__(8) u64 tmem_full_bar[2];
    __shared__ __align__(8) u64 tmem_empty_bar[2];
    __shared__ u32 tmem_base_holder;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.y;
    const int qi = (int)qidx[q];
    const uint8_t *Mq = M8 + (i64)q * NB * KS * GM_TILE_BYTES;
    const int npairs = NB * (NB + 1) / 2;

    if (threadIdx.x == 0) {
        for (int s = 0; s < GM_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full_bar[a], 1);
            mbar_init(&tmem_empty_bar[a], 4);  // one arrive per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         smem_u32(&tmem_base_holder)),
                     "r"(GM_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tmem_base = tmem_base_holder;

    if (warp == 0) {
        // ===== producer =====
        if (lane == 0) {
            int stage = 0;
            u32 phase = 0;
            for (int p = blockIdx.x; p < npairs; p += gridDim.x) {
                int I, J;
                unrank_tile_pair(p, I, J);
                for (int ks = 0; ks < KS; ++ks) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    uint8_t *dst = gm_smem + (size_t)stage * 2 * GM_TILE_BYTES;
                    mbar_arrive_expect_tx(&full_bar[stage], 2u * GM_TILE_BYTES);
                    bulk_g2s(dst, Mq + ((i64)I * KS + ks) * GM_TILE_BYTES, GM_TILE_BYTES, &full_bar[stage]);
                    bulk_g2s(dst + GM_TILE_BYTES, Mq + ((i64)J * KS + ks) * GM_TILE_BYTES, GM_TILE_BYTES,
                             &full_bar[stage]);
                    if (++stage == GM_STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            int stage = 0;
            u32 phase = 0, tile_it = 0;
            for (int p = blockIdx.x; p < npairs; p += gridDim.x, ++tile_it) {
                const u32 acc = tile_it & 1u;             // accumulator stage
                const u32 use = (tile_it >> 1) & 1u;      // parity of this stage's use count
                mbar_wait(&tmem_empty_bar[acc], use ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const u32 tmem_d = tmem_base + acc * (u32)GM_TILE;
                for (int ks = 0; ks < KS; ++ks) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const u32 a0 = smem_u32(gm_smem + (size_t)stage * 2 * GM_TILE_BYTES);
                    const u32 b0 = a0 + GM_TILE_BYTES;
#pragma unroll
                    for (int k = 0; k < GM_KSTAGE / 32; ++k) {  // K = 32 bytes = 2 chunk planes per instruction
                        tc_mma_i8(tmem_d, umma_desc(a0 + k * 2 * GM_CHUNK_PLANE),
                                  umma_desc(b0 + k * 2 * GM_CHUNK_PLANE), GM_IDESC, (u32)((ks | k) != 0));
                    }
                    tc_commit(&empty_bar[stage]);  // smem stage is free once these MMAs have read it
                    if (++stage == GM_STAGES) { stage = 0; phase ^= 1u; }
                }
                tc_commit(&tmem_full_bar[acc]);  // accumulator complete
            }
        }
    } else {
        // ===== epilogue: warps 2..5 own TMEM lane quarters (warp % 4) =====
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        u64 count = 0;
        u32 tile_it = 0;
        for (int p = blockIdx.x; p < npairs; p += gridDim.x, ++tile_it) {
            int I, J;
            unrank_tile_pair(p, I, J);
            const u32 acc = tile_it & 1u, use = (tile_it >> 1) & 1u;
            mbar_wait(&tmem_full_bar[acc], use);
            tc_fence_after();
            const int c1 = I * GM_TILE + row;
            const bool row_ok = c1 < n && c1 != qi;
            // interior tiles (off the diagonal, fully inside n, not holding the query's column) only count zeros
            const bool plain = I != J && (i64)(J + 1) * GM_TILE <= n && !(qi >= J * GM_TILE && qi < (J + 1) * GM_TILE);
            u32 zeros = 0;
#pragma unroll 1
            for (int cb = 0; cb < GM_TILE / 32; ++cb) {
                u32 v[32];
                tc_ld_32x32(tmem_base + ((u32)(quarter * 32) << 16) + acc * (u32)GM_TILE + (u32)(cb * 32), v);
                if (plain) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) zeros += (u32)(v[j] == 0u);
                } else {
                    const int c2base = J * GM_TILE + cb * 32;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int c2 = c2base + j;
                        zeros += (u32)(v[j] == 0u && c2 > c1 && c2 < n && c2 != qi);
                    }
                }
            }
            if (row_ok) count += zeros;
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
        }
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) count += __shfl_xor_sync(0xffffffffu, count, s);
        if (lane == 0 && count) atomicAdd((u64 *)&out[q], count);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(GM_TMEM_COLS)
                     : "memory");
    }
}

// ---------------------------------------------------------------------------------------------
// int8 tensor-pipe probe: how fast can this chip retire tcgen05.mma.kind::i8 (M = 128, N = 128 or 256,
// K = 32) when nothing else is in the way?  One CTA per SM (or two), one thread issues `iters` MMAs on
// operand tiles that stay in shared memory, one commit, one wait.  Gives the MEASURED denominator for the
// Gram kernel's roofline fraction (MEASURED_PEAKS.json only has bf16).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) i8_peak_kernel(const int iters, const int ncols) {
    extern __shared__ __align__(1024) uint8_t pk_smem[];  // A tile 16 KB | B tile 32 KB (zeros are fine)
    __shared__ __align__(8) u64 done_bar;
    __shared__ u32 tmem_holder;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (16384 + 32768) / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(pk_smem)[i] = make_uint4(0x01010101u, 0x01000100u, 0u, 0x01010101u);
    if (threadIdx.x == 0) {
        mbar_init(&done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_holder)),
                     "r"((u32)ncols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy smem writes -> async proxy (MMA)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tmem_base = tmem_holder;
    if (warp == 1 && lane == 0) {
        const u32 a0 = smem_u32(pk_smem), b0 = a0 + 16384;
        // N = ncols: B tile has ncols rows -> chunk plane = ncols * 16 bytes
        const u32 planeB = (u32)ncols * 16u;
        const u32 idesc = (2u << 4) | ((u32)(ncols >> 3) << 17) | ((u32)(GM_TILE >> 4) << 24);
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                u64 da = umma_desc(a0 + k * 2 * GM_CHUNK_PLANE);
                u64 db = 0;
                db |= (u64)(((b0 + k * 2 * planeB) >> 4) & 0x3fffu);
                db |= (u64)((planeB >> 4) & 0x3fffu) << 16;
                db |= (u64)((128u >> 4) & 0x3fffu) << 32;
                db |= (u64)1 << 46;
                tc_mma_i8(tmem_base, da, db, idesc, (u32)((it | k) != 0));
            }
        }
        tc_commit(&done_bar);
        mbar_wait(&done_bar, 0);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((u32)ncols)
                     : "memory");
    }
}

// best of {N = 128, N = 256} x {1, 2 CTAs per SM}; returns int8 ops/s (2 ops per MAC)
int probe_int8_peak(sd_ctx *ctx, double *ops_per_s) {
    cudaStream_t st = ctx->stream;
    const size_t smem = 16384 + 32768;
    SD_CUDA(cudaFuncSetAttribute(i8_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEvent_t e0, e1;
    SD_CUDA(cudaEventCreate(&e0));
    SD_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    const int iters = 4000;
    for (int ncols = 128; ncols <= 256; ncols <<= 1) {
        for (int per_sm = 1; per_sm <= 2; ++per_sm) {
            const int grid = ctx->sm_count * per_sm;
            i8_peak_kernel<<<grid, 128, smem, st>>>(200, ncols);  // warm-up
            SD_CUDA(cudaEventRecord(e0, st));
            i8_peak_kernel<<<grid, 128, smem, st>>>(iters, ncols);
            SD_CUDA(cudaEventRecord(e1, st));
            SD_CUDA(cudaStreamSynchronize(st));
            SD_CUDA(cudaGetLastError());
            float ms = 0.f;
            SD_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            const double ops = 2.0 * 128.0 * (double)ncols * 32.0 * 4.0 * (double)iters * (double)grid;
            const double rate = ops / ((double)ms * 1e-3);
            if (rate > best) best = rate;
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ops_per_s = best;
    return SD_OK;
}

int bd_strict_gemm_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq,
                          i64 *d_out) {
    if (n < 1 || T < 1 || ld < n || nq < 0) {
        set_error("strict band depth (gemm): bad shape");
        return SD_ERR_INVALID;
    }
    if (n >= (1ll << 30)) {
        set_error("strict band depth (gemm): n too large");
        return SD_ERR_UNSUPPORTED;
    }
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)nq * sizeof(i64), st));
    if (nq == 0) return SD_OK;
    const int NB = (int)ceil_div(n, GM_TILE);
    const int KS = (int)ceil_div(T, GM_TSTEP);
    if (2 * KS > 65535) {
        set_error("strict band depth (gemm): T too large");
        return SD_ERR_UNSUPPORTED;
    }
    const size_t per_q = (size_t)NB * KS * GM_TILE_BYTES;
    i64 QB = (i64)((2ull << 30) / per_q);
    if (QB < 1) QB = 1;
    if (QB > 16384) QB = 16384;
    if (QB > nq) QB = nq;
    SD_TRY(ctx->buf[BUF_MASK].reserve((size_t)QB * per_q));
    uint8_t *M8 = ctx->buf[BUF_MASK].as<uint8_t>();
    const size_t smem = (size_t)GM_STAGES * 2 * GM_TILE_BYTES;
    SD_CUDA(cudaFuncSetAttribute(bd_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int npairs = NB * (NB + 1) / 2;
    int G = npairs < 32 ? npairs : 32;  // CTAs per query: few enough that concurrent queries' masks stay in L2
    for (i64 q0 = 0; q0 < nq; q0 += QB) {
        const int nqb = (int)(nq - q0 < QB ? nq - q0 : QB);
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_MASKS));
        bd_mask8_kernel<<<dim3((unsigned)NB, (unsigned)(2 * KS), (unsigned)ceil_div(nqb, GM_MQ)), GM_TILE, 0, st>>>(
            dX, T, n, ld, d_q + q0, nqb, NB, KS, M8, ctx->d_status);
        SD_TRY(prof_end(ctx));
        ctx->last.launches++;
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_PAIRS));
        bd_gram_kernel<<<dim3((unsigned)G, (unsigned)nqb), GM_THREADS, smem, st>>>(M8, NB, KS, n, d_q + q0, d_out + q0);
        SD_TRY(prof_end(ctx));
        ctx->last.launches++;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
