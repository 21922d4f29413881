// Matrix DFT (prysm/fttools.py:155-232, forward apply) as a tcgen05 / TMEM complex GEMM for complex64.
//
//   out(My,Mx) = norm * Ey(My,Ny) @ a(Ny,Nx) @ Ex(Mx,Nx)^T
//
// Mapping onto the 5th-generation tensor cores
//   * Complex -> real.  A complex matrix stored interleaved is a real matrix with twice the columns.
//     With the basis expanded once per executor to  B'[2j]   = ( E_re[j,:], -E_im[j,:] ) interleaved,
//                                                   B'[2j+1] = ( E_im[j,:],  E_re[j,:] ) interleaved,
//     the product  C'(m, 2j+c) = sum_k' A'(m,k') B'(2j+c,k')  is the complex product a @ E^T with its
//     (re, im) pairs already interleaved: the user's array is consumed exactly as it lies in memory,
//     both operands are K-major, and 8 real flops are spent per complex MAC (no wasted work).
//   * fp32 accuracy from TF32 MMAs.  x = hi + lo with hi = x truncated to TF32 (what the tensor core
//     reads from an fp32 operand) and lo = x - hi (exact).  a*b ~= hi*hi + hi*lo + lo*hi: three
//     kind::tf32 MMAs per K step, the two small products into a second TMEM accumulator so their low
//     bits survive, summed in the epilogue.  Dropped term lo*lo ~ 2^-22.
//   * Association.  (a @ Ex^T) first, written TRANSPOSED by the epilogue (TMEM lanes are output rows,
//     so for a fixed column the 32 lanes of a warp store 32 consecutive elements: coalesced for free);
//     then out^T' = T1^T' @ Ey'^T with split-K over the long contraction and a small reduce kernel that
//     applies `norm` and lands the result in (My,Mx) orientation.  Same flop count as the reference's
//     left-first order for square problems; the result is the same sum.
//
//   * Accumulation.  The tensor core's fp32 accumulate truncates: measured error grows linearly with the
//     number of accumulation steps (1.5e-5 at K' = 8192).  The main accumulator is therefore drained every
//     CHUNK K-blocks into fp32 registers (round-to-nearest adds on the CUDA cores, two epilogue threads per
//     output row), which brings the result under 1e-6 of the fp64 reference; the correction accumulator is
//     2^-11 smaller and runs undrained.
//
// Kernel shape: one 128 x 256 output tile per CTA (UMMA M=128, N=256, K=8), 4-stage TMA -> smem ring of
// 64-byte-swizzled K-major tiles (A_hi, A_lo 8 KB each; B_hi, B_lo 16 KB each; 48 KB per stage),
// warp 0 = TMA producer, warp 1 = MMA issuer (one elected thread), warp 2 = TMEM allocator,
// warps 4-11 = epilogue (tcgen05.ld 32x32b; lane quarter = warp % 4, column half = (warp - 4) / 4).  All 512 TMEM columns are used:
// 256 for the main accumulator, 256 for the correction accumulator.
#include <cuda.h>

#include "mdft_tc.cuh"

namespace pb {
namespace {

// K extent of a pipeline stage, in fp32 = one 64-byte swizzle row; 48 KB stages, a ring of 4.  Stages twice as deep
// (128-byte swizzle, 96 KB, a ring of 2) were measured and dropped: the MMA of one 32-deep stage takes ~0.84 us, less than
// the L2 -> shared latency of the next stage's 80 KB plus the lo-split behind it, and with two stages only one load is
// ever in flight: the tensor pipe sat at 66 % (profiles/r02_ncu_mdft_summary.txt).  Four stages keep three loads in flight.
constexpr int BM = 128, BN = 256, BK = 16;
constexpr int STAGES = 4;
constexpr int NTHREADS = 384;   // warp 0 TMA, 1 MMA, 2-3 TMEM alloc + TF32 lo-split converters, 4-11 epilogue
constexpr uint32_t A_TILE = BM * BK * 4;             // 8 KB
constexpr uint32_t B_TILE = BN * BK * 4;             // 16 KB
constexpr uint32_t STAGE_BYTES = 2 * A_TILE + 2 * B_TILE;  // 48 KB
constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// K-major, swizzled: rows of BK fp32 (64 B), 8-row groups 8 rows apart
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);   // start address
    d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)((8 * BK * 4) >> 4) << 32;      // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
    d |= (uint64_t)4 << 61;                        // SWIZZLE_64B
    return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct GemmParams {
    int kblocks;        // K blocks of BK handled by one CTA
    int chunk;          // K blocks accumulated in TMEM between drains of the main accumulator
    int mode;           // 0: write complex transposed (stage 1); 1: write fp32 transposed split-K partials
    float* out_hi;      // mode 0: T1^T hi as complex (float2) [N/2][ldo]; mode 1: ws [split][N][ldo]
    float* out_lo;      // mode 0: T1^T lo
    long long ldo;      // leading dimension of the transposed output, in output elements
    long long split_stride;  // mode 1: elements between split-K partial planes
};

// TF32 split with ROUNDING: hi = rn_tf32(x), lo = rn_tf32(x - hi).  Both parts are exactly representable in TF32, so the
// tensor core's own conversion (a truncation of the low 13 mantissa bits) leaves them untouched.  Splitting by truncation
// instead (hi = x with the low bits cleared, lo = x - hi read truncated) is one-sided: every product comes out low by up
// to ~2^-22 and the bias adds up coherently -- measured 8.4e-7 (field) / 1.7e-6 (intensity) at 4096^2 -> 512^2 against
// the fp64 reference; with rounding the residual is two-sided.
__device__ __forceinline__ float tf32_trunc(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }
__device__ __forceinline__ float tf32_rn(float v) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
    return __uint_as_float(u);
}

__global__ void __launch_bounds__(NTHREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmAhi, const __grid_constant__ CUtensorMap tmBhi,
               const __grid_constant__ CUtensorMap tmBlo, const GemmParams p) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* full = bars;              // [STAGES]  TMA -> MMA
    uint64_t* empty = bars + STAGES;    // [STAGES]  MMA -> TMA
    uint64_t* conv = bars + 2 * STAGES; // [STAGES]  converters -> MMA: the lo tiles of the stage are in shared memory
    uint64_t* tmem_full = bars + 3 * STAGES;       // MMA -> epilogue: a chunk is complete in TMEM
    uint64_t* tmem_empty = bars + 3 * STAGES + 1;  // epilogue -> MMA: the main accumulator was drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int kb0 = blockIdx.z * p.kblocks;
    const int CHUNK = p.chunk;
    const int nchunks = (p.kblocks + CHUNK - 1) / CHUNK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBlo) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); mbar_init(&conv[s], 64); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 8);  // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {  // all 512 TMEM columns: [0,256) main accumulator, [256,512) correction accumulator
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            for (int kb = 0; kb < p.kblocks; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                unsigned char* st = smem + s * STAGE_BYTES;
                mbar_expect_tx(&full[s], A_TILE + 2 * B_TILE);
                const int kc = (kb0 + kb) * BK;
                tma_load_2d(st, &tmAhi, kc, m0, &full[s]);                 // fp32 A: read as TF32 it IS the hi part
                tma_load_2d(st + 2 * A_TILE, &tmBhi, kc, n0, &full[s]);
                tma_load_2d(st + 2 * A_TILE + B_TILE, &tmBlo, kc, n0, &full[s]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            // instruction descriptor: D = F32, A = B = TF32, both K-major, N = 256, M = 128
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint32_t d_main = tmem_base, d_corr = tmem_base + 256;
            for (int kb = 0; kb < p.kblocks; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                const int c = kb / CHUNK, kin = kb - c * CHUNK;
                if (kin == 0 && c > 0) {  // the epilogue must have drained the previous chunk
                    mbar_wait(tmem_empty, (c - 1) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                mbar_wait(&conv[s], ph);   // TMA landed AND the converter warps wrote the lo tiles
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
                const uint64_t a_hi = make_desc(sa), a_lo = make_desc(sa + A_TILE);
                const uint64_t b_hi = make_desc(sa + 2 * A_TILE), b_lo = make_desc(sa + 2 * A_TILE + B_TILE);
#pragma unroll
                for (int ks = 0; ks < BK / 8; ++ks) {
                    const uint64_t adv = (uint64_t)(ks * 32 >> 4);  // 8 tf32 = 32 B along K inside the swizzle row
                    umma_tf32(d_main, a_hi + adv, b_hi + adv, idesc, (kin | ks) != 0);
                    umma_tf32(d_corr, a_hi + adv, b_lo + adv, idesc, (kb | ks) != 0);
                    umma_tf32(d_corr, a_lo + adv, b_hi + adv, idesc, 1u);
                }
                umma_commit(&empty[s]);   // frees the smem stage once these MMAs have read it
                if (kin == CHUNK - 1 || kb == p.kblocks - 1) umma_commit(tmem_full);  // chunk complete
            }
        }
    } else if (warp == 2 || warp == 3) {
        // ===== converters: lo = x - tf32(x) for the A tile, element for element in the swizzled layout.
        // The TF32 split used to be a streaming pre-pass over the whole input plus a second operand array; forming it on
        // the tile in shared memory removes that pass and the loads of the A_lo tiles.
        const int ct = threadIdx.x - 2 * 32;
        for (int kb = 0; kb < p.kblocks; ++kb) {
            const int s = kb % STAGES;
            const uint32_t ph = (kb / STAGES) & 1;
            mbar_wait(&full[s], ph);
            float4* st = reinterpret_cast<float4*>(smem + s * STAGE_BYTES);
            auto split = [&](float4* hi, float4* lo, int n4) {
                // hi = the value as the tensor core will read it (fp32 -> TF32 is a truncation): left in place, not
                // rewritten; lo = rn_tf32(x - hi) captures that truncation exactly and is itself TF32-exact, so the
                // split is unbiased at no extra shared-memory traffic.  All loads of a batch are issued before the first
                // use: the conversion sits between the TMA landing and the MMA issue, its latency is on the critical path.
                constexpr int BATCH = 8;     // tiles are multiples of 64 * BATCH float4
                for (int i0 = ct; i0 < n4; i0 += 64 * BATCH) {
                    float4 v[BATCH];
#pragma unroll
                    for (int j = 0; j < BATCH; ++j) v[j] = hi[i0 + 64 * j];
#pragma unroll
                    for (int j = 0; j < BATCH; ++j)
                        lo[i0 + 64 * j] = make_float4(tf32_rn(v[j].x - tf32_trunc(v[j].x)), tf32_rn(v[j].y - tf32_trunc(v[j].y)),
                                                      tf32_rn(v[j].z - tf32_trunc(v[j].z)), tf32_rn(v[j].w - tf32_trunc(v[j].w)));
                }
            };
            split(st, st + A_TILE / 16, A_TILE / 16);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core (async proxy) reads
            mbar_arrive(&conv[s]);
        }
    } else if (warp >= 4) {
        // ===== epilogue: drain chunks into registers, then transposed global stores =====
        const int q = warp & 3;              // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;    // which 128 of the 256 tile columns
        const int m = m0 + q * 32 + lane;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + half * 128;
        float tot[128];
#pragma unroll
        for (int i = 0; i < 128; ++i) tot[i] = 0.f;
        for (int c = 0; c < nchunks; ++c) {
            mbar_wait(tmem_full, c & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int c0 = 0; c0 < 128; c0 += 16) {
                uint32_t a[16];
                tmem_ld16(taddr + c0, a);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 16; ++i) tot[c0 + i] += __uint_as_float(a[i]);
            }
            if (c + 1 < nchunks) {
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(tmem_empty);
            }
        }
        // every MMA (including the correction products) has completed: fold the correction accumulator in
#pragma unroll
        for (int c0 = 0; c0 < 128; c0 += 16) {
            uint32_t b[16];
            tmem_ld16(taddr + 256 + c0, b);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 16; ++i) tot[c0 + i] += __uint_as_float(b[i]);
        }
        const int nb = n0 + half * 128;
        if (p.mode == 0) {
            float2* __restrict__ hi = reinterpret_cast<float2*>(p.out_hi);
#pragma unroll
            for (int c = 0; c < 128; c += 2) {
                const long long o = (long long)((nb + c) >> 1) * p.ldo + m;
                hi[o] = make_float2(tot[c], tot[c + 1]);
            }
        } else {
            float* __restrict__ ws = p.out_hi + (long long)blockIdx.z * p.split_stride;
#pragma unroll
            for (int c = 0; c < 128; ++c) ws[(long long)(nb + c) * p.ldo + m] = tot[c];
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// =====================================================================================================
// Stream-K form of tc_gemm_kernel for grids that do not fill the GPU (stage 1 at C3 is 128 tiles on 148 SMs).
// The work of a launch -- tiles x K-blocks, in units of one drain chunk -- is cut into gridDim.x equal contiguous
// ranges, one per CTA (one CTA per SM).  A range covers the tail of one tile, possibly whole tiles, and the head of
// another: the CTA walks its SEGMENTS (tile, K-block range) through the same TMA / converter / MMA / epilogue pipelines
// as the classic kernel (ring stage and chunk phase counters simply run on across segments).  The segment that STARTS a
// tile's K range owns the tile's output; it is its CTA's last segment.  Every segment that starts inside a tile is its
// CTA's FIRST: it writes its partial tile to the CTA's slot of the workspace and publishes it (gpu-scope fence +
// counter) before the CTA goes on, so a partial is never published after a wait.  The owner adds the partials of CTAs
// g+1, g+2, ... in that fixed order (deterministic) and stores as the classic kernel does; by the time it gets there
// they have long been published.  (Owning by the LAST piece instead chains every CTA behind its predecessor: 4.8 ms.)
// =====================================================================================================
struct SkParams {
    GemmParams g;        // g.kblocks = K-blocks per TILE; g.chunk divides it; g.mode = 0
    int ntn;             // tiles along N
    int ntiles;          // tiles of the launch
    float scale;         // applied in the owner's store (1 for stage 1, the executor norm for stage 2)
    float* part;         // [gridDim.x][256][128] partial tiles, column-major inside the tile
    int* flags;          // [gridDim.x] epilogue warps of CTA g that have published its partial (zeroed before the launch)
};

struct SkSeg { int tile, kb0, kb1, m0, n0; };
// segment of the CTA's range [u0, u1) that starts at unit u
__device__ __forceinline__ SkSeg sk_segment(int u, int u1, int upt, int chunk, int ntn) {
    SkSeg s;
    s.tile = u / upt;
    const int ub = u - s.tile * upt;
    const int ue = min(upt, ub + (u1 - u));
    s.kb0 = ub * chunk; s.kb1 = ue * chunk;
    s.m0 = (s.tile / ntn) * BM; s.n0 = (s.tile % ntn) * BN;
    return s;
}

__global__ void __launch_bounds__(NTHREADS, 1)
tc_gemm_sk_kernel(const __grid_constant__ CUtensorMap tmAhi, const __grid_constant__ CUtensorMap tmBhi,
                  const __grid_constant__ CUtensorMap tmBlo, const SkParams sp) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* full = bars;              // [STAGES]  TMA -> converters
    uint64_t* empty = bars + STAGES;    // [STAGES]  MMA -> TMA
    uint64_t* conv = bars + 2 * STAGES; // [STAGES]  converters -> MMA
    uint64_t* tmem_full = bars + 3 * STAGES;       // MMA -> epilogue: a chunk is complete in TMEM
    uint64_t* tmem_empty = bars + 3 * STAGES + 1;  // epilogue -> MMA: the accumulators were read
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 2);

    const GemmParams& p = sp.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int CHUNK = p.chunk;
    const int upt = p.kblocks / CHUNK;                         // units (chunks) per tile
    const long long U = (long long)sp.ntiles * upt;
    const int G = gridDim.x, g = blockIdx.x;
    const int u0 = (int)(U * g / G), u1 = (int)(U * (g + 1) / G);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBlo) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); mbar_init(&conv[s], 64); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 8);  // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            int i = 0;   // K-blocks of this CTA so far: ring stage and phase run on across segments
            for (int u = u0; u < u1;) {
                const SkSeg sg = sk_segment(u, u1, upt, CHUNK, sp.ntn);
                for (int kb = sg.kb0; kb < sg.kb1; ++kb, ++i) {
                    const int s = i % STAGES;
                    const uint32_t ph = (i / STAGES) & 1;
                    mbar_wait(&empty[s], ph ^ 1);
                    unsigned char* st = smem + s * STAGE_BYTES;
                    mbar_expect_tx(&full[s], A_TILE + 2 * B_TILE);
                    const int kc = kb * BK;
                    tma_load_2d(st, &tmAhi, kc, sg.m0, &full[s]);
                    tma_load_2d(st + 2 * A_TILE, &tmBhi, kc, sg.n0, &full[s]);
                    tma_load_2d(st + 2 * A_TILE + B_TILE, &tmBlo, kc, sg.n0, &full[s]);
                }
                u += (sg.kb1 - sg.kb0) / CHUNK;
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint32_t d_main = tmem_base, d_corr = tmem_base + 256;
            int i = 0, c = 0;   // K-blocks and chunks of this CTA so far
            for (int u = u0; u < u1;) {
                const SkSeg sg = sk_segment(u, u1, upt, CHUNK, sp.ntn);
                for (int kb = sg.kb0; kb < sg.kb1; ++kb, ++i) {
                    const int s = i % STAGES;
                    const uint32_t ph = (i / STAGES) & 1;
                    const int kin = kb % CHUNK;          // segments start on chunk boundaries
                    if (kin == 0 && c > 0) {  // the epilogue must have read the previous chunk (and, at a segment end, the correction accumulator)
                        mbar_wait(tmem_empty, (c - 1) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    }
                    mbar_wait(&conv[s], ph);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
                    const uint64_t a_hi = make_desc(sa), a_lo = make_desc(sa + A_TILE);
                    const uint64_t b_hi = make_desc(sa + 2 * A_TILE), b_lo = make_desc(sa + 2 * A_TILE + B_TILE);
#pragma unroll
                    for (int ks = 0; ks < BK / 8; ++ks) {
                        const uint64_t adv = (uint64_t)(ks * 32 >> 4);
                        umma_tf32(d_main, a_hi + adv, b_hi + adv, idesc, (kin | ks) != 0);
                        umma_tf32(d_corr, a_hi + adv, b_lo + adv, idesc, ((kb - sg.kb0) | ks) != 0);
                        umma_tf32(d_corr, a_lo + adv, b_hi + adv, idesc, 1u);
                    }
                    umma_commit(&empty[s]);
                    if (kin == CHUNK - 1) { umma_commit(tmem_full); ++c; }
                }
                u += (sg.kb1 - sg.kb0) / CHUNK;
            }
        }
    } else if (warp == 2 || warp == 3) {
        // ===== converters: lo part of the A tile, see tc_gemm_kernel =====
        const int ct = threadIdx.x - 2 * 32;
        const int nkb = (u1 - u0) * CHUNK;
        for (int i = 0; i < nkb; ++i) {
            const int s = i % STAGES;
            const uint32_t ph = (i / STAGES) & 1;
            mbar_wait(&full[s], ph);
            float4* hi = reinterpret_cast<float4*>(smem + s * STAGE_BYTES);
            float4* lo = hi + A_TILE / 16;
            constexpr int BATCH = 8;
            for (int i0 = ct; i0 < (int)(A_TILE / 16); i0 += 64 * BATCH) {
                float4 v[BATCH];
#pragma unroll
                for (int j = 0; j < BATCH; ++j) v[j] = hi[i0 + 64 * j];
#pragma unroll
                for (int j = 0; j < BATCH; ++j)
                    lo[i0 + 64 * j] = make_float4(tf32_rn(v[j].x - tf32_trunc(v[j].x)), tf32_rn(v[j].y - tf32_trunc(v[j].y)),
                                                  tf32_rn(v[j].z - tf32_trunc(v[j].z)), tf32_rn(v[j].w - tf32_trunc(v[j].w)));
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_arrive(&conv[s]);
        }
    } else if (warp >= 4) {
        // ===== epilogue: per segment drain its chunks; then publish a partial tile or (tile owner) gather and store =====
        const int q = warp & 3;              // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;    // which 128 of the 256 tile columns
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + half * 128;
        const int total_chunks = u1 - u0;
        const long long slot = (long long)(half * 128) * BM + q * 32 + lane;   // this thread's first element of a partial tile
        int c = 0;
        for (int u = u0; u < u1;) {
            const SkSeg sg = sk_segment(u, u1, upt, CHUNK, sp.ntn);
            const int nseg = (sg.kb1 - sg.kb0) / CHUNK;
            float tot[128];
#pragma unroll
            for (int i = 0; i < 128; ++i) tot[i] = 0.f;
            for (int cs = 0; cs < nseg; ++cs) {
                mbar_wait(tmem_full, c & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int c0 = 0; c0 < 128; c0 += 16) {
                    uint32_t a[16];
                    tmem_ld16(taddr + c0, a);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int i = 0; i < 16; ++i) tot[c0 + i] += __uint_as_float(a[i]);
                }
                if (cs == nseg - 1) {   // the segment's MMAs are complete: fold its correction accumulator in
#pragma unroll
                    for (int c0 = 0; c0 < 128; c0 += 16) {
                        uint32_t b[16];
                        tmem_ld16(taddr + 256 + c0, b);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int i = 0; i < 16; ++i) tot[c0 + i] += __uint_as_float(b[i]);
                    }
                }
                ++c;
                if (c < total_chunks) {
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tmem_empty);
                }
            }
            if (sg.kb0 > 0) {
                // a tail or middle piece of its tile: always the FIRST segment of this CTA, so it is published early and
                // never after a wait -- the tile's owner (below) finds it ready when it gets there
                float* __restrict__ dst = sp.part + (long long)g * (BM * BN) + slot;
#pragma unroll
                for (int cc = 0; cc < 128; ++cc) __stcg(dst + (long long)cc * BM, tot[cc]);
                __syncwarp();
                if (lane == 0) { __threadfence(); atomicAdd(sp.flags + g, 1); }
            } else {
                if (sg.kb1 < p.kblocks) {
                    // the head of a tile whose K range continues in CTAs g+1, g+2, ...: this CTA owns the tile (it is its LAST
                    // segment) and adds their partials in that fixed order
                    const long long tile_u1 = (long long)(sg.tile + 1) * upt;
                    for (int gp = g + 1; gp < G; ++gp) {
                        if (lane == 0) { while (ld_acquire_gpu(sp.flags + gp) < 8) __nanosleep(64); }
                        __syncwarp();
                        const float* __restrict__ src = sp.part + (long long)gp * (BM * BN) + slot;
#pragma unroll
                        for (int cc = 0; cc < 128; ++cc) tot[cc] += __ldcg(src + (long long)cc * BM);
                        if (U * (gp + 1) / G >= tile_u1) break;   // that piece reached the tile's last K-block
                    }
                }
                const int m = sg.m0 + q * 32 + lane;
                const int nb = sg.n0 + half * 128;
                float2* __restrict__ hi = reinterpret_cast<float2*>(p.out_hi);
#pragma unroll
                for (int cc = 0; cc < 128; cc += 2) {
                    const long long o = (long long)((nb + cc) >> 1) * p.ldo + m;
                    hi[o] = make_float2(sp.scale * tot[cc], sp.scale * tot[cc + 1]);
                }
            }
            u += nseg;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// complex basis E (m,n) -> real expansion (2m, 2n), hi and lo
__global__ void expand_basis_kernel(const float2* __restrict__ E, int m, int n, float* __restrict__ hi, float* __restrict__ lo) {
    const long long tot = (long long)m * n;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(i / n), l = (int)(i - (long long)j * n);
        const float2 e = E[i];
        const long long r0 = (long long)(2 * j) * (2 * n) + 2 * l, r1 = r0 + 2 * n;
        const float v00 = e.x, v01 = -e.y, v10 = e.y, v11 = e.x;
        const float h00 = tf32_rn(v00), h01 = tf32_rn(v01), h10 = tf32_rn(v10), h11 = tf32_rn(v11);
        hi[r0] = h00; hi[r0 + 1] = h01; hi[r1] = h10; hi[r1 + 1] = h11;
        lo[r0] = tf32_rn(v00 - h00); lo[r0 + 1] = tf32_rn(v01 - h01); lo[r1] = tf32_rn(v10 - h10); lo[r1 + 1] = tf32_rn(v11 - h11);
    }
}

// out(i,j) = norm * sum_s ws[s][2i+c][j]
__global__ void reduce_splits_kernel(const float* __restrict__ ws, int splits, int my, int mx, float norm, float2* __restrict__ out) {
    const long long tot = (long long)my * mx;
    const long long plane = (long long)2 * my * mx;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e / mx), j = (int)(e - (long long)i * mx);
        float re = 0.f, im = 0.f;
        for (int s = 0; s < splits; ++s) {
            re += ws[s * plane + (long long)(2 * i) * mx + j];
            im += ws[s * plane + (long long)(2 * i + 1) * mx + j];
        }
        out[e] = make_float2(norm * re, norm * im);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_map(Handle* h, CUtensorMap* map, const void* base, long long rows, long long cols, int box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        cudaDriverEntryPointQueryResult q;
        void* f = nullptr;
        PB_CUDA(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q));
        if (!f || q != cudaDriverEntryPointSuccess) return fail(h, PB_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        fn = reinterpret_cast<EncodeTiledFn>(f);
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)cols * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, PB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return PB_OK;
}

// C'(M x N) = A'(M x K) @ B'(N x K)^T on the tensor cores; see GemmParams for the output modes
int launch_gemm(Handle* h, const float* A, const float* Bhi, const float* Blo, int M, int N, long long K,
                int splits, const GemmParams& gp, cudaStream_t st) {
    CUtensorMap mAhi, mBhi, mBlo;
    PB_TRY(make_map(h, &mAhi, A, M, K, BM));
    PB_TRY(make_map(h, &mBhi, Bhi, N, K, BN));
    PB_TRY(make_map(h, &mBlo, Blo, N, K, BN));
    if (attr_needed(h, reinterpret_cast<const void*>(tc_gemm_kernel)))
        PB_CUDA(h, cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    dim3 grid(M / BM, N / BN, splits);
    tc_gemm_kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(mAhi, mBhi, mBlo, gp);
    PB_LAUNCH_CHECK(h);
    return PB_OK;
}

constexpr int SK_MAX_CTAS = 160;
constexpr long long SK_WORK_BYTES = (long long)SK_MAX_CTAS * BM * BN * 4 + 4096;   // partial tiles + flags

// stream-K form (mode 0 only): `work` = SK_WORK_BYTES of scratch
int launch_gemm_sk(Handle* h, const float* A, const float* Bhi, const float* Blo, int M, int N, long long K,
                   const GemmParams& gp, float scale, void* work, cudaStream_t st) {
    CUtensorMap mAhi, mBhi, mBlo;
    PB_TRY(make_map(h, &mAhi, A, M, K, BM));
    PB_TRY(make_map(h, &mBhi, Bhi, N, K, BN));
    PB_TRY(make_map(h, &mBlo, Blo, N, K, BN));
    if (attr_needed(h, reinterpret_cast<const void*>(tc_gemm_sk_kernel)))
        PB_CUDA(h, cudaFuncSetAttribute(tc_gemm_sk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    SkParams sp;
    sp.g = gp;
    sp.scale = scale;
    sp.ntn = N / BN;
    sp.ntiles = (M / BM) * (N / BN);
    sp.part = reinterpret_cast<float*>(work);
    sp.flags = reinterpret_cast<int*>(reinterpret_cast<char*>(work) + (long long)SK_MAX_CTAS * BM * BN * 4);
    const int grid = std::min(h->sm_count, SK_MAX_CTAS);
    PB_CUDA(h, cudaMemsetAsync(sp.flags, 0, SK_MAX_CTAS * sizeof(int), st));
    tc_gemm_sk_kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(mAhi, mBhi, mBlo, sp);
    PB_LAUNCH_CHECK(h);
    return PB_OK;
}

// Stream-K pays where the tile grid leaves a good part of the SMs idle and each tile is cut into 2-4 pieces (the owner's
// gather of the other pieces stays short); it needs whole drain chunks per tile and enough chunks to spread over the SMs.
bool use_stream_k(int tiles, int kblocks, int chunk, int sm_count) {
    return kblocks % chunk == 0 && tiles % sm_count != 0 && 5 * tiles < 4 * sm_count && 4 * tiles >= sm_count &&
           (long long)tiles * (kblocks / chunk) >= 4LL * sm_count;
}

int pick_splits(int ny) {
    // stage 2 has only (Mx/128)*(2My/256) tiles; split its long contraction (2*Ny) to fill the GPU
    const long long kblocks = 2LL * ny / BK;
    int s = 8;
    while (s > 1 && (kblocks % s != 0 || kblocks / s < 128 / BK)) s >>= 1;   // at least 128 K elements per split
    return s;
}

}  // namespace

bool mdft_tc_shape_ok(int my, int ny, int mx, int nx) {
    return my % 128 == 0 && mx % 128 == 0 && ny % 128 == 0 && nx % 16 == 0 && ny >= 128 && nx >= 16;
}


}  // namespace pb

using namespace pb;

extern "C" int pb_mdft_tc_supported(int my, int ny, int mx, int nx) { return mdft_tc_shape_ok(my, ny, mx, nx) ? 1 : 0; }

extern "C" int pb_mdft_tc_expand(pb_handle_t hh, const void* E, int m, int n, void* hi, void* lo, void* stream) {
    PB_ENTER(hh);
    if (m < 1 || n < 1 || !E || !hi || !lo) return fail(h, PB_ERR_INVALID, "bad expand arguments");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const long long tot = (long long)m * n;
    const int g = (int)std::min<long long>((tot + 255) / 256, (long long)h->sm_count * 16);
    expand_basis_kernel<<<g, 256, 0, st>>>((const float2*)E, m, n, (float*)hi, (float*)lo);
    PB_LAUNCH_CHECK(h);
    return PB_OK;
}

extern "C" long long pb_mdft_tc_work_bytes(int my, int ny, int mx, int nx) {
    (void)nx;
    const long long t1 = 2LL * ny * mx * 4;                   // T1^T (complex mx x ny)
    const long long ws = (long long)pick_splits(ny) * 2 * my * mx * 4;
    return t1 + ws + 4096 + SK_WORK_BYTES;
}

extern "C" int pb_mdft_tc_apply(pb_handle_t hh, const void* ExB_hi, const void* ExB_lo, const void* EyB_hi,
                                const void* EyB_lo, int my, int ny, int mx, int nx, const void* a, void* out, double norm,
                                void* work, void* stream) {
    PB_ENTER(hh);
    if (!mdft_tc_shape_ok(my, ny, mx, nx)) return fail(h, PB_ERR_UNSUPPORTED, "shape not covered by the tensor-core MDFT");
    if (!ExB_hi || !ExB_lo || !EyB_hi || !EyB_lo || !a || !out || !work) return fail(h, PB_ERR_INVALID, "null pointer");
    // TMA needs 16-byte aligned global base addresses (the 1 KB alignment of the swizzle atoms is a shared-memory matter);
    // every sub-buffer of `work` below starts at a multiple of 16 bytes given the shape constraints
    if (((uintptr_t)a & 15) || ((uintptr_t)work & 15)) return fail(h, PB_ERR_INVALID, "data / work must be 16-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int splits = pick_splits(ny);
    // 64 K elements (8 main accumulation steps) per drain: < 1e-6 of the fp64 result at any K (measured, in K elements
    // per drain: 512 -> 2e-6, 256 -> 1.5e-6, 128 -> 1.2e-6, 64 -> 9e-7 on random data; the drains hide behind the
    // L2-bound mainloop)
    constexpr int chunk = 2 * 32 / BK;   // in K-blocks of BK
    float* t1 = reinterpret_cast<float*>(work);
    float* ws = t1 + 2LL * ny * mx;
    char* skw = reinterpret_cast<char*>(ws + (long long)splits * 2 * my * mx);
    skw += (16 - ((uintptr_t)skw & 15)) & 15;
    {   // stage 1: T1^T(mx, ny) = (a @ Ex^T)^T : M = ny rows of a, N = 2*mx expanded basis rows, K = 2*nx
        GemmParams gp{(int)(2LL * nx / BK), chunk, 0, t1, nullptr, (long long)ny, 0};
        // stream-K when the tile grid leaves a good part of the SMs idle (1024^2 <-> 1024^2: 64 tiles on 148 SMs, 371 -> 346 us
        // for the coronagraph round trip); at C3 (128 tiles) it is neutral -- 358.7 against 356.5 us -- and not used.
        if (use_stream_k((ny / BM) * (2 * mx / BN), gp.kblocks, chunk, h->sm_count))
            PB_TRY(launch_gemm_sk(h, (const float*)a, (const float*)ExB_hi, (const float*)ExB_lo, ny, 2 * mx, 2LL * nx, gp, 1.0f, skw, st));
        else PB_TRY(launch_gemm(h, (const float*)a, (const float*)ExB_hi, (const float*)ExB_lo, ny, 2 * mx, 2LL * nx, 1, gp, st));
    }
    // stage 2: out^T' = T1^T' @ Ey'^T : M = mx, N = 2*my, K = 2*ny.  Few tiles and a long contraction: stream-K over all SMs
    // with the owner's store landing the result, scaled by `norm`, directly in (My, Mx) complex orientation (same index
    // arithmetic as stage 1's transposed complex store with ldo = mx) -- no partial planes, no reduce kernel: the 1024^2 <->
    // 1024^2 coronagraph round trip went from 340 to 249 us.  With very few tiles (C3: 16, i.e. 9 pieces per tile) the owner's
    // serial gather costs more than it saves (373.6 against 357.6 us): those, and shapes too small for it, take split-K + reduce.
    {
        const int kb2 = (int)(2LL * ny / BK);
        if (use_stream_k((mx / BM) * (2 * my / BN), kb2, chunk, h->sm_count)) {
            GemmParams gp{kb2, chunk, 0, reinterpret_cast<float*>(out), nullptr, (long long)mx, 0};
            return launch_gemm_sk(h, t1, (const float*)EyB_hi, (const float*)EyB_lo, mx, 2 * my, 2LL * ny, gp, (float)norm, skw, st);
        }
    }
    {   // split-K partials transposed into ws[s][2my][mx]
        GemmParams gp{(int)(2LL * ny / BK / splits), chunk, 1, ws, nullptr, (long long)mx, 2LL * my * mx};
        PB_TRY(launch_gemm(h, t1, (const float*)EyB_hi, (const float*)EyB_lo, mx, 2 * my, 2LL * ny, splits, gp, st));
    }
    {
        const long long tot = (long long)my * mx;
        const int g = (int)std::min<long long>((tot + 255) / 256, (long long)h->sm_count * 8);
        reduce_splits_kernel<<<g, 256, 0, st>>>(ws, splits, my, mx, (float)norm, (float2*)out);
        PB_LAUNCH_CHECK(h);
    }
    return PB_OK;
}
