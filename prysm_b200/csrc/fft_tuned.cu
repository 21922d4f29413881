// Tuned register-resident FFT kernels for the headline path: Wavefront.focus / unfocus with Q = 2
// on N x N complex64 pupils, N in {512, 1024, 2048}  (reference prysm/propagation/fft.py:7-65).
//
// Algebra.  K = 2N.  focus = fftshift(FFT2_K(ifftshift(pad(x)))).  Along one axis, with q = x
// zero-extended to K:   U[k] = (-dir*i)^k * Q[k]   (the centred pad + ifftshift is a circular
// shift by K/4), and the zero half makes the first radix-2 level trivial:
//      Q[2j]   = FFT_N(x)[j]                    ("even" half, lane A)
//      Q[2j+1] = FFT_N(x * w_K^n)[j]            ("odd" half,  lane B)
// so every length-K transform of the padded data is two length-N transforms of the un-padded
// data, the shifts are sign patterns / index rotations at the store, and no zero is ever read,
// written or multiplied.
//
// Packed arithmetic.  sm_100 issues two fp32 operations per instruction on 64-bit register pairs
// (FADD2 / FMUL2 / FFMA2).  Each thread therefore carries BOTH half-transforms of its line in
// structure-of-arrays form -- re = (re_A, re_B), im = (im_A, im_B) -- and every butterfly, twiddle
// multiply and store acts on the pair: the instruction count of the FFT is halved and the kernels
// move from issue-bound to FP32-pipe-bound.  The two lanes differ only in their inputs
// (lane B = x * w_32^n, immediates) and in the stage-1 twiddle (w_K^t folded into lane B's table entry).
//
// Data flow (columns first so that the K x K output is written by the row kernel in full rows with
// 128-bit stores):
//   focus_col_kernel : FFT_N down T adjacent columns of the pupil, both halves ->
//                      intermediate [2][N][N] (plane p, row j  <->  output row 2j+p, rotated by K/2)
//   focus_row_kernel : persistent; per intermediate row both half-transforms; thread owns outputs
//                      (2j, 2j+1) and stores them as one float4.  Rows arrive by bulk async copy
//                      (cp.async.bulk + mbarrier), one row ahead.
//   HBM traffic: pupil 8N^2 once, output 8K^2 once; the 16N^2-byte intermediate (64 MiB at N = 2048)
//   is written and re-read through the 126 MB L2.
//
// FFT_N engine: N/16 threads per line, 16 points x 2 lanes per thread in registers, radix
// 16 x 16 x N/256, two shared-memory exchanges of float4 (1-in-16 padded, conflict free).
#include "fft_engine.cuh"

namespace pb {
namespace {


// ---- column pass: both half-transforms down T adjacent columns -------------------------------------
template <int L, bool INV, int T>
__global__ void __launch_bounds__(T * L / 16) focus_col_kernel(const FocusParams p) {
    using G = Geo<L>;
    extern __shared__ __align__(128) float4 smem4[];
    float4* plan_s = smem4 + T * (G::SBUF + 2);                       // the twiddle plan, bulk-copied once
    uint64_t* bar = reinterpret_cast<uint64_t*>(plan_s + G::PLAN);
    const int c = threadIdx.x % T, t = threadIdx.x / T;
    const int col = blockIdx.x * T + c;
    const long long fb = blockIdx.y;                                   // field of the batch
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
        mbar_expect_tx(bar, G::PLAN * sizeof(float4));
        bulk_g2s(plan_s, p.plan, G::PLAN * sizeof(float4), bar);
    }
    __syncthreads();
    P2 v[16];
    float2 x[16];
    if (p.in_kind == PB_IN_COMPLEX) {
        const float2* __restrict__ src = reinterpret_cast<const float2*>(p.in) + fb * p.in_bs + col + (long long)t * p.in_ld;
        const long long step = (long long)G::NT * p.in_ld;
#pragma unroll
        for (int n = 0; n < 16; ++n) x[n] = ld_stream(src + n * step);
    } else {
        const float* __restrict__ opd = reinterpret_cast<const float*>(p.in) + fb * p.in_bs + col;
        const long long ab = fb * p.amp_bs + col;
#pragma unroll
        for (int n = 0; n < 16; ++n) {
            const long long off = (long long)(n * G::NT + t) * p.in_ld;
            float a = 1.0f;
            if (p.amp_kind == PB_AMP_REAL) a = __ldg(reinterpret_cast<const float*>(p.amp) + ab + off);
            else if (p.amp_kind == PB_AMP_U8) a = __ldg(reinterpret_cast<const unsigned char*>(p.amp) + ab + off) ? 1.0f : 0.0f;
            float2 e = make_float2(0.f, 0.f);
            if (a != 0.0f) {
                e = expi_turns(p.kturns * (double)__ldg(opd + off), 0.0f);
                e.x *= a; e.y *= a;
            }
            x[n] = e;
        }
    }
#define PB_X(n) x[n]
    PB_MAKE_LANES_16(v, INV, PB_X)
#undef PB_X
    float4* S = smem4 + c * (G::SBUF + 2);  // +2: skews the T buffers across banks
    mbar_wait(bar, 0);
    fft_two_stages<L, INV, 1>(v, t, S, plan_s + G::TW1, plan_s + G::TW2, SyncCta(), SyncCta());
    fft_last_stage_load<L, INV>(v, t, S);
#pragma unroll
    for (int g = 0; g < G::GI; ++g) dftR<G::R3, INV>(v + g * G::R3);
    // (-dir*i)^k with k = 2j + lane; j = t + g*NT + 256*kk has the parity of t
    const float sgn = (t & 1) ? -1.0f : 1.0f;
    float2* __restrict__ dA = p.tmp + fb * (2LL * L * L) + col + (long long)t * L;
    float2* __restrict__ dB = dA + (long long)L * L;
#pragma unroll
    for (int g = 0; g < G::GI; ++g)
#pragma unroll
        for (int kk = 0; kk < G::R3; ++kk) {
            const P2 y = v[g * G::R3 + kk];
            const long long o = (long long)(g * G::NT + 256 * kk) * L;
            st_stream(dA + o, make_float2(sgn * y.re.x, sgn * y.im.x));
            // lane B times (-dir*i): forward (+i): (-im, re); inverse (-i): (im, -re)
            st_stream(dB + o, INV ? make_float2(sgn * y.im.y, -sgn * y.re.y) : make_float2(-sgn * y.im.y, sgn * y.re.y));
        }
}

// ---- row pass: persistent, both half-transforms of one intermediate row per iteration ---------------
template <int L, bool INV>
__global__ void __launch_bounds__(L / 16) focus_row_kernel(const FocusParams p) {
    using G = Geo<L>;
    constexpr int NT = G::NT, R3 = G::R3, GI = G::GI;
    constexpr uint32_t ROW_BYTES = L * sizeof(float2);
    extern __shared__ __align__(128) unsigned char smraw[];
    float4* S = reinterpret_cast<float4*>(smraw);                // SBUF exchange
    float2* inb = reinterpret_cast<float2*>(S + G::SBUF);        // L-element input row
    uint64_t* bar = reinterpret_cast<uint64_t*>(inb + L);        // 1 mbarrier
    const int t = threadIdx.x;
    int r = blockIdx.x;
    if (t == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
        if (r < p.nrows) {
            mbar_expect_tx(bar, ROW_BYTES);
            bulk_g2s(inb, p.tmp + (long long)r * L, ROW_BYTES, bar);
        }
    }
    __syncthreads();
    const float sgn = ((t & 1) ? -1.0f : 1.0f) * p.scale;
    for (int it = 0; r < p.nrows; ++it, r += gridDim.x) {
        P2 v[16];
        mbar_wait(bar, it & 1);
        {
            const float2* __restrict__ row = inb + t;
#define PB_X(n) row[(n) * NT]
            PB_MAKE_LANES_16(v, INV, PB_X)
#undef PB_X
        }
        const int rn = r + gridDim.x;
        auto sync_and_prefetch = [&]() {
            __syncthreads();  // every thread holds its inputs in registers: the row buffer is free
            if (t == 0 && rn < p.nrows) {
                mbar_expect_tx(bar, ROW_BYTES);
                bulk_g2s(inb, p.tmp + (long long)rn * L, ROW_BYTES, bar);
            }
        };
        fft_two_stages<L, INV, 0>(v, t, S, p.plan + G::TW1, p.plan + G::TW2, sync_and_prefetch, SyncCta());
        fft_last_stage_load<L, INV>(v, t, S);
        __syncthreads();  // exchange buffer is free for the next row
#pragma unroll
        for (int g = 0; g < GI; ++g) dftR<R3, INV>(v + g * R3);
        const int fb = r / (2 * L), rf = r - fb * (2 * L);   // field of the batch, row within its [2][L] planes
        const int phs = rf / L, rr = rf - phs * L;
        const int orow = (2 * rr + phs + L) & (2 * L - 1);  // fftshift along y
        if (p.out_kind == PB_OUT_COMPLEX) {
            float4* __restrict__ dst = reinterpret_cast<float4*>(reinterpret_cast<float2*>(p.out) + fb * p.out_bs + (long long)orow * p.out_ld);
#pragma unroll
            for (int g = 0; g < GI; ++g)
#pragma unroll
                for (int kk = 0; kk < R3; ++kk) {
                    const int j = t + g * NT + 256 * kk;
                    const P2 y = v[g * R3 + kk];
                    // U[2j] = (-1)^j A,  U[2j+1] = (-1)^j (-dir*i) B ; fftshift along x: pair index (j + L/2) mod L
                    const float4 o = INV ? make_float4(sgn * y.re.x, sgn * y.im.x, sgn * y.im.y, -sgn * y.re.y)
                                         : make_float4(sgn * y.re.x, sgn * y.im.x, -sgn * y.im.y, sgn * y.re.y);
                    st_stream(dst + ((j + L / 2) & (L - 1)), o);
                }
        } else {
            float2* __restrict__ dst = reinterpret_cast<float2*>(reinterpret_cast<float*>(p.out) + fb * p.out_bs + (long long)orow * p.out_ld);
            const float2 s2 = make_float2(p.scale * p.scale, p.scale * p.scale);
            const float2 wgt = make_float2(p.weight, p.weight);
#pragma unroll
            for (int g = 0; g < GI; ++g)
#pragma unroll
                for (int kk = 0; kk < R3; ++kk) {
                    const int j = t + g * NT + 256 * kk;
                    const P2 y = v[g * R3 + kk];
                    float2 I = __fmul2_rn(s2, __ffma2_rn(y.re, y.re, __fmul2_rn(y.im, y.im)));
                    float2* q = dst + ((j + L / 2) & (L - 1));
                    if (p.out_kind == PB_OUT_ACCUMULATE) I = __ffma2_rn(wgt, I, *q);
                    *q = I;
                }
        }
    }
}

// =====================================================================================================
// v2 pipeline: same arithmetic, different traffic.
//   * The intermediate is TILE-MAJOR: [field][plane p][j / 4][column tile = col / 4][j % 4][col % 4] complex64, i.e. the
//     4 x 4 block (4 output rows of one plane, 4 adjacent columns) is one 128-byte line.  A warp of the column kernel
//     (8 consecutive j x 4 columns) stores two full lines per instruction instead of eight 32-byte sectors in eight
//     lines -- the LSU pressure (`lg_throttle`) of the row-major layout is gone.
//   * The column kernel is persistent (one 512-thread CTA per SM walks the tiles of all fields of the launch) and takes
//     its 4-column input tile by tensor TMA (box = 4 columns x 256 rows, 32-byte runs gathered into a contiguous
//     [row][4] image that aliases the exchange buffers); the tile after next is requested as soon as the exchange
//     buffers are free, so it lands while the last butterflies and the stores of the current tile run.
//   * The row kernel (one 512-thread CTA per SM, four line groups, see GeoR4) gathers one intermediate row per group
//     (512 runs of 32 bytes, 128 bytes apart) with two tensor-TMA boxes into a contiguous row buffer; the transform and
//     the stores are those of the v1 row kernel.
// =====================================================================================================


template <int L, bool INV, int HALF>
__device__ __forceinline__ void focus_col4_group(const CUtensorMap& in_map, const FocusParams& p, float4* smem4, uint64_t* bar) {
    using G = Geo<L>;
    using G2 = Geo2<L>;
    using G4 = Geo4<L>;
    constexpr int NT = G::NT;
    const int lt = threadIdx.x & (2 * NT - 1);                       // thread within the group
    const int cp = lt & 1, t = lt >> 1;
    const float4* __restrict__ stage = smem4 + G4::STAGE;
    const float2* __restrict__ plan = reinterpret_cast<const float2*>(smem4 + G4::PLAN2);
    float4* S = smem4 + (HALF * 2 + cp) * G4::XBUF;
    const SyncGroup gsync{1 + HALF, 2 * NT};
    // the intermediate is re-read by the row kernel from L2: evict_last; the input is read once: evict_first
    const uint64_t pol_tmp = l2_policy(2), pol_in = l2_policy(1);
    auto request_tile = [&](int ww) {   // one thread: gather tile ww = (field, column tile) into the staging area
        const int fb = ww / G2::TILES, tile = ww - fb * G2::TILES;
        mbar_expect_tx(bar + 1, (uint32_t)(L * 4 * sizeof(float2)));
#pragma unroll
        for (int b = 0; b < G2::NBOX_IN; ++b)
            tma_load_3d(smem4 + G4::STAGE + b * G2::BOXR * 2, &in_map, tile * 4, b * G2::BOXR, fb, bar + 1, pol_in);
    };
    unsigned int* released = reinterpret_cast<unsigned int*>(bar + 2);   // warps that hold the inputs of the current tile, summed over tiles
    if (HALF == 0 && lt == 0) {
        mbar_expect_tx(bar, (uint32_t)(G4::PLANLEN * sizeof(float2)));
        bulk_g2s(smem4 + G4::PLAN2, p.plan, (uint32_t)(G4::PLANLEN * sizeof(float2)), bar);
        if ((int)blockIdx.x < p.ntiles) request_tile(blockIdx.x);
    }
    const float sgn = (t & 1) ? -1.0f : 1.0f;
    float2 u = make_float2(1.f, 0.f);
    if (HALF) { float sn, cs; sincospif(-(float)t / (float)L, &sn, &cs); u = make_float2(cs, sn); }   // w_2L^t = exp(-i pi t / L)
    mbar_wait(bar, 0);   // plan
    int it = 0;
    for (int w = blockIdx.x; w < p.ntiles; w += gridDim.x, ++it) {
        const int fb = w / G2::TILES, tile = w - fb * G2::TILES;
        auto sync = [&]() { gsync(); };
        P2 v[16];
        {
            float4 x[16];   // (col, col + 1) x (re, im)
            mbar_wait(bar + 1, it & 1);
            const float4* __restrict__ sg = stage + lt;   // ((n*NT + t)*2 + cp)
#pragma unroll
            for (int n = 0; n < 16; ++n) x[n] = sg[n * NT * 2];
            // lanes = the two columns; HALF 1 multiplies both by w_32^n (the n-dependent part of the input ramp)
#define PB_LANES2(n)                                                                                              \
            if (HALF == 0) v[n] = {make_float2(x[n].x, x[n].z), make_float2(x[n].y, x[n].w)};                          \
            else {                                                                                                     \
                const P2 a_ = make_lanes<INV, n>(make_float2(x[n].x, x[n].y)), b_ = make_lanes<INV, n>(make_float2(x[n].z, x[n].w)); \
                v[n] = {make_float2(a_.re.y, b_.re.y), make_float2(a_.im.y, b_.im.y)};                                 \
            }
            PB_LANES2(0) PB_LANES2(1) PB_LANES2(2) PB_LANES2(3) PB_LANES2(4) PB_LANES2(5) PB_LANES2(6) PB_LANES2(7)
            PB_LANES2(8) PB_LANES2(9) PB_LANES2(10) PB_LANES2(11) PB_LANES2(12) PB_LANES2(13) PB_LANES2(14) PB_LANES2(15)
#undef PB_LANES2
            __syncwarp();
            if ((threadIdx.x & 31) == 0) {   // this warp holds its inputs: one of 16 releases of the staging area per tile;
                __threadfence_block();       // the LAST warp to release it requests the next tile on the spot
                const unsigned int n = atomicAdd(released, 1u) + 1u;
                __threadfence_block();
                if (n == (unsigned int)(it + 1) * (4 * NT / 32) && w + (int)gridDim.x < p.ntiles) {
                    fence_proxy_async();
                    request_tile(w + gridDim.x);
                }
            }
        }
        fft_two_stages_u<L, INV, HALF>(v, t, S, plan + G4::TW1, plan + G4::TW2, u, sync);
        fft_last_stage_load<L, INV>(v, t, S);
        sync();   // this group's exchange buffers are free for its next tile
#pragma unroll
        for (int g = 0; g < G::GI; ++g) dftR<G::R3, INV>(v + g * G::R3);
        // tile-major store: element (plane, j, tile, c) at ((plane*L/4 + j/4) * TILES + tile) * 16 + (j%4)*4 + c ; c = 2 cp
        float4* __restrict__ dst = reinterpret_cast<float4*>(
            p.tmp + fb * (2LL * L * L) + (long long)HALF * L * L + ((long long)(t >> 2) * G2::TILES + tile) * 16 + (t & 3) * 4 + 2 * cp);
#pragma unroll
        for (int g = 0; g < G::GI; ++g)
#pragma unroll
            for (int kk = 0; kk < G::R3; ++kk) {
                const P2 y = v[g * G::R3 + kk];
                const long long o = (long long)((g * NT + 256 * kk) >> 2) * (G2::TILES * 8);   // float4 units
                // (-dir*i)^k with k = 2j + HALF; j has the parity of t.  HALF 1: times (-dir*i): forward (-im, re), inverse (im, -re)
                float4 q;
                if (HALF == 0) q = make_float4(sgn * y.re.x, sgn * y.im.x, sgn * y.re.y, sgn * y.im.y);
                else q = INV ? make_float4(sgn * y.im.x, -sgn * y.re.x, sgn * y.im.y, -sgn * y.re.y)
                             : make_float4(-sgn * y.im.x, sgn * y.re.x, -sgn * y.im.y, sgn * y.re.y);
                st_hint(dst + o, q, pol_tmp);
            }
    }
}

template <int L, bool INV>
__global__ void __launch_bounds__(Geo4<L>::THREADS) focus_col4_kernel(const __grid_constant__ CUtensorMap in_map, const FocusParams p) {
    using G = Geo<L>;
    using G2 = Geo2<L>;
    using G4 = Geo4<L>;
    extern __shared__ __align__(128) float4 smem4[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(smem4) + G4::BAR_OFF);   // [0] plan [1] tile full [2] tile free
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        *reinterpret_cast<unsigned int*>(bar + 2) = 0u;   // release counter of the staging area
        mbar_fence_init();
    }
    __syncthreads();
    const int grp = threadIdx.x / (2 * G::NT);
    if (grp == 0) focus_col4_group<L, INV, 0>(in_map, p, smem4, bar);
    else focus_col4_group<L, INV, 1>(in_map, p, smem4, bar);
}

template <int L, bool INV>
__global__ void __launch_bounds__(4 * L / 16) focus_row4_kernel(const __grid_constant__ CUtensorMap tmp_map, const FocusParams p) {
    using G = Geo<L>;
    using G2 = Geo2<L>;
    using G4 = Geo4<L>;
    using R4 = GeoR4<L>;
    constexpr int NT = G::NT, R3 = G::R3, GI = G::GI;
    constexpr uint32_t ROW_BYTES = L * sizeof(float2);
    extern __shared__ __align__(128) unsigned char smraw[];
    const int grp = threadIdx.x / NT, t = threadIdx.x - grp * NT;
    float4* S = reinterpret_cast<float4*>(smraw + grp * R4::GROUP);      // this group's exchange buffer
    float2* inb = reinterpret_cast<float2*>(S + G::SBUF);                 // ... and L-element input row
    const float2* __restrict__ plan = reinterpret_cast<const float2*>(smraw + R4::PLAN_OFF);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smraw + R4::BAR_OFF);   // [0] plan, [1 + grp] row of group grp
    uint64_t* bar = bars + 1 + grp;
    // the intermediate is dead after this read, the output is not read again here: both evict_first
    const uint64_t pol_tmp = l2_policy(1), pol_out = l2_policy(1);
    auto request_row = [&](int R) {   // one thread: gather intermediate row R = (field, plane, j) into `inb`
        const int fb = R / (2 * L), rf = R - fb * (2 * L);
        const int ph = rf / L, j = rf - ph * L;
        const int grow = (fb * 2 + ph) * (L / 4) + (j >> 2);
        mbar_expect_tx(bar, ROW_BYTES);
#pragma unroll
        for (int b = 0; b < G2::NBOX_ROW; ++b) tma_load_4d(inb + b * G2::BOXT * 4, &tmp_map, 0, j & 3, b * G2::BOXT, grow, bar, pol_tmp);
    };
    int r = blockIdx.x * 4 + grp;
    const int rstep = gridDim.x * 4;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 5; ++i) mbar_init(bars + i, 1);
        mbar_fence_init();
        mbar_expect_tx(bars, (uint32_t)(G4::PLANLEN * sizeof(float2)));
        bulk_g2s(smraw + R4::PLAN_OFF, p.plan, (uint32_t)(G4::PLANLEN * sizeof(float2)), bars);
    }
    __syncthreads();
    if (t == 0 && r < p.nrows) request_row(r);
    const SyncGroup gsync{1 + grp, NT};
    float2 u;
    { float sn, cs; sincospif(-(float)t / (float)L, &sn, &cs); u = make_float2(cs, sn); }   // w_2L^t
    const float sgn = ((t & 1) ? -1.0f : 1.0f) * p.scale;
    mbar_wait(bars, 0);
    for (int it = 0; r < p.nrows; ++it, r += rstep) {
        P2 v[16];
        mbar_wait(bar, it & 1);
        {
            const float2* __restrict__ row = inb + t;
#define PB_X(n) row[(n) * NT]
            PB_MAKE_LANES_16(v, INV, PB_X)
#undef PB_X
        }
        const int rn = r + rstep;
        // ---- stage 1
        dft16<INV>(v);
        v[0] = mul_tw<INV>(v[0], make_float4(1.0f, u.x, 0.0f, u.y));
#pragma unroll
        for (int k = 1; k < 16; ++k) {
            const float2 w = plan[G4::TW1 + k * NT + t];
            const float2 wb = make_float2(fmaf(w.x, u.x, -w.y * u.y), fmaf(w.x, u.y, w.y * u.x));
            v[k] = mul_tw<INV>(v[k], make_float4(w.x, wb.x, w.y, wb.y));
        }
        {
            float4* __restrict__ d = S + t * 17;
#pragma unroll
            for (int k = 0; k < 16; ++k) d[k] = pack(v[k]);
        }
        gsync();   // every thread of the group holds its inputs in registers: the row buffer is free
        if (t == 0 && rn < p.nrows) {
            fence_proxy_async();
            request_row(rn);
        }
        {
            const float4* __restrict__ s4 = S + pad16(t);
#pragma unroll
            for (int n = 0; n < 16; ++n) v[n] = unpack(s4[n * (NT + NT / 16)]);
        }
        gsync();
        // ---- stage 2
        dft16<INV>(v);
        {
            const int m = t >> 4, a = t & 15;
#pragma unroll
            for (int k = 1; k < 16; ++k) {
                const float2 w = plan[G4::TW2 + (k - 1) * (NT / 16) + m];
                v[k] = mul_tw<INV>(v[k], make_float4(w.x, w.x, w.y, w.y));
            }
            float4* __restrict__ d = S + m * 272 + a;
#pragma unroll
            for (int k = 0; k < 16; ++k) d[17 * k] = pack(v[k]);
        }
        gsync();
        fft_last_stage_load<L, INV>(v, t, S);
        gsync();  // exchange buffer is free for the next row
#pragma unroll
        for (int g = 0; g < GI; ++g) dftR<R3, INV>(v + g * R3);
        const int fb = r / (2 * L), rf = r - fb * (2 * L);   // field of the batch, row within its [2][L] planes
        const int phs = rf / L, rr = rf - phs * L;
        const int orow = (2 * rr + phs + L) & (2 * L - 1);  // fftshift along y
        if (p.out_kind == PB_OUT_COMPLEX) {
            float4* __restrict__ dst = reinterpret_cast<float4*>(reinterpret_cast<float2*>(p.out) + fb * p.out_bs + (long long)orow * p.out_ld);
#pragma unroll
            for (int g = 0; g < GI; ++g)
#pragma unroll
                for (int kk = 0; kk < R3; ++kk) {
                    const int j = t + g * NT + 256 * kk;
                    const P2 y = v[g * R3 + kk];
                    const float4 o = INV ? make_float4(sgn * y.re.x, sgn * y.im.x, sgn * y.im.y, -sgn * y.re.y)
                                         : make_float4(sgn * y.re.x, sgn * y.im.x, -sgn * y.im.y, sgn * y.re.y);
                    st_hint(dst + ((j + L / 2) & (L - 1)), o, pol_out);
                }
        } else {
            float2* __restrict__ dst = reinterpret_cast<float2*>(reinterpret_cast<float*>(p.out) + fb * p.out_bs + (long long)orow * p.out_ld);
            const float2 s2 = make_float2(p.scale * p.scale, p.scale * p.scale);
            const float2 wgt = make_float2(p.weight, p.weight);
#pragma unroll
            for (int g = 0; g < GI; ++g)
#pragma unroll
                for (int kk = 0; kk < R3; ++kk) {
                    const int j = t + g * NT + 256 * kk;
                    const P2 y = v[g * R3 + kk];
                    float2 I = __fmul2_rn(s2, __ffma2_rn(y.re, y.re, __fmul2_rn(y.im, y.im)));
                    float2* q = dst + ((j + L / 2) & (L - 1));
                    if (p.out_kind == PB_OUT_ACCUMULATE) I = __ffma2_rn(wgt, I, ld_stream(q));
                    st_hint(q, I, pol_out);
                }
        }
    }
}


// plan table, see Geo<L>
template <int L>
int get_focus_plan(Handle* h, const float4** out) {
    using G = Geo<L>;
    TwKey key{L, PB_C64, 11};
    auto it = h->tables.find(key);
    if (it != h->tables.end()) { *out = reinterpret_cast<const float4*>(it->second); return PB_OK; }
    auto w = [&](long long num, long long den) {  // exp(-2 pi i num/den), argument reduced exactly
        num %= den;
        const double a = -2.0 * 3.14159265358979323846 * (double)num / (double)den;
        return std::complex<double>(cos(a), sin(a));
    };
    std::vector<float4> tab(G::PLAN);
    for (int k = 0; k < 16; ++k)
        for (int t = 0; t < G::NT; ++t) {
            const std::complex<double> a = w((long long)t * k, L), b = w((long long)t * (2 * k + 1), 2 * L);
            tab[G::TW1 + k * G::NT + t] = make_float4((float)a.real(), (float)b.real(), (float)a.imag(), (float)b.imag());
        }
    for (int k = 1; k < 16; ++k)
        for (int m = 0; m < G::NT / 16; ++m) {
            const std::complex<double> a = w(16LL * m * k, L);
            tab[G::TW2 + (k - 1) * (G::NT / 16) + m] = make_float4((float)a.real(), (float)a.real(), (float)a.imag(), (float)a.imag());
        }
    void* d = nullptr;
    PB_CUDA(h, cudaMalloc(&d, tab.size() * sizeof(float4)));
    PB_CUDA(h, cudaMemcpy(d, tab.data(), tab.size() * sizeof(float4), cudaMemcpyHostToDevice));
    h->tables[key] = d;
    *out = reinterpret_cast<const float4*>(d);
    return PB_OK;
}


template <int L, bool INV>
int launch_focus(Handle* h, FocusParams p, int batch, cudaStream_t st) {
    using G = Geo<L>;
    constexpr int T = 4;
    const size_t smem_col = (size_t)(T * (G::SBUF + 2) + G::PLAN) * sizeof(float4) + 2 * sizeof(uint64_t);
    const size_t smem_row = (size_t)G::SBUF * sizeof(float4) + (size_t)L * sizeof(float2) + 2 * sizeof(uint64_t);
    // Resident row CTAs per SM: as many as leave >= 64 KB of the unified L1/shared array as L1 -- the 34 KB twiddle plan is
    // re-read by every line and must hit there.  (Left to itself the driver picks the 228 KB carve-out and the plan
    // streams from L2 at ~300 cycles a load.)
    const size_t unified = 256 * 1024, l1_keep = 64 * 1024;
    const int row_ctas = std::max(1, (int)((unified - l1_keep) / (smem_row + 1024)));
    PB_TRY(set_smem_attrs(h, focus_col_kernel<L, INV, T>, smem_col, 1));
    PB_TRY(set_smem_attrs(h, focus_row_kernel<L, INV>, smem_row, row_ctas));
    PB_TRY(get_focus_plan<L>(h, &p.plan));
    p.nrows = batch * 2 * L;
    focus_col_kernel<L, INV, T><<<dim3(L / T, batch), T * G::NT, smem_col, st>>>(p);
    PB_LAUNCH_CHECK(h);
    focus_row_kernel<L, INV><<<std::min(h->sm_count * row_ctas, p.nrows), L / 16, smem_row, st>>>(p);
    PB_LAUNCH_CHECK(h);
    return PB_OK;
}

}  // namespace

// ---- TMA descriptors, cached in the handle by (base pointer, geometry) -----------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_map_c64(Handle* h, const MapKey& key, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                const cuuint32_t* box, const CUtensorMap** out) {
    auto it = h->maps.find(key);
    if (it != h->maps.end()) { *out = &it->second; return PB_OK; }
    static EncodeTiledFn fn = nullptr;   // a driver entry point: process-wide, not per device
    if (!fn) {
        cudaDriverEntryPointQueryResult q;
        void* f = nullptr;
        PB_CUDA(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q));
        if (!f || q != cudaDriverEntryPointSuccess) return fail(h, PB_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        fn = reinterpret_cast<EncodeTiledFn>(f);
    }
    if (h->maps.size() > 256) h->maps.clear();
    CUtensorMap m;
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_UINT64, (cuuint32_t)rank, const_cast<void*>(key.base), dims, strides_bytes, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, PB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    *out = &(h->maps[key] = m);
    return PB_OK;
}

namespace {


template <int L, bool INV>
int launch_focus2(Handle* h, FocusParams p, int batch, cudaStream_t st) {
    using G = Geo<L>;
    using G2 = Geo2<L>;
    using G4 = Geo4<L>;
    using R4 = GeoR4<L>;
    auto colk = focus_col4_kernel<L, INV>;
    auto rowk = focus_row4_kernel<L, INV>;
    PB_TRY(set_smem_attrs(h, colk, G4::SMEM, 1));
    PB_TRY(set_smem_attrs(h, rowk, R4::SMEM, 1));
    const float2* plan = nullptr;
    PB_TRY(get_col4_plan<L>(h, &plan));
    p.plan = reinterpret_cast<const float4*>(plan);   // both kernels read the float2 plan of Geo4
    p.nrows = batch * 2 * L;
    p.ntiles = batch * G2::TILES;
    // (descriptors are copied out at once: the handle's cache may be flushed by the next lookup)
    const CUtensorMap* map = nullptr;
    CUtensorMap in_m, tmp_m;
    {   // intermediate: [group = (field, plane, j/4)][tile][j%4][c]
        const cuuint64_t dims[4] = {4, 4, (cuuint64_t)G2::TILES, (cuuint64_t)batch * 2 * (L / 4)};
        const cuuint64_t str[3] = {32, 128, (cuuint64_t)G2::TILES * 128};
        const cuuint32_t box[4] = {4, 1, (cuuint32_t)G2::BOXT, 1};
        PB_TRY(get_map_c64(h, MapKey{p.tmp, 1, L, batch, 0, 0}, 4, dims, str, box, &map));
        tmp_m = *map;
    }
    {   // input: (field, row, column) complex64; box = one 4-column run of 256 rows
        const cuuint64_t dims[3] = {(cuuint64_t)L, (cuuint64_t)L, (cuuint64_t)batch};
        const cuuint64_t str[2] = {(cuuint64_t)p.in_ld * 8, (cuuint64_t)(batch > 1 ? p.in_bs : (long long)L * p.in_ld) * 8};
        const cuuint32_t box[3] = {4, (cuuint32_t)G2::BOXR, 1};
        PB_TRY(get_map_c64(h, MapKey{p.in, 2, L, batch, p.in_ld, batch > 1 ? p.in_bs : 0}, 3, dims, str, box, &map));
        in_m = *map;
    }
    // column pass: one CTA per SM walks the tiles of all fields of the launch
    colk<<<std::min(h->sm_count, p.ntiles), G4::THREADS, G4::SMEM, st>>>(in_m, p);
    PB_LAUNCH_CHECK(h);
    // row pass: one CTA per SM, four line groups per CTA, plan in shared memory
    rowk<<<std::min(h->sm_count, (p.nrows + 3) / 4), 4 * G::NT, R4::SMEM, st>>>(tmp_m, p);
    PB_LAUNCH_CHECK(h);
    return PB_OK;
}

// =====================================================================================================
// Register-engine version of the generic axis pass (AxisPass semantics, complex64 in/out) for
// L in {1024, 2048, 4096}: two lines per thread group ride the two packed lanes.  ROWS: one CTA = 2 rows;
// COLS: one CTA = TP pairs of adjacent columns.  Used by pb_fft2 / pb_axis_dft / pb_angular_spectrum for
// every power-of-two pass the focus kernels above do not cover (CZT, FFTDFT, free space, psf -> otf).
// =====================================================================================================
__device__ __forceinline__ float2 cmul_s(float2 a, float2 b, int conj) {
    return conj ? make_float2(fmaf(a.x, b.x, a.y * b.y), fmaf(a.y, b.x, -a.x * b.y))
                : make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}

// DENSE: the whole line is populated and kept -- no pad window, no rotation, no crop, an even number of lines, complex
// input (free-space steps at Q = 1, plain transforms): the per-element window tests and index arithmetic of the general
// form (about as many integer instructions as there are floating-point ones) compile away.
template <int L, bool INV, bool COLS, int TP, bool RT, bool PM, bool DENSE>
__global__ void __launch_bounds__((COLS ? TP : 1) * L / 16, (RT && (!COLS || TP == 1) && L >= 4096) ? 2 : 0) axis_reg_kernel(const AxisPass p, const float2* __restrict__ tw1,
                                                                            const float2* __restrict__ tw2) {
    using G = Geo<L>;
    constexpr int NT = G::NT;
    extern __shared__ __align__(16) float4 smem4[];
    const int c = COLS ? threadIdx.x % TP : 0, t = COLS ? threadIdx.x / TP : threadIdx.x;
    const int b0 = (blockIdx.x * (COLS ? TP : 1) + c) * 2;   // lines b0 (lane A) and b0 + 1 (lane B)
    const bool hasA = DENSE || b0 < p.nb, hasB = DENSE || b0 + 1 < p.nb;
    // column passes: a thread's two lines are adjacent columns, i.e. 16 contiguous bytes per sample -- one 128-bit access
    // instead of two 64-bit ones (half the LSU instructions and sector requests of the pass: `lg_throttle` was its second
    // stall).  vin / vout: unit line stride, even pitch, 16-byte aligned base, both lines present (host: dispatch_axis_reg).
    const bool vin = COLS && (DENSE || ((p.batch_contiguous & 2) && hasB));
    const bool vout = COLS && (DENSE || ((p.batch_contiguous & 4) && hasB));
    const float2* __restrict__ in = reinterpret_cast<const float2*>(p.in);
    const float2* __restrict__ pre_e = reinterpret_cast<const float2*>(p.pre_e);
    const float2* __restrict__ pre_b = reinterpret_cast<const float2*>(p.pre_b);
    float2 pbA = make_float2(1.f, 0.f), pbB = pbA;
    if (pre_b) { if (hasA) pbA = pre_b[b0]; if (hasB) pbB = pre_b[b0 + 1]; }
    P2 v[16];
#pragma unroll
    for (int n = 0; n < 16; ++n) {
        const int j = n * NT + t;
        int li = j;
        if (!DENSE) {
            int pp = j + p.rot_in;
            if (pp >= L) pp -= L;
            li = pp - p.in_off;
        }
        float2 xa = make_float2(0.f, 0.f), xb = xa;
        if (DENSE || (li >= 0 && li < p.n_in)) {
            const long long o = (long long)b0 * p.ibs + (long long)li * p.ies;
            if (!DENSE && p.in_kind == PB_IN_REAL) {   // real field (the PSF going to transform_psf): imaginary part 0
                const float* __restrict__ inr = reinterpret_cast<const float*>(p.in);
                if (hasA) xa.x = __ldg(inr + o);
                if (hasB) xb.x = __ldg(inr + o + p.ibs);
            } else if (vin) {
                const float4 q = ld_stream4(reinterpret_cast<const float4*>(in + o));
                xa = make_float2(q.x, q.y); xb = make_float2(q.z, q.w);
            } else {
                if (hasA) xa = ld_stream(in + o);
                if (hasB) xb = ld_stream(in + o + p.ibs);
            }
            if (pre_e) { const float2 w = pre_e[j - p.pre_off]; xa = cmul_s(xa, w, p.pre_e_conj); xb = cmul_s(xb, w, p.pre_e_conj); }
            if (pre_b) { xa = cmul_s(xa, pbA, p.pre_b_conj); xb = cmul_s(xb, pbB, p.pre_b_conj); }
        }
        v[n] = {make_float2(xa.x, xb.x), make_float2(xa.y, xb.y)};
    }
    if (PM) {
        // full-matrix pre-multiplier (the phase screen of a free-space chain), same access pattern as the input.  A loop of
        // its own: the 32 loads are independent of the input loads above and of each other, so they overlap, and the
        // product is one packed complex multiply per point (lane A x mA, lane B x mB).
        const float2* __restrict__ pm = reinterpret_cast<const float2*>(p.pre_mat);
#pragma unroll
        for (int n = 0; n < 16; ++n) {
            const int j = n * NT + t;
            int li = j;
            if (!DENSE) {
                int pp = j + p.rot_in;
                if (pp >= L) pp -= L;
                li = pp - p.in_off;
            }
            if (DENSE || (li >= 0 && li < p.n_in)) {
                const long long om = (long long)b0 * p.pmi_bs + (long long)li * p.pmi_es;
                float2 ma = make_float2(1.f, 0.f), mb = ma;
                if (hasA) ma = ld_stream(pm + om);
                if (hasB) mb = ld_stream(pm + om + p.pmi_bs);
                const float4 w = make_float4(ma.x, mb.x, ma.y, mb.y);
                v[n] = p.pre_mat_conj ? mul_tw<true>(v[n], w) : mul_tw<false>(v[n], w);
            }
        }
    }
    // TP interleaved lines per CTA: consecutive exchange buffers are offset by 32 / TP banks (8 / TP float4 of padding), so
    // that the 8 threads of a 128-bit wavefront (8 / TP consecutive t  x  TP lines) cover all 32 banks
    float4* S = smem4 + c * (G::SBUF + 8 / (COLS ? TP : 1) % 8);
    fft_two_stages<L, INV, 2>(v, t, S, tw1, tw2, SyncCta(), SyncCta());
    fft_last_stage_load<L, INV>(v, t, S);
#pragma unroll
    for (int g = 0; g < G::GI; ++g) dftR<G::R3, INV>(v + g * G::R3);
    const float2* __restrict__ post_e = reinterpret_cast<const float2*>(p.post_e);
    const float2* __restrict__ post_b = reinterpret_cast<const float2*>(p.post_b);
    float2 qbA = make_float2(1.f, 0.f), qbB = qbA;
    if (post_b) { if (hasA) qbA = post_b[b0]; if (hasB) qbB = post_b[b0 + 1]; }
    const float scale = (float)p.scale;
    float2* __restrict__ out = reinterpret_cast<float2*>(p.out);
    if (RT) {
        // Round trip (free-space propagation along this axis): the spectrum is multiplied by the transfer
        // factors post_e[k] * post_b[line] and transformed straight back.  The forward pass leaves thread t
        // with X[t + NT*(g + GI*kk)], which IS the inverse pass's stage-1 register layout (n = g + GI*kk):
        // the data never leaves the registers between the two transforms.
        P2 w[16];
#pragma unroll
        for (int g = 0; g < G::GI; ++g)
#pragma unroll
            for (int kk = 0; kk < G::R3; ++kk) {
                const int k = t + g * NT + 256 * kk;
                const P2 y = v[g * G::R3 + kk];
                float2 ya = make_float2(y.re.x, y.im.x), yb = make_float2(y.re.y, y.im.y);
                if (post_e) { const float2 m = post_e[k - p.post_off]; ya = cmul_s(ya, m, p.post_e_conj); yb = cmul_s(yb, m, p.post_e_conj); }
                if (post_b) { ya = cmul_s(ya, qbA, p.post_b_conj); yb = cmul_s(yb, qbB, p.post_b_conj); }
                w[g + G::GI * kk] = {make_float2(ya.x, yb.x), make_float2(ya.y, yb.y)};
            }
        __syncthreads();   // all last-stage reads of S are done before the inverse pass overwrites it
        fft_two_stages<L, !INV, 2>(w, t, S, tw1, tw2, SyncCta(), SyncCta());
        fft_last_stage_load<L, !INV>(w, t, S);
#pragma unroll
        for (int g = 0; g < G::GI; ++g) dftR<G::R3, !INV>(w + g * G::R3);
        if (COLS && p.out_kind != PB_OUT_COMPLEX && (p.batch_contiguous & 8) && hasB) {
            // |.|^2 of a column pass onto a real plane, both columns of the thread as one aligned float2.  Three passes over
            // the thread's 16 samples -- form the intensities, read ALL the previous plane values, then store -- because a
            // read-modify-write per sample serialises: the compiler may not move sample i+1's load above sample i's store to
            // the same array, and sixteen DRAM latencies in a row were the C4 column pass's top stall (long_scoreboard 8.2).
            float* __restrict__ outr = reinterpret_cast<float*>(p.out);
            const float s2 = scale * scale, wgt = (float)p.weight;
            auto out_q = [&](int j) -> int {   // output sample of transform index j, or -1 when it is cropped away
                if (DENSE) return j;
                int q = j - p.crop_off + p.rot_out;
                if (q < 0) q += L;
                if (q >= L) q -= L;
                return q < p.n_out ? q : -1;
            };
            float2 I[16];
#pragma unroll
            for (int g = 0; g < G::GI; ++g)
#pragma unroll
                for (int kk = 0; kk < G::R3; ++kk) {
                    const int q = out_q(t + g * NT + 256 * kk);
                    const P2 y = w[g * G::R3 + kk];
                    float2 ya = make_float2(y.re.x, y.im.x), yb = make_float2(y.re.y, y.im.y);
                    if (p.post_e2 && q >= 0) {
                        const float2 m = reinterpret_cast<const float2*>(p.post_e2)[q];
                        ya = cmul_s(ya, m, p.post_e2_conj); yb = cmul_s(yb, m, p.post_e2_conj);
                    }
                    I[g * G::R3 + kk] = make_float2(s2 * fmaf(ya.x, ya.x, ya.y * ya.y), s2 * fmaf(yb.x, yb.x, yb.y * yb.y));
                }
            if (p.out_kind == PB_OUT_ACCUMULATE) {
#pragma unroll
                for (int g = 0; g < G::GI; ++g)
#pragma unroll
                    for (int kk = 0; kk < G::R3; ++kk) {
                        const int q = out_q(t + g * NT + 256 * kk);
                        if (q < 0) continue;
                        const float2 prev = *reinterpret_cast<const float2*>(outr + (long long)b0 * p.obs + (long long)q * p.oes);
                        float2& v2 = I[g * G::R3 + kk];
                        v2 = make_float2(fmaf(wgt, v2.x, prev.x), fmaf(wgt, v2.y, prev.y));
                    }
            }
#pragma unroll
            for (int g = 0; g < G::GI; ++g)
#pragma unroll
                for (int kk = 0; kk < G::R3; ++kk) {
                    const int q = out_q(t + g * NT + 256 * kk);
                    if (q < 0) continue;
                    *reinterpret_cast<float2*>(outr + (long long)b0 * p.obs + (long long)q * p.oes) = I[g * G::R3 + kk];
                }
            return;
        }
#pragma unroll
        for (int g = 0; g < G::GI; ++g)
#pragma unroll
            for (int kk = 0; kk < G::R3; ++kk) {
                const int j = t + g * NT + 256 * kk;
                int q = j;
                if (!DENSE) {
                    q = j - p.crop_off + p.rot_out;
                    if (q < 0) q += L;
                    if (q >= L) q -= L;
                    if (q >= p.n_out) continue;
                }
                const P2 y = w[g * G::R3 + kk];
                float2 ya = make_float2(y.re.x, y.im.x), yb = make_float2(y.re.y, y.im.y);
                if (p.post_e2) {  // final multiplier, indexed by the output sample (the CZT's a(m)*phase(m))
                    const float2 m = reinterpret_cast<const float2*>(p.post_e2)[q];
                    ya = cmul_s(ya, m, p.post_e2_conj); yb = cmul_s(yb, m, p.post_e2_conj);
                }
                const long long o = (long long)b0 * p.obs + (long long)q * p.oes;
                if (p.out_kind == PB_OUT_COMPLEX) {
                    if (vout) st_stream(reinterpret_cast<float4*>(out + o), make_float4(ya.x * scale, ya.y * scale, yb.x * scale, yb.y * scale));
                    else {
                        if (hasA) st_stream(out + o, make_float2(ya.x * scale, ya.y * scale));
                        if (hasB) st_stream(out + o + p.obs, make_float2(yb.x * scale, yb.y * scale));
                    }
                } else {   // |.|^2 (or weight * |.|^2 added to the plane): the complex field is never written
                    float* __restrict__ outr = reinterpret_cast<float*>(p.out);
                    const float s2 = scale * scale, wgt = (float)p.weight;
                    float ia = s2 * fmaf(ya.x, ya.x, ya.y * ya.y), ib = s2 * fmaf(yb.x, yb.x, yb.y * yb.y);
                    if (p.out_kind == PB_OUT_ACCUMULATE) {
                        if (hasA) ia = fmaf(wgt, ia, outr[o]);
                        if (hasB) ib = fmaf(wgt, ib, outr[o + p.obs]);
                    }
                    if (hasA) outr[o] = ia;
                    if (hasB) outr[o + p.obs] = ib;
                }
            }
        return;
    }
#pragma unroll
    for (int g = 0; g < G::GI; ++g)
#pragma unroll
        for (int kk = 0; kk < G::R3; ++kk) {
            const int k = t + g * NT + 256 * kk;
            int q = k;
            if (!DENSE) {
                q = k - p.crop_off + p.rot_out;
                if (q < 0) q += L;
                if (q >= L) q -= L;
                if (q >= p.n_out) continue;
            }
            const P2 y = v[g * G::R3 + kk];
            float2 ya = make_float2(y.re.x, y.im.x), yb = make_float2(y.re.y, y.im.y);
            if (post_e) { const float2 w = post_e[k - p.post_off]; ya = cmul_s(ya, w, p.post_e_conj); yb = cmul_s(yb, w, p.post_e_conj); }
            if (post_b) { ya = cmul_s(ya, qbA, p.post_b_conj); yb = cmul_s(yb, qbB, p.post_b_conj); }
            const long long o = (long long)b0 * p.obs + (long long)q * p.oes;
            if (vout) st_stream(reinterpret_cast<float4*>(out + o), make_float4(ya.x * scale, ya.y * scale, yb.x * scale, yb.y * scale));
            else {
                if (hasA) st_stream(out + o, make_float2(ya.x * scale, ya.y * scale));
                if (hasB) st_stream(out + o + p.obs, make_float2(yb.x * scale, yb.y * scale));
            }
        }
}

// plain twiddle tables: tw1[(k-1)*NT + t] = w_L^(t k), tw2[(k-1)*NT/16 + m] = w_L^(16 m k), contiguous
template <int L>
int get_plain_plan(Handle* h, const float2** tw1, const float2** tw2) {
    using G = Geo<L>;
    TwKey key{L, PB_C64, 12};
    const float2* base = nullptr;
    auto it = h->tables.find(key);
    if (it != h->tables.end()) base = reinterpret_cast<const float2*>(it->second);
    else {
        std::vector<std::complex<double>> tab(15 * G::NT + 15 * (G::NT / 16));
        auto w = [&](long long num, long long den) {
            num %= den;
            const double a = -2.0 * 3.14159265358979323846 * (double)num / (double)den;
            return std::complex<double>(cos(a), sin(a));
        };
        for (int k = 1; k < 16; ++k)
            for (int t = 0; t < G::NT; ++t) tab[(k - 1) * G::NT + t] = w((long long)t * k, L);
        for (int k = 1; k < 16; ++k)
            for (int m = 0; m < G::NT / 16; ++m) tab[15 * G::NT + (k - 1) * (G::NT / 16) + m] = w(16LL * m * k, L);
        const void* d = nullptr;
        PB_TRY(upload_table(h, key, tab, &d));
        base = reinterpret_cast<const float2*>(d);
    }
    *tw1 = base;
    *tw2 = base + 15 * G::NT;
    return PB_OK;
}

template <int L, bool INV, bool COLS, bool RT, bool PM = false, bool DENSE = false, int TPC = 2>
int launch_axis_reg(Handle* h, const AxisPass& p, cudaStream_t st) {
    using G = Geo<L>;
    constexpr int TP = COLS ? TPC : 1;
    const size_t smem = (size_t)TP * (G::SBUF + 8 / TP % 8) * sizeof(float4);
    if (attr_needed(h, reinterpret_cast<const void*>(axis_reg_kernel<L, INV, COLS, TP, RT, PM, DENSE>))) {
        PB_CUDA(h, cudaFuncSetAttribute(axis_reg_kernel<L, INV, COLS, TP, RT, PM, DENSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // keep >= 64 KB of L1 for the twiddle tables (see launch_focus)
        const size_t unified = 256 * 1024, l1_keep = 64 * 1024;
        const int ctas = std::max<int>(1, (int)((unified - l1_keep) / (smem + 1024)));
        const int pct = (int)std::min<size_t>(100, ((size_t)ctas * (smem + 1024) * 100 + h->max_smem_optin - 1) / h->max_smem_optin);
        PB_CUDA(h, cudaFuncSetAttribute(axis_reg_kernel<L, INV, COLS, TP, RT, PM, DENSE>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    }
    const float2 *tw1 = nullptr, *tw2 = nullptr;
    PB_TRY(get_plain_plan<L>(h, &tw1, &tw2));
    const int lines_per_cta = 2 * TP;
    const int grid = (p.nb + lines_per_cta - 1) / lines_per_cta;
    axis_reg_kernel<L, INV, COLS, TP, RT, PM, DENSE><<<grid, TP * G::NT, smem, st>>>(p, tw1, tw2);
    PB_LAUNCH_CHECK(h);
    return PB_OK;
}

template <int L>
int dispatch_axis_reg(Handle* h, const AxisPass& p0, cudaStream_t st) {
    AxisPass p = p0;
    const bool cols = p.batch_contiguous != 0;
    // 128-bit accesses of the column passes (two adjacent columns per thread): unit line stride, even pitch, aligned base
    const bool vec_in = cols && p.in_kind == PB_IN_COMPLEX && p.ibs == 1 && !(p.ies & 1) && !((uintptr_t)p.in & 15);
    const bool vec_out = cols && p.out_kind == PB_OUT_COMPLEX && p.obs == 1 && !(p.oes & 1) && !((uintptr_t)p.out & 15);
    const bool vec_int = cols && p.out_kind != PB_OUT_COMPLEX && p.obs == 1 && !(p.oes & 1) && !((uintptr_t)p.out & 7);
    if (cols) p.batch_contiguous = 1 | (vec_in ? 2 : 0) | (vec_out ? 4 : 0) | (vec_int ? 8 : 0);
    // the whole line populated and kept, lines in pairs, complex in: the index logic of the general kernel compiles away
    const bool dense = p.rot_in == 0 && p.in_off == 0 && p.n_in == L && p.crop_off == 0 && p.rot_out == 0 && p.n_out == L &&
                       !(p.nb & 1) && p.in_kind == PB_IN_COMPLEX && !p.post_e2 && p.pre_off == 0 && p.post_off == 0 &&
                       (!cols || (!(p.nb & 3) && vec_in && vec_out));
    if (p.pre_mat) {   // the screened first pass of a free-space step: rows, plain transform
        if (cols || p.roundtrip) return PB_ERR_UNSUPPORTED;
        if (dense) return p.dir < 0 ? launch_axis_reg<L, false, false, false, true, true>(h, p, st) : launch_axis_reg<L, true, false, false, true, true>(h, p, st);
        return p.dir < 0 ? launch_axis_reg<L, false, false, false, true>(h, p, st) : launch_axis_reg<L, true, false, false, true>(h, p, st);
    }
    if (dense && L >= 2048) {   // the free-space passes and plain transforms of the large configurations
        if (p.roundtrip) {
            if (cols) return p.dir < 0 ? launch_axis_reg<L, false, true, true, false, true>(h, p, st) : launch_axis_reg<L, true, true, true, false, true>(h, p, st);
        } else if (!cols) {
            return p.dir < 0 ? launch_axis_reg<L, false, false, false, false, true>(h, p, st) : launch_axis_reg<L, true, false, false, false, true>(h, p, st);
        } else {
            return p.dir < 0 ? launch_axis_reg<L, false, true, false, false, true>(h, p, st) : launch_axis_reg<L, true, true, false, false, true>(h, p, st);
        }
    }
    if (p.roundtrip) {
        if (p.dir < 0) return cols ? launch_axis_reg<L, false, true, true>(h, p, st) : launch_axis_reg<L, false, false, true>(h, p, st);
        return cols ? launch_axis_reg<L, true, true, true>(h, p, st) : launch_axis_reg<L, true, false, true>(h, p, st);
    }
    if (p.dir < 0) return cols ? launch_axis_reg<L, false, true, false>(h, p, st) : launch_axis_reg<L, false, false, false>(h, p, st);
    return cols ? launch_axis_reg<L, true, true, false>(h, p, st) : launch_axis_reg<L, true, false, false>(h, p, st);
}

}  // namespace

int try_tuned_axis_pass(Handle* h, const AxisPass& p, cudaStream_t st) {
    if (p.dtype != PB_C64 || p.in_kind == PB_IN_AMP_OPD) return PB_ERR_UNSUPPORTED;
    if (p.out_kind != PB_OUT_COMPLEX && !p.roundtrip) return PB_ERR_UNSUPPORTED;   // |.|^2 stores: round-trip epilogue only
    if (p.pre_e2 || (p.post_e2 && !p.roundtrip) || p.post_mat) return PB_ERR_UNSUPPORTED;
    if (p.Llog != p.L || (p.Llog_out != 0 && p.Llog_out != p.L)) return PB_ERR_UNSUPPORTED;
    // any batch: a single line (the kernel spectrum of a CZT plan, built per wavelength) takes 23 us on the generic
    // kernel's six synchronised radix-4 stages and a fraction of that here
    switch (p.L) {
        case 1024: return dispatch_axis_reg<1024>(h, p, st);
        case 2048: return dispatch_axis_reg<2048>(h, p, st);
        case 4096: return dispatch_axis_reg<4096>(h, p, st);
        default: return PB_ERR_UNSUPPORTED;
    }
}

// fields per launch pair: more than one evens out the tails (512 column tiles on 148 SMs = 3.46 waves at N = 2048).
// The intermediates of a group (64 MiB each at N = 2048) no longer fit L2 together and spill to HBM, which has the
// headroom: measured 87.3 / 78.8 / 76.7 / 75.7 us per field at 1 / 2 / 4 / 8.
constexpr int FOCUS_FIELDS_PER_LAUNCH = 8;

int try_tuned_fft2_batch(Handle* h, int dtype, const void* in, int in_kind, const void* amp, int amp_kind, double kturns,
                         int batch, long long in_bs, long long amp_bs, int ny, int nx, long long in_ld, int ky, int kx, int dir,
                         double scale, int shift_in, int shift_out, void* out, int out_kind, double weight, int oy, int ox,
                         long long out_ld, long long out_bs, cudaStream_t st) {
    if (dtype != PB_C64 || ny != nx || ky != 2 * ny || kx != 2 * nx || !shift_in || !shift_out || oy != ky || ox != kx)
        return PB_ERR_UNSUPPORTED;
    if (nx != 512 && nx != 1024 && nx != 2048) return PB_ERR_UNSUPPORTED;
    if (in_kind == PB_IN_REAL) return PB_ERR_UNSUPPORTED;
    if (out_kind == PB_OUT_COMPLEX ? (out_ld & 1) || (out_bs & 1) || ((uintptr_t)out & 15) : (out_ld & 1) || (out_bs & 1) || ((uintptr_t)out & 7))
        return PB_ERR_UNSUPPORTED;  // vector stores need aligned rows
    const int N = nx;
    // the v2 kernels take their input tiles by tensor TMA: complex input, 16-byte aligned base and even pitches (so that
    // every group's base stays aligned); everything else (the fused phase-screen input, odd pitches) runs the v1 kernels
    const bool tma_ok = in_kind == PB_IN_COMPLEX && !((uintptr_t)in & 15) && !(in_ld & 1) && !(in_bs & 1);
    const int per = std::min(batch, FOCUS_FIELDS_PER_LAUNCH);
    void* tmp = nullptr;
    PB_TRY(ensure_scratch(h, 0, (size_t)per * 2 * N * N * sizeof(float2), &tmp));
    const size_t in_elt = in_kind == PB_IN_COMPLEX ? sizeof(float2) : sizeof(float);
    const size_t amp_elt = amp_kind == PB_AMP_U8 ? 1 : sizeof(float);
    const size_t out_elt = out_kind == PB_OUT_COMPLEX ? sizeof(float2) : sizeof(float);
    for (int b0 = 0; b0 < batch; b0 += per) {
        const int nb = std::min(per, batch - b0);
        FocusParams p;
        p.in = reinterpret_cast<const char*>(in) + (size_t)b0 * in_bs * in_elt;
        p.in_kind = in_kind;
        p.amp = amp ? reinterpret_cast<const char*>(amp) + (size_t)b0 * amp_bs * amp_elt : nullptr;
        p.amp_kind = amp_kind; p.kturns = kturns; p.in_ld = in_ld;
        p.tmp = reinterpret_cast<float2*>(tmp);
        p.plan = nullptr;
        p.out = reinterpret_cast<char*>(out) + (size_t)b0 * out_bs * out_elt;
        p.out_ld = out_ld; p.out_kind = out_kind; p.scale = (float)scale; p.weight = (float)weight;
        p.nrows = 0; p.ntiles = 0;
        p.in_bs = in_bs; p.amp_bs = amp_bs; p.out_bs = out_bs;
        int rc;
        if (tma_ok) {
            if (dir < 0) rc = N == 512 ? launch_focus2<512, false>(h, p, nb, st) : N == 1024 ? launch_focus2<1024, false>(h, p, nb, st) : launch_focus2<2048, false>(h, p, nb, st);
            else rc = N == 512 ? launch_focus2<512, true>(h, p, nb, st) : N == 1024 ? launch_focus2<1024, true>(h, p, nb, st) : launch_focus2<2048, true>(h, p, nb, st);
        } else if (dir < 0) rc = N == 512 ? launch_focus<512, false>(h, p, nb, st) : N == 1024 ? launch_focus<1024, false>(h, p, nb, st) : launch_focus<2048, false>(h, p, nb, st);
        else rc = N == 512 ? launch_focus<512, true>(h, p, nb, st) : N == 1024 ? launch_focus<1024, true>(h, p, nb, st) : launch_focus<2048, true>(h, p, nb, st);
        if (rc != PB_OK) return rc;
    }
    return PB_OK;
}

int try_tuned_fft2(Handle* h, int dtype, const void* in, int in_kind, const void* amp, int amp_kind, double kturns,
                   int ny, int nx, long long in_ld, int ky, int kx, int dir, double scale, int shift_in, int shift_out,
                   void* out, int out_kind, double weight, int oy, int ox, long long out_ld, cudaStream_t st) {
    return try_tuned_fft2_batch(h, dtype, in, in_kind, amp, amp_kind, kturns, 1, 0, 0, ny, nx, in_ld, ky, kx, dir, scale,
                                shift_in, shift_out, out, out_kind, weight, oy, ox, out_ld, 0, st);
}


}  // namespace pb
