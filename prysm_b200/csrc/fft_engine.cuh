// Register-resident packed-lane FFT engine of the tuned kernels (fft_tuned.cu): radix-16 butterflies on
// two packed fp32 lanes, the two-exchange FFT_L skeleton, async-copy / TMA plumbing, and the geometry of the focus pipeline.
// Everything device-side lives in an anonymous namespace (each translation unit gets its own copy).
#pragma once
#include <algorithm>
#include "fft_tuned.cuh"

namespace pb {

// TMA descriptor (complex64 elements as UINT64), cached in the handle by (base pointer, geometry); defined in fft_tuned.cu
int get_map_c64(Handle* h, const MapKey& key, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                const cuuint32_t* box, const CUtensorMap** out);

namespace {

#define PB_SQRT1_2 0.70710678118654752440f
#define PB_C1_8 0.92387953251128675613f   // cos(pi/8)
#define PB_S1_8 0.38268343236508977173f   // sin(pi/8)

// two complex numbers (lane A, lane B), structure of arrays
struct P2 { float2 re, im; };

__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ P2 operator+(P2 a, P2 b) { return {__fadd2_rn(a.re, b.re), __fadd2_rn(a.im, b.im)}; }
__device__ __forceinline__ P2 operator-(P2 a, P2 b) { return {__fadd2_rn(a.re, neg2(b.re)), __fadd2_rn(a.im, neg2(b.im))}; }
// multiply by w4 = exp(-+ i pi/2):  -i forward, +i inverse
template <bool INV> __device__ __forceinline__ P2 mul_w4(P2 a) { return INV ? P2{neg2(a.im), a.re} : P2{a.im, neg2(a.re)}; }
// multiply both lanes by w = (c, -+ s)
template <bool INV> __device__ __forceinline__ P2 mul_cs(P2 a, float c, float s) {
    const float2 C = make_float2(c, c), S = make_float2(s, s);
    if (INV) return {__ffma2_rn(a.re, C, neg2(__fmul2_rn(a.im, S))), __ffma2_rn(a.im, C, __fmul2_rn(a.re, S))};
    return {__ffma2_rn(a.re, C, __fmul2_rn(a.im, S)), __ffma2_rn(a.im, C, neg2(__fmul2_rn(a.re, S)))};
}
// per-lane twiddle: w = (wre, wim) pairs as stored in the tables (forward sign); INV conjugates
template <bool INV> __device__ __forceinline__ P2 mul_tw(P2 a, float4 w) {
    const float2 wr = make_float2(w.x, w.y), wi = make_float2(w.z, w.w);
    if (INV) return {__ffma2_rn(a.re, wr, __fmul2_rn(a.im, wi)), __ffma2_rn(a.im, wr, neg2(__fmul2_rn(a.re, wi)))};
    return {__ffma2_rn(a.re, wr, neg2(__fmul2_rn(a.im, wi))), __ffma2_rn(a.im, wr, __fmul2_rn(a.re, wi))};
}

template <bool INV> __device__ __forceinline__ void dft2(P2& a, P2& b) {
    P2 s = a + b, d = a - b;
    a = s; b = d;
}
template <bool INV> __device__ __forceinline__ void dft4(P2& x0, P2& x1, P2& x2, P2& x3) {
    P2 s02 = x0 + x2, d02 = x0 - x2, s13 = x1 + x3, d13 = mul_w4<INV>(x1 - x3);
    x0 = s02 + s13; x2 = s02 - s13; x1 = d02 + d13; x3 = d02 - d13;
}
template <bool INV> __device__ __forceinline__ void dft8(P2* v) {
    P2 e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6];
    P2 o0 = v[1], o1 = v[3], o2 = v[5], o3 = v[7];
    dft4<INV>(e0, e1, e2, e3);
    dft4<INV>(o0, o1, o2, o3);
    o1 = mul_cs<INV>(o1, PB_SQRT1_2, PB_SQRT1_2);
    o2 = mul_w4<INV>(o2);
    o3 = mul_cs<INV>(o3, -PB_SQRT1_2, PB_SQRT1_2);
    v[0] = e0 + o0; v[4] = e0 - o0;
    v[1] = e1 + o1; v[5] = e1 - o1;
    v[2] = e2 + o2; v[6] = e2 - o2;
    v[3] = e3 + o3; v[7] = e3 - o3;
}
template <bool INV> __device__ __forceinline__ void dft16(P2* v) {
    P2 e[8], o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { e[i] = v[2 * i]; o[i] = v[2 * i + 1]; }
    dft8<INV>(e);
    dft8<INV>(o);
    o[1] = mul_cs<INV>(o[1], PB_C1_8, PB_S1_8);
    o[2] = mul_cs<INV>(o[2], PB_SQRT1_2, PB_SQRT1_2);
    o[3] = mul_cs<INV>(o[3], PB_S1_8, PB_C1_8);
    o[4] = mul_w4<INV>(o[4]);
    o[5] = mul_cs<INV>(o[5], -PB_S1_8, PB_C1_8);
    o[6] = mul_cs<INV>(o[6], -PB_SQRT1_2, PB_SQRT1_2);
    o[7] = mul_cs<INV>(o[7], -PB_C1_8, PB_S1_8);
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i] = e[i] + o[i]; v[i + 8] = e[i] - o[i]; }
}
template <int R, bool INV> __device__ __forceinline__ void dftR(P2* v) {
    if (R == 2) dft2<INV>(v[0], v[1]);
    else if (R == 4) dft4<INV>(v[0], v[1], v[2], v[3]);
    else if (R == 8) dft8<INV>(v);
    else dft16<INV>(v);
}

__device__ __forceinline__ float4 pack(P2 a) { return make_float4(a.re.x, a.re.y, a.im.x, a.im.y); }
__device__ __forceinline__ P2 unpack(float4 a) { return {make_float2(a.x, a.y), make_float2(a.z, a.w)}; }

// lane A = x, lane B = x * w_32^n (the n-dependent part of the odd half's input ramp), compile-time n
template <bool INV, int n> __device__ __forceinline__ P2 make_lanes(float2 x) {
    // w_32^n = (cos(2 pi n/32), -sin(2 pi n/32))
    constexpr float C[16] = {1.0f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                             0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f,
                             0.19509032201612826785f, 0.0f, -0.19509032201612826785f, -0.38268343236508977173f,
                             -0.55557023301960222474f, -0.70710678118654752440f, -0.83146961230254523708f,
                             -0.92387953251128675613f, -0.98078528040323044913f};
    constexpr float Sn[16] = {0.0f, 0.19509032201612826785f, 0.38268343236508977173f, 0.55557023301960222474f,
                              0.70710678118654752440f, 0.83146961230254523708f, 0.92387953251128675613f,
                              0.98078528040323044913f, 1.0f, 0.98078528040323044913f, 0.92387953251128675613f,
                              0.83146961230254523708f, 0.70710678118654752440f, 0.55557023301960222474f,
                              0.38268343236508977173f, 0.19509032201612826785f};
    const float c = C[n], s = INV ? -Sn[n] : Sn[n];          // x * (c - i s)
    float2 b;
    if (n == 0) b = x;
    else if (n == 8) b = make_float2(x.y * s, -x.x * s);     // c = 0
    else b = make_float2(fmaf(x.x, c, x.y * s), fmaf(x.y, c, -x.x * s));
    return {make_float2(x.x, b.x), make_float2(x.y, b.y)};
}

__device__ __forceinline__ int pad16(int a) { return a + (a >> 4); }

// ---- cache-policy loads / stores --------------------------------------------------------------------
// The only data with reuse inside an SM is the twiddle plan: it is pinned in L1 (evict_last) and every
// streaming access bypasses L1 allocation so that it cannot displace the plan.
__device__ __forceinline__ float4 ld_plan(const float4* p) {
    float4 r;
    asm("ld.global.nc.L1::evict_last.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float2 ld_stream(const float2* p) {
    float2 r;
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ld_stream4(const float4* p) {
    float4 r;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(float4* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream(float2* p, float2 v) {
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}

// ---- async-copy plumbing (cp.async.bulk = the 1-D TMA path; completion on an mbarrier) -------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
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

// ---- tensor TMA (cp.async.bulk.tensor): strided gathers of 32-byte runs into contiguous shared memory ----
__device__ __forceinline__ uint64_t l2_policy(int kind) {   // 0 evict_normal, 1 evict_first, 2 evict_last
    uint64_t pol;
    if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;"
        ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, uint64_t* bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4, %5}], [%6], %7;"
        ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar)), "l"(pol) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void st_hint(float4* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint(float2* p, float2 v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(p), "f"(v.x), "f"(v.y), "l"(pol) : "memory");
}

template <int L> struct Geo {
    static constexpr int NT = L / 16;          // threads per line
    static constexpr int R3 = L / 256;         // last radix
    static constexpr int GI = 16 / R3;         // last-stage items per thread
    static constexpr int SBUF = L + L / 16;    // padded exchange buffer, float4 elements
    // plan table layout (float4 elements):
    //   TW1[k][t], k < 16 : (w_L^(tk).re, (w_L^(tk) w_2L^t).re, w_L^(tk).im, (w_L^(tk) w_2L^t).im)
    //   TW2[k-1][m], 1 <= k < 16, m < NT/16 : (wr, wr, wi, wi), w = w_L^(16 m k)
    static constexpr int TW1 = 0, TW2 = 16 * NT, PLAN = 16 * NT + 15 * (NT / 16);
};

// First two radix-16 stages on both lanes.  In: v[n] = lanes of x[n*NT + t].  Out: stage-2 results in S
// (float4, 1-in-16 padded, position-major): final-stage item i in [0, 256) reads S[pad16(n*256 + i)],
// n < L/256, and after the radix-(L/256) dft holds X[i + 256*k].
// Twiddle sources: 0 = float4 plan in global memory (L1 evict_last), 1 = float4 plan in shared memory,
// 2 = "plain" float2 tables in global memory, the same twiddle for both lanes (k = 1..15 only).
template <int KIND> __device__ __forceinline__ float4 load_tw(const void* base, int idx) {
    if (KIND == 1) return reinterpret_cast<const float4*>(base)[idx];
    if (KIND == 0) return ld_plan(reinterpret_cast<const float4*>(base) + idx);
    float2 w;
    asm("ld.global.nc.L1::evict_last.v2.f32 {%0, %1}, [%2];" : "=f"(w.x), "=f"(w.y) : "l"(reinterpret_cast<const float2*>(base) + idx));
    return make_float4(w.x, w.x, w.y, w.y);
}

template <int L, bool INV, int KIND, class Sync1, class Sync>
__device__ __forceinline__ void fft_two_stages(P2 (&v)[16], const int t, float4* __restrict__ S,
                                               const void* __restrict__ tw1, const void* __restrict__ tw2, Sync1 sync1,
                                               Sync sync) {
    using G = Geo<L>;
    constexpr int NT = G::NT;
    dft16<INV>(v);
    if (KIND == 2) {  // tw1[(k-1)*NT + t]
#pragma unroll
        for (int k = 1; k < 16; ++k) v[k] = mul_tw<INV>(v[k], load_tw<KIND>(tw1, (k - 1) * NT + t));
    } else {          // tw1[k*NT + t], k = 0 carries lane B's w_2L^t
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = mul_tw<INV>(v[k], load_tw<KIND>(tw1, k * NT + t));
    }
    {
        float4* __restrict__ d = S + t * 17;
#pragma unroll
        for (int k = 0; k < 16; ++k) d[k] = pack(v[k]);
    }
    sync1();
    {
        const float4* __restrict__ s = S + pad16(t);
#pragma unroll
        for (int n = 0; n < 16; ++n) v[n] = unpack(s[n * (NT + NT / 16)]);
    }
    sync();
    dft16<INV>(v);
    const int m = t >> 4, a = t & 15;
#pragma unroll
    for (int k = 1; k < 16; ++k) v[k] = mul_tw<INV>(v[k], load_tw<KIND>(tw2, (k - 1) * (NT / 16) + m));
    {
        float4* __restrict__ d = S + m * 272 + a;
#pragma unroll
        for (int k = 0; k < 16; ++k) d[17 * k] = pack(v[k]);
    }
    sync();
}

// final radix-(L/256) stage inputs: afterwards v[g*R3 + n] holds the n-th input of item t + g*NT
template <int L, bool INV>
__device__ __forceinline__ void fft_last_stage_load(P2 (&v)[16], const int t, const float4* __restrict__ S) {
    using G = Geo<L>;
    const float4* __restrict__ s = S + pad16(t);
#pragma unroll
    for (int g = 0; g < G::GI; ++g)
#pragma unroll
        for (int n = 0; n < G::R3; ++n) v[g * G::R3 + n] = unpack(s[n * 272 + g * (G::NT + G::NT / 16)]);
}

#define PB_MAKE_LANES_16(v, INV, X)                                                                         \
    v[0] = make_lanes<INV, 0>(X(0));   v[1] = make_lanes<INV, 1>(X(1));   v[2] = make_lanes<INV, 2>(X(2));     \
    v[3] = make_lanes<INV, 3>(X(3));   v[4] = make_lanes<INV, 4>(X(4));   v[5] = make_lanes<INV, 5>(X(5));     \
    v[6] = make_lanes<INV, 6>(X(6));   v[7] = make_lanes<INV, 7>(X(7));   v[8] = make_lanes<INV, 8>(X(8));     \
    v[9] = make_lanes<INV, 9>(X(9));   v[10] = make_lanes<INV, 10>(X(10)); v[11] = make_lanes<INV, 11>(X(11)); \
    v[12] = make_lanes<INV, 12>(X(12)); v[13] = make_lanes<INV, 13>(X(13)); v[14] = make_lanes<INV, 14>(X(14)); \
    v[15] = make_lanes<INV, 15>(X(15));

struct SyncCta { __device__ __forceinline__ void operator()() const { __syncthreads(); } };

struct FocusParams {
    // column kernel input
    const void* in; int in_kind; const void* amp; int amp_kind; double kturns; long long in_ld;
    float2* tmp;            // [2][N][N] intermediate (plane 0: even output rows, plane 1: odd)
    const float4* plan;     // Geo<N> plan table
    // row kernel output
    void* out; long long out_ld; int out_kind; float scale; float weight;
    int nrows;              // row kernel: batch * 2N
    // batch of independent fields in one launch pair (blockIdx.y in the column kernel; rows of all fields in the row
    // kernel's persistent loop): element strides of in / amp / out in units of their own scalar type
    long long in_bs, amp_bs, out_bs;
    // v2 pipeline
    int ntiles;             // column kernel: batch * N / T tiles, walked by a persistent grid
};

template <int L> struct Geo2 {
    static constexpr int T = 4;                      // columns per tile
    static constexpr int TILES = L / T;              // tiles per field
    static constexpr int BOXR = 256;                 // rows per input box
    static constexpr int NBOX_IN = L / BOXR;
    static constexpr int BOXT = (TILES < 256 ? TILES : 256);   // tiles per row-gather box
    static constexpr int NBOX_ROW = TILES / BOXT;
};

// Column kernel of the v2 pipeline.  One CTA per SM, 16 compute warps + 1 producer warp:
//   * two independent 256-thread GROUPS (named barriers, own exchange buffers): group h computes half-transform h
//     (h = 0: FFT_N(x) -> plane 0; h = 1: FFT_N(x w_K^n) (-dir i) -> plane 1) of the CTA's 4-column tiles.  A thread's
//     two packed lanes are two ADJACENT COLUMNS, so both lanes use the same twiddle, the tile image is read with
//     128-bit shared-memory loads and the tile-major stores are float4 (two columns): four full 128-byte lines per
//     warp instruction.  The groups drift apart by up to one tile, so the exchange phases of one overlap the butterfly
//     phases of the other (the v1 column kernel ran one 16-warp line group in lock step: FP32 pipe 25 %).
//   * the 4-column x L-row input tile (64 KB) is gathered ONCE for both halves by tensor TMA (box = 4 columns x 256
//     rows) into a staging area of its own; the last of the 16 warps to have the inputs of tile i in registers (a
//     shared-memory counter) requests tile i+1 on the spot -- most of a tile time of lead (the gather of 2048 32-byte
//     runs takes ~2-3 us).
//   * one twiddle plan for both halves (float2 entries, 17 KB): half 1's stage-1 twiddles are the plan's times the
//     per-thread constant w_2L^t (its input ramp x w_K^n = x w_32^(n/NT) w_2L^t; the w_32 part is a compile-time constant).
template <int L> struct Geo4 {
    using G = Geo<L>;
    static constexpr int XBUF = G::SBUF + 4;                 // +4 float4 = 16 words: adjacent buffers land on complementary banks
    static constexpr int STAGE = 4 * XBUF;                   // float4 offset of the staging area (multiple of 8: 128-byte aligned)
    static constexpr int PLAN2 = STAGE + 2 * L;              // float4 offset of the float2 plan
    static constexpr int TW1 = 0, TW2 = 16 * G::NT, PLANLEN = 16 * G::NT + 15 * (G::NT / 16);   // float2 elements
    static constexpr size_t BAR_OFF = (size_t)PLAN2 * 16 + (size_t)((PLANLEN * 8 + 15) / 16) * 16;
    static constexpr size_t SMEM = BAR_OFF + 4 * sizeof(uint64_t);
    static constexpr int THREADS = 4 * G::NT;                // 2 groups x 2 column pairs x NT
};

struct SyncGroup {   // named barrier of one 256-thread group (ids 1 and 2; 0 is __syncthreads)
    int id, n;
    __device__ __forceinline__ void operator()() const { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
};

// the first two radix-16 stages with ONE twiddle for both lanes: float2 plan in shared memory, times u (HALF 1)
template <int L, bool INV, int HALF, class Sync>
__device__ __forceinline__ void fft_two_stages_u(P2 (&v)[16], const int t, float4* __restrict__ S, const float2* __restrict__ tw1,
                                                 const float2* __restrict__ tw2, const float2 u, Sync sync) {
    using G = Geo<L>;
    constexpr int NT = G::NT;
    dft16<INV>(v);
    if (HALF) v[0] = mul_tw<INV>(v[0], make_float4(u.x, u.x, u.y, u.y));
#pragma unroll
    for (int k = 1; k < 16; ++k) {
        float2 w = tw1[k * NT + t];
        if (HALF) w = make_float2(fmaf(w.x, u.x, -w.y * u.y), fmaf(w.x, u.y, w.y * u.x));
        v[k] = mul_tw<INV>(v[k], make_float4(w.x, w.x, w.y, w.y));
    }
    {
        float4* __restrict__ d = S + t * 17;
#pragma unroll
        for (int k = 0; k < 16; ++k) d[k] = pack(v[k]);
    }
    sync();
    {
        const float4* __restrict__ s = S + pad16(t);
#pragma unroll
        for (int n = 0; n < 16; ++n) v[n] = unpack(s[n * (NT + NT / 16)]);
    }
    sync();
    dft16<INV>(v);
    const int m = t >> 4, a = t & 15;
#pragma unroll
    for (int k = 1; k < 16; ++k) {
        const float2 w = tw2[(k - 1) * (NT / 16) + m];
        v[k] = mul_tw<INV>(v[k], make_float4(w.x, w.x, w.y, w.y));
    }
    {
        float4* __restrict__ d = S + m * 272 + a;
#pragma unroll
        for (int k = 0; k < 16; ++k) d[17 * k] = pack(v[k]);
    }
    sync();
}

// Row kernel of the v2 pipeline: ONE 512-thread CTA per SM = four independent 128-thread line groups (named barriers, own
// exchange buffer, own row buffer and mbarrier) that share the float2 twiddle plan of the column kernel in shared memory.
// Against an earlier form with three 128-thread CTAs per SM and the float4 plan in L1 (measured and removed, DESIGN 4.1):
// 16 instead of 12 warps per SM, stage-1 twiddles are 64-bit shared-memory loads (lane B's twiddle = lane A's times the per-thread constant w_2L^t, four scalar
// FP32 operations) instead of 128-bit L1 loads whose latency shows up as the kernel's top stall, and the whole unified
// array is shared memory (no L1 working set to protect).
template <int L> struct GeoR4 {
    using G = Geo<L>;
    static constexpr size_t GROUP = (size_t)G::SBUF * 16 + (size_t)L * 8;       // exchange + row buffer, bytes (multiple of 128)
    static constexpr size_t PLAN_OFF = 4 * GROUP;
    static constexpr size_t BAR_OFF = PLAN_OFF + (size_t)((Geo4<L>::PLANLEN * 8 + 15) / 16) * 16;
    static constexpr size_t SMEM = BAR_OFF + 8 * sizeof(uint64_t);
};

template <class K> int set_smem_attrs(Handle* h, K kernel, size_t smem, int ctas_per_sm) {
    if (!attr_needed(h, reinterpret_cast<const void*>(kernel))) return PB_OK;
    PB_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int pct = (int)std::min<size_t>(100, ((size_t)ctas_per_sm * (smem + 1024) * 100 + h->max_smem_optin - 1) / h->max_smem_optin);
    PB_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    return PB_OK;
}

// column-kernel plan of the v2 pipeline: float2 entries, one twiddle for both lanes (see Geo4)
template <int L>
int get_col4_plan(Handle* h, const float2** out) {
    using G4 = Geo4<L>;
    using G = Geo<L>;
    TwKey key{L, PB_C64, 13};
    auto it = h->tables.find(key);
    if (it != h->tables.end()) { *out = reinterpret_cast<const float2*>(it->second); return PB_OK; }
    std::vector<std::complex<double>> tab(G4::PLANLEN);
    auto w = [&](long long num, long long den) {  // exp(-2 pi i num/den), argument reduced exactly
        num %= den;
        const double a = -2.0 * 3.14159265358979323846 * (double)num / (double)den;
        return std::complex<double>(cos(a), sin(a));
    };
    for (int k = 0; k < 16; ++k)
        for (int t = 0; t < G::NT; ++t) tab[G4::TW1 + k * G::NT + t] = w((long long)t * k, L);
    for (int k = 1; k < 16; ++k)
        for (int m = 0; m < G::NT / 16; ++m) tab[G4::TW2 + (k - 1) * (G::NT / 16) + m] = w(16LL * m * k, L);
    const void* d = nullptr;
    PB_TRY(upload_table(h, key, tab, &d));
    *out = reinterpret_cast<const float2*>(d);
    return PB_OK;
}

}  // namespace
}  // namespace pb
