// rdv_policy_tc.cuh -- the actor forward (model.predict of the SB3 MlpPolicy, monte_carlo.py:128-133) on the
// 5th-generation tensor cores: tcgen05.mma with TMEM accumulators AND TMEM-resident A operands.  tile_setup /
// tile_forward / tile_teardown are used by two kernels: policy_tc_kernel below (rdv_policy_forward, stand-alone,
// observations from HBM) and rollout_kernel in rdv_b200.cu (the actor of every step of a fused rollout,
// observations from the env state in registers).  The set-up is split: the CTA-wide part (mbarriers, TMEM) and
// stage_weights, which any set of threads can run into any WeightSet -- the policy-table rollout has one weight set per
// group and restages it when the group's tile uses another actor.
//
// A group of 128 threads owns tiles of 128 environments (UMMA M = 128, one env per thread / TMEM lane):
//
//   obs tile: one 8.7 KB bulk copy (cp.async.bulk, mbarrier complete_tx) into shared memory, prefetched one tile
//             ahead; every thread splits its row into two fp16 halves, hi = fp16(x) and lo = fp16(x - hi)
//   layer 1: D[128x64] = A0[128x32] W0^T    2 K-steps x 3 products; the bias rides in a padding column
//   tcgen05.ld D -> registers, tanh, split -> A1 hi to TMEM (tcgen05.st), A1 lo to shared memory
//   layer 2: D[128x64] = A1 W1^T            4 K-steps x 3
//   tcgen05.ld D -> + bias, tanh, split -> A2
//   layer 3: D[128x16] = A2 W2^T            4 K-steps x 3 (6 outputs padded to N = 16)
//   tcgen05.ld D -> + bias, clip -> actions
//
// Every product is three MMAs of halves (a_lo b_hi + a_hi b_lo + a_hi b_hi, fp32 accumulation) so the result has
// fp32-level accuracy, like the reference's torch policy: 11 + 11 significant bits per operand.  The halves are
// fp16 (kind::f16, K = 16 per MMA): observations, tanh outputs and weights are O(1), far inside the fp16 range, lo
// is exact down to 2^-24 in absolute terms, and a layer costs half the MMAs of a TF32 split (kind::tf32, K = 8) --
// the small-N MMAs of this MLP are issue-rate bound, so that is half the tensor time:
// [B200] 19.5 us against 23.2 for 131,072 rows, worst deviation from an fp64 evaluation 2.7e-6 against 5.0e-6 (the
// MMA truncates the TF32 lo half; the fp16 halves are rounded to nearest).  The hi part of the activations never
// leaves the tensor-memory: the two products that use it are issued in the "TS" form of tcgen05.mma (A from TMEM,
// lane = row, one 32-bit column per pair of K elements, k even in the low half); only the lo part goes through
// shared memory (K-major, no swizzle).  That halves the shared-memory footprint of
// a tile, so a CTA runs FOUR 128-thread groups side by side (512 threads, shared weights; private mbarriers,
// named barriers, 128 TMEM columns each: D @ +0..63, A hi @ +64..127): while one group waits for its MMAs or its
// TMEM loads, three others run their tanh epilogues.  Per group a single thread issues the MMAs and commits them
// to an mbarrier.  exp(2x) = 2^(2 log2(e) x): the factor 2 log2(e) is folded into W0, b0, W1, b1 when the weights
// are split (once per CTA), so a hidden unit costs MUFU.EX2, a quarter of a MUFU.RCP, a handful of FP32 operations
// and the split.
//
// Shared-memory operands use the canonical no-swizzle K-major UMMA layout: 8-row x 16-byte core matrices, rows of
// a core matrix 16 B apart, 8-row groups SBO = 128 B apart, the two 16-byte K-chunks of a K-step
// LBO = rows*16 B apart, i.e. with CHUNK = 8 fp16 elements per 16 bytes element (r, k) lives at
// ((k / CHUNK) * rows + r) * 16 + (k % CHUNK) * 2 bytes.
// (Descriptor bit layouts: CUTLASS cute/arch/mma_sm100_desc.hpp; instruction forms: cute/arch/mma_sm100_umma.hpp.)
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "rdv_b200.h"
#include "rdv_policy.cuh"

namespace rdv {
namespace tc {

constexpr int TM = 128;                 // envs per tile = UMMA M = threads per group
constexpr int H = 64;                   // hidden width
typedef uint16_t elem_t;                // operand element in shared memory: fp16 bits
constexpr int KSTEP = 16, CHUNK = 8;    // K of one MMA; elements of one 16-byte chunk of a core-matrix row
constexpr int K0 = 32;                  // 17 inputs + 1 bias column, padded to 2 K-steps of 16
constexpr int N3 = 16;                  // 6 outputs padded to the smallest legal UMMA N for M = 128
constexpr int GROUPS = 4;               // independent 128-thread tile pipelines per CTA
constexpr uint32_t GROUP_COLS = 128;    // TMEM columns per group: D @ +0..63 (D3 @ +0..15), A hi @ +64..127
constexpr uint32_t TMEM_COLS = GROUPS * GROUP_COLS;
constexpr uint32_t A_COL = 64;
constexpr int OBS_TILE = TM * RDV_OBS_DIM;              // floats of one observation tile (8704 B, 16 B multiple)
constexpr float TANH_SCALE = 2.8853900817779268f;       // 2 log2(e)

// one actor's weights as the MMAs read them: split hi / lo, tanh factor folded in (28.3 KiB)
struct WeightSet {
    alignas(16) elem_t w0h[K0 * H], w0l[K0 * H];                 // [chunk][n][CHUNK]
    alignas(16) elem_t w1h[H * H], w1l[H * H];
    alignas(16) elem_t w2h[H * N3], w2l[H * N3];
    float b1[H], b2[N3], std[8];                                 // std = exp(log_std) (0 without a Gaussian head)
};
static_assert(sizeof(WeightSet) % 16 == 0, "weight sets must stay 16-byte aligned");
// what a tile forward needs: lo activations per group (NA tiles), NW weight sets, MMA mbarriers, the TMEM base
template <int NA, int NW>
struct TileSmemT {
    alignas(16) elem_t al[NA][H * TM];                           // lo part of the activations, [group][chunk][row][CHUNK]
    WeightSet w[NW];
    uint64_t mma_bar[GROUPS];
    uint32_t tmem_base, pad[3];
};
typedef TileSmemT<GROUPS, 1> TileSmem;  // one weight set shared by every group of the CTA
typedef TileSmemT<2, 2> TableSmem;      // policy tables: two groups of 128 threads, each with its own weight set
// the stand-alone kernel adds the bulk-copy landing zone of the next observation tile
struct Smem {
    TileSmem t;
    float obs[GROUPS][OBS_TILE];
    uint64_t obs_bar[GROUPS];
};
static_assert(sizeof(TileSmem) % 16 == 0, "observation landing zone must stay 16-byte aligned");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 64-bit shared-memory matrix descriptor (SWIZZLE_NONE, K-major), see header comment.
__device__ __forceinline__ uint64_t umma_desc(const void *p, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = (uint64_t)((smem_u32(p) >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;                                        // descriptor version of sm_100
    return d;
}
// 32-bit instruction descriptor: D = F32, A = B = F16 (format 0 in bits 7 and 10), both K-major, M = 128, N = n.
__device__ __forceinline__ uint32_t umma_idesc(int n)
{
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}
// D += A B with A described in shared memory ("SS")
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
// D += A B with A read from tensor memory ("TS"): 128 lanes x 8 columns at tmem_a
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :: "r"(tmem_d), "r"(tmem_a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred P1;\n\tLAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 16 consecutive columns of this thread's TMEM lane -> registers; the registers are valid after tmem_ld_wait
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
// wait for the outstanding tcgen05.ld; the registers are tied to the wait so no use can be scheduled above it
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
           "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// the two halves of a float: hi = the value rounded to fp16, lo = what is left, rounded likewise (11 + 11 significant
// bits, lo exact down to 2^-24 in absolute terms)
__device__ __forceinline__ void split2(float a, float b, uint32_t &hi, uint32_t &lo)
{
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}

// bulk copy global -> shared, completion counted in bytes on an mbarrier (one thread issues both)
__device__ __forceinline__ void bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// weights [N_VALID][K_VALID] row-major (+ optional bias as column K_VALID), times `scale` -> chunked K-major
// hi / lo, zero padded to N_PAD x K_PAD.  Two phases so that the global loads of all three layers are in flight
// together before the first value is used.
template <int NT, int N_VALID, int K_VALID, int N_PAD, int K_PAD>
struct WeightTile {
    static constexpr int PER = (N_PAD * K_PAD + NT - 1) / NT;
    float x[PER];
    // t: the calling thread's index among the NT staging threads
    __device__ __forceinline__ void fetch(const float *__restrict__ w, const float *__restrict__ bias_col, int t)
    {
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int idx = t + i * NT;
            const int nn = idx / K_PAD, k = idx % K_PAD;
            x[i] = 0.0f;
            if (idx < N_PAD * K_PAD && nn < N_VALID) {
                if (k < K_VALID) x[i] = __ldg(w + nn * K_VALID + k);
                else if (k == K_VALID && bias_col) x[i] = __ldg(bias_col + nn);
            }
        }
    }
    __device__ __forceinline__ void store(float scale, elem_t *wh, elem_t *wl, int t) const
    {
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int idx = t + i * NT;
            if (idx < N_PAD * K_PAD) {
                const int nn = idx / K_PAD, k = idx % K_PAD;
                const int o = ((k / CHUNK) * N_PAD + nn) * CHUNK + (k % CHUNK);
                const float v = x[i] * scale;
                const __half hi = __float2half_rn(v);
                wh[o] = __half_as_ushort(hi);
                wl[o] = __half_as_ushort(__float2half_rn(v - __half2float(hi)));
            }
        }
    }
};

// one layer: D[128 x n] (TMEM column d_col) = A[128 x KSTEP*ksteps] W^T, three products of halves, issued by the
// calling thread.  A hi: TMEM columns a_hi + 8 kk .. + 7 (one 32-bit column per pair of fp16 elements); A lo: shared
// memory.  A K-step is two 16-byte chunks per row.
__device__ __forceinline__ void issue_layer(uint32_t a_hi, const elem_t *al, uint32_t tmem_d, const elem_t *wh,
                                            const elem_t *wl, int n, int ksteps, uint64_t *bar)
{
    const uint32_t idesc = umma_idesc(n);
    const uint32_t lbo_a = TM * 16, lbo_b = (uint32_t)n * 16;
    for (int kk = 0; kk < ksteps; ++kk) {
        const uint64_t a_lo = umma_desc(al + (size_t)kk * 2 * TM * CHUNK, lbo_a, 128);
        const uint64_t b_hi = umma_desc(wh + (size_t)kk * 2 * n * CHUNK, lbo_b, 128);
        const uint64_t b_lo = umma_desc(wl + (size_t)kk * 2 * n * CHUNK, lbo_b, 128);
        umma_ss(tmem_d, a_lo, b_hi, idesc, kk > 0 ? 1u : 0u);
        umma_ts(tmem_d, a_hi + 8 * kk, b_lo, idesc, 1u);
        umma_ts(tmem_d, a_hi + 8 * kk, b_hi, idesc, 1u);
    }
    umma_commit(bar);
}

// named barrier of group g (`threads` = 128, or fewer in the last group of a CTA that is not a multiple of 128)
__device__ __forceinline__ void group_sync(int g, int threads)
{
    asm volatile("bar.sync %0, %1;" :: "r"(1 + g), "r"(threads) : "memory");
}

// exp-form tanh of four pre-scaled arguments z = 2 log2(e) x:  t = 1 - 2 / (1 + 2^z).  The MUFU unit (16 lanes per
// SM) is the busiest pipe of the epilogue, so the four reciprocals share ONE MUFU.RCP: with a_i = 1 + 2^z_i,
// 1 / a_0 = a_1 (a_2 a_3) / (a_0 a_1 a_2 a_3) and so on -- nine FMULs on the FMA pipe instead of three RCPs.
// z is clamped to 31 (tanh already rounds to 1 in fp32 there), so the product of four stays below 2^127.
__device__ __forceinline__ void tanh_scaled4(const float (&z)[4], float (&t)[4])
{
    float a[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fminf(z[j], 31.0f)));
        a[j] = e + 1.0f;
    }
    const float p01 = a[0] * a[1], p23 = a[2] * a[3];
    float rinv;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rinv) : "f"(p01 * p23));
    const float r01 = rinv * p23, r23 = rinv * p01;             // 1 / (a0 a1), 1 / (a2 a3)
    t[0] = fmaf(-2.0f, r01 * a[1], 1.0f);
    t[1] = fmaf(-2.0f, r01 * a[0], 1.0f);
    t[2] = fmaf(-2.0f, r23 * a[3], 1.0f);
    t[3] = fmaf(-2.0f, r23 * a[2], 1.0f);
}

// hidden-layer epilogue: D (64 columns of this thread's lane) -> tanh -> A hi (TMEM) / A lo (shared), the TMEM load
// of the next 16 columns in flight while the current 16 are processed
template <bool BIAS>
__device__ __forceinline__ void hidden_epilogue(uint32_t lane_addr, const float *bias, elem_t *al, int r)
{
    uint32_t va[16], vb[16];
    tmem_ld16_issue(lane_addr, va);
    tmem_ld_wait(va);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint32_t (&cur)[16] = (q & 1) ? vb : va;
        uint32_t (&nxt)[16] = (q & 1) ? va : vb;
        if (q < 3) tmem_ld16_issue(lane_addr + 16 * (q + 1), nxt);
        float t[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float z[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                z[j] = __uint_as_float(cur[4 * c + j]);
                if (BIAS) z[j] += bias[16 * q + 4 * c + j];
            }
            tanh_scaled4(z, reinterpret_cast<float (&)[4]>(t[4 * c]));
        }
        // 16 activations = 8 packed TMEM columns (hi) and two 16-byte chunks of this row (lo)
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) split2(t[2 * j], t[2 * j + 1], hi[j], lo[j]);
        reinterpret_cast<uint4 *>(al)[(2 * q) * TM + r] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        reinterpret_cast<uint4 *>(al)[(2 * q + 1) * TM + r] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
        tmem_st8(lane_addr + A_COL + 8 * q, hi);
        if (q < 3) tmem_ld_wait(nxt);
    }
    tmem_st_wait();
}

// NT threads (t = 0 .. NT-1 among them) split the weights of pi into w: hi / lo, tanh factor folded in, biases and
// std.  The caller orders the stores before the MMAs that read w (fence.proxy.async, then a barrier of the NT threads).
template <int NT>
__device__ __forceinline__ void stage_weights(const RdvPolicy &pi, WeightSet &w, int t)
{
    WeightTile<NT, H, RDV_OBS_DIM, H, K0> t0;
    WeightTile<NT, H, H, H, H> t1;
    WeightTile<NT, RDV_ACT_DIM, H, N3, H> t2;
    t0.fetch(pi.w0, pi.b0, t);
    t1.fetch(pi.w1, nullptr, t);
    t2.fetch(pi.w2, nullptr, t);
    const float bias1 = t < H ? __ldg(pi.b1 + t) : 0.0f;
    const float bias2 = t < RDV_ACT_DIM ? __ldg(pi.b2 + t) : 0.0f;
    const float lstd = (t < RDV_ACT_DIM && pi.log_std) ? __ldg(pi.log_std + t) : 0.0f;
    t0.store(TANH_SCALE, w.w0h, w.w0l, t);
    t1.store(TANH_SCALE, w.w1h, w.w1l, t);
    t2.store(1.0f, w.w2h, w.w2l, t);
    if (t < H) w.b1[t] = bias1 * TANH_SCALE;
    if (t < N3) w.b2[t] = bias2;
    if (t < 8) w.std[t] = (t < RDV_ACT_DIM && pi.log_std) ? expf(lstd) : 0.0f;
}
// The CTA-wide part of the set-up, in two halves: the groups' MMA mbarriers (thread 0) ...
template <class S>
__device__ __forceinline__ void tile_init_barriers(S &s)
{
    if (threadIdx.x == 0) {
#pragma unroll
        for (int g = 0; g < GROUPS; ++g)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&s.mma_bar[g])) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
}
// ... and 512 TMEM columns (warp 0), then the fences and a __syncthreads that also publish any weights staged before
// it.  Returns the TMEM base address.
template <class S>
__device__ __forceinline__ uint32_t tile_alloc(S &s)
{
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(&s.tmem_base)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return s.tmem_base;
}
// The CTA-wide part alone (mbarriers, TMEM): kernels whose groups stage their own weight sets.
template <class S>
__device__ __forceinline__ uint32_t tile_cta_setup(S &s)
{
    tile_init_barriers(s);
    return tile_alloc(s);
}
// Whole CTA of NT threads, once per launch: the CTA-wide part around ONE weight set that every group uses.
template <int NT>
__device__ __forceinline__ uint32_t tile_setup(const RdvPolicy &pi, TileSmem &s)
{
    tile_init_barriers(s);
    stage_weights<NT>(pi, s.w[0], threadIdx.x);
    return tile_alloc(s);
}
// Whole CTA, after the last tile_forward.
__device__ __forceinline__ void tile_teardown(uint32_t tmem_all)
{
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_all), "r"(TMEM_COLS) : "memory");
}

// One tile through the actor, called by all `threads` threads of group g (thread r owns row r = its TMEM lane).
// al / bar: the group's lo-activation tile and MMA mbarrier; w: the weight set the group applies.
// x: the row's 17 observations; out: the actor's mean action, NOT clipped.  `after_issue` runs on the issuing
// thread right after the layer-1 MMAs are queued (every thread of the group is past its use of shared staging).
template <class F>
__device__ __forceinline__ void tile_forward(elem_t *al, uint64_t *bar, const WeightSet &w, int g, int r, int threads,
                                             const float (&x)[RDV_OBS_DIM], uint32_t tmem, uint32_t &phase,
                                             float (&out)[RDV_ACT_DIM], F &&after_issue)
{
    const uint32_t lane_addr = tmem + ((uint32_t)(r & ~31) << 16);         // this warp's 32 TMEM lanes
    // ---- A0: the observation row and the constant 1 of the bias column, hi -> TMEM, lo -> shared ----
    {
        // (values beyond the fp16 range are clamped: the first layer's tanh is saturated long before)
        uint32_t hi[K0 / 2], lo[K0 / 2];
#pragma unroll
        for (int j = 0; j < K0 / 2; ++j) {
            float v[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int k = 2 * j + u;
                v[u] = k < RDV_OBS_DIM ? fminf(60000.0f, fmaxf(-60000.0f, x[k < RDV_OBS_DIM ? k : 0]))
                                       : (k == RDV_OBS_DIM ? 1.0f : 0.0f);
            }
            split2(v[0], v[1], hi[j], lo[j]);
        }
#pragma unroll
        for (int c = 0; c < K0 / CHUNK; ++c)
            reinterpret_cast<uint4 *>(al)[c * TM + r] = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
        tmem_st16(lane_addr + A_COL, hi);
        tmem_st_wait();
    }
    fence_async_smem();
    tc_fence_before();
    group_sync(g, threads);
    // ---- layer 1 ----
    if (r == 0) {
        tc_fence_after();
        issue_layer(tmem + A_COL, al, tmem, w.w0h, w.w0l, H, K0 / KSTEP, bar);
        after_issue();
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    hidden_epilogue<false>(lane_addr, nullptr, al, r);
    fence_async_smem();
    tc_fence_before();
    group_sync(g, threads);
    // ---- layer 2 (D is reused: the layer-1 epilogue has drained it) ----
    if (r == 0) {
        tc_fence_after();
        issue_layer(tmem + A_COL, al, tmem, w.w1h, w.w1l, H, H / KSTEP, bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    hidden_epilogue<true>(lane_addr, w.b1, al, r);
    fence_async_smem();
    tc_fence_before();
    group_sync(g, threads);
    // ---- layer 3 ----
    if (r == 0) {
        tc_fence_after();
        issue_layer(tmem + A_COL, al, tmem, w.w2h, w.w2l, N3, H / KSTEP, bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    {
        uint32_t v[16];
        tmem_ld16_issue(lane_addr, v);
        tmem_ld_wait(v);
#pragma unroll
        for (int j = 0; j < RDV_ACT_DIM; ++j) out[j] = __uint_as_float(v[j]) + w.b2[j];
    }
    // the next tile's A0 stores and layer-1 MMAs are ordered after these loads by the fences around its first
    // group_sync
    tc_fence_before();
}

__global__ void __launch_bounds__(GROUPS * TM, 1) policy_tc_kernel(const RdvPolicy pi, const float *obs, float *actions, int64_t n)
{
    extern __shared__ __align__(128) unsigned char raw[];
    Smem &s = *reinterpret_cast<Smem *>(raw);
    const int g = threadIdx.x / TM, r = threadIdx.x % TM;                  // group, row in tile
    uint64_t *obs_bar = &s.obs_bar[g];
    // tile t belongs to CTA t % grid and, there, to group (t / grid) % GROUPS: consecutive tiles go to different SMs, so
    // the per-SM tile counts differ by at most one (131,072 rows = 1,024 tiles over 148 SMs: 6 or 7 tiles each; the
    // group-major order of round 1 gave 108 SMs 8 tiles and 40 SMs 4)
    const int64_t tiles = (n + TM - 1) / TM, stride = (int64_t)gridDim.x * GROUPS;
    const int64_t first = (int64_t)blockIdx.x + (int64_t)g * gridDim.x;
    const bool bulk_ok = (reinterpret_cast<uintptr_t>(obs) & 15) == 0;        // cp.async.bulk needs 16-byte alignment

    // the first observation tile is in flight while the weights are split
    if (r == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(obs_bar)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (bulk_ok && first < tiles && (first + 1) * TM <= n)
            bulk_load(s.obs[g], obs + first * OBS_TILE, OBS_TILE * 4, obs_bar);
    }
    const uint32_t tmem_all = tile_setup<GROUPS * TM>(pi, s.t);
    const uint32_t tmem = tmem_all + (uint32_t)g * GROUP_COLS;             // this group's columns
    uint32_t mma_phase = 0, obs_phase = 0;

    for (int64_t tile = first; tile < tiles; tile += stride) {
        const int64_t env = tile * TM + r;
        const bool valid = env < n, staged = bulk_ok && (tile + 1) * TM <= n;
        float x[RDV_OBS_DIM], a[RDV_ACT_DIM];
        if (staged) {
            mbar_wait(obs_bar, obs_phase);
            obs_phase ^= 1;
#pragma unroll
            for (int k = 0; k < RDV_OBS_DIM; ++k) x[k] = s.obs[g][r * RDV_OBS_DIM + k];
        } else {
#pragma unroll
            for (int k = 0; k < RDV_OBS_DIM; ++k) x[k] = valid ? obs[env * RDV_OBS_DIM + k] : 0.0f;
        }
        tile_forward(s.t.al[g], &s.t.mma_bar[g], s.t.w[0], g, r, TM, x, tmem, mma_phase, a, [&] {
            // bulk copy of this group's next tile: every thread has consumed the landing zone
            const int64_t next = tile + stride;
            if (bulk_ok && next < tiles && (next + 1) * TM <= n) bulk_load(s.obs[g], obs + next * OBS_TILE, OBS_TILE * 4, obs_bar);
        });
        if (valid) {
#pragma unroll
            for (int j = 0; j < RDV_ACT_DIM; ++j) actions[env * RDV_ACT_DIM + j] = fminf(1.0f, fmaxf(-1.0f, a[j]));   // np.clip
        }
    }
    tile_teardown(tmem_all);
}

}  // namespace tc
}  // namespace rdv
