// rdv_lstm.cuh -- one step of sb3_contrib's RecurrentPPO "MlpLstmPolicy" (main_rnn.py: one 256-wide LSTM layer, then
// the default [64, 64] Tanh heads) on the 5th-generation tensor cores, built from the primitives of rdv_policy_tc.cuh
// (UMMA descriptors, TS/SS MMAs, TMEM loads/stores, mbarriers, fp16 hi/lo split).  One kernel body, templated on what
// follows the LSTM (LstmHead): the deterministic actor (rdv_lstm_policy_step), or the collection step's actor with
// the sampled Gaussian head and critic with the value head in one grid (rdv_lstm_actor_critic_step).
//
// A CTA of 256 threads holds TWO tiles of 128 envs (one group per tile, thread = env = TMEM lane, UMMA M = 128):
//
//   A = [obs(17) | 0 x 15 | h(256)]  K = 288 = 18 K-steps; hi -> TMEM (144 columns), lo -> shared (72 KiB)
//   gates, 16 chunks of 16 hidden units: D[128 x 64] = A W_c^T, W_c = the rows i, f, g, o of those 16 units; the
//     bias b_ih + b_hh is added to D in fp32 in the epilogue, not carried through the MMA accumulation (a stressed
//     forget bias of ~3 would sit in every partial sum and cost its rounding at each of the 54 accumulations); the CTA splits W_c (fp32 from L2) into fp16 hi / lo ONCE (72 KiB of shared
//     memory) and both groups multiply their tile by it: 18 K-steps x 3 products per tile
//   epilogue per chunk: c' = s(f) c + s(i) tanh(g), h' = s(o) tanh(c') -> h_out, c_out (fp32, structure of arrays)
//   head: A = h' (read back from h_out, K = 256), D[128 x 64] = A W0^T, tanh -> A, D = A W1^T, tanh -> A,
//     D[128 x 16] = A W2^T (6 outputs padded to N = 16), + b2, clip
//
// Every product is three MMAs of fp16 halves with fp32 accumulation (a_lo b_hi + a_hi b_lo + a_hi b_hi), as in the MLP
// actor, with the weights staged times 2^10 (see LSTM_WSCALE); the activation functions are the accurate expf /
// tanhf, not the exp2-form of the MLP's epilogue, so that the state stays at fp32 accuracy over many recurrent steps.
//
// Budgets per CTA: TMEM 512 columns = 2 x (D 64 + A hi 144, at +0 / +64 of the group's 256); shared memory 222,064 B
// (2 x 73,728 lo-activation tiles, 73,728 B weight stage, biases, mbarriers).  The weight stage holds one gate chunk
// at a time, then W0, then W1 and W2.  L2 traffic: 1.21 MB of fp32 weights per CTA pass, i.e. per 256 envs.
#pragma once
#include "rdv_policy_tc.cuh"

namespace rdv {
namespace tc {

constexpr int LH = 256;                                 // LSTM hidden width
constexpr int LSTM_TILES = 2;                           // tiles (groups of 128 threads) per CTA
constexpr int LSTM_THREADS = LSTM_TILES * TM;
constexpr uint32_t LSTM_TILE_COLS = 256;                // TMEM columns per group: D @ +0..63, A hi @ +64..207
constexpr int HU = 16;                                  // hidden units per gate chunk
constexpr int GN = 4 * HU;                              // gate rows per chunk (i, f, g, o of HU units) = UMMA N
constexpr int KA = K0 + LH;                             // [obs | 1 | pad] + h = 288
// Every weight is staged times 2^10 (exact) and D is scaled back by 2^-10 in fp32: the lo half of a weight of magnitude
// |w| then stays a normal fp16 number down to |w| = 2.4e-4 instead of 0.25 (below that fp16 rounds it to 2^-24 in
// absolute terms, which for |w| ~ 0.05 costs ~20x the precision of the fp32 weight).  hi must stay finite: fp16 rounds
// 65520 up to infinity, so |w| < 65520 / 1024 = 63.984375 (LSTM_WEIGHT_LIMIT of _native.py).
constexpr float LSTM_WSCALE = 1024.0f, LSTM_WUNSCALE = 1.0f / 1024.0f;
static_assert(LSTM_TILES * LSTM_TILE_COLS <= TMEM_COLS, "TMEM budget");
static_assert(A_COL + KA / 2 <= LSTM_TILE_COLS, "A hi must fit the group's TMEM columns");

struct LstmSmem {
    alignas(16) elem_t al[LSTM_TILES][KA * TM];          // lo part of each group's A operand, [chunk][row][CHUNK]
    alignas(16) elem_t wh[GN * KA], wl[GN * KA];         // weight stage, [chunk][n][CHUNK]
    float gb[GN], b0[H], b1[H], b2[N3];                  // gb: b_ih + b_hh of the staged gate chunk
    uint64_t mma_bar[GROUPS];                            // tile_cta_setup initialises GROUPS barriers; 2 are used
    uint32_t tmem_base, pad[3];
};
static_assert(sizeof(LstmSmem) <= 227 * 1024, "shared-memory budget");

// 32 consecutive K elements (K-steps 2b, 2b + 1) of this thread's row of an A operand: hi -> 16 TMEM columns at
// a_hi + 16 b (this lane), lo -> four 16-byte chunks of the row in al
__device__ __forceinline__ void stage_a32(const float (&v)[32], uint32_t a_hi, elem_t *al, int r, int b)
{
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) split2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
#pragma unroll
    for (int c = 0; c < 4; ++c)
        reinterpret_cast<uint4 *>(al)[(4 * b + c) * TM + r] = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
    tmem_st16(a_hi + 16 * b, hi);
}

// The LSTM_THREADS threads split the gate rows of hidden units c HU .. c HU + HU - 1 into the weight stage: stage row
// nn = gate * HU + u is torch row gate * LH + c HU + u; columns 0..16 W_ih, 17..31 zero, 32.. W_hh; gb[nn] = b_ih + b_hh.
// Thread t splits 16-byte chunks (q, nn) with nn fastest, so a warp's shared-memory stores are contiguous.
__device__ __forceinline__ void stage_gate_chunk(const RdvLstmPolicy &pi, int c, elem_t *wh, elem_t *wl, float *gb, int t)
{
    if (t < GN) {
        const int64_t row = (int64_t)(t / HU) * LH + c * HU + t % HU;
        gb[t] = __ldg(pi.bias_ih + row) + __ldg(pi.bias_hh + row);
    }
    constexpr int PER = GN * (KA / CHUNK) / LSTM_THREADS;
    static_assert(PER * LSTM_THREADS == GN * (KA / CHUNK), "gate chunk must split evenly");
    float x[PER][CHUNK];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int idx = t + i * LSTM_THREADS, q = idx / GN, nn = idx % GN;
        const int64_t row = (int64_t)(nn / HU) * LH + c * HU + nn % HU;
        if (q >= K0 / CHUNK) {
            const float *src = pi.weight_hh + row * LH + (q - K0 / CHUNK) * CHUNK;
#pragma unroll
            for (int e = 0; e < CHUNK; ++e) x[i][e] = __ldg(src + e);
        } else {
#pragma unroll
            for (int e = 0; e < CHUNK; ++e) {
                const int k = q * CHUNK + e;
                x[i][e] = k < RDV_OBS_DIM ? __ldg(pi.weight_ih + row * RDV_OBS_DIM + k) : 0.0f;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int idx = t + i * LSTM_THREADS, q = idx / GN, nn = idx % GN;
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) split2(x[i][2 * j] * LSTM_WSCALE, x[i][2 * j + 1] * LSTM_WSCALE, hi[j], lo[j]);
        reinterpret_cast<uint4 *>(wh)[q * GN + nn] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        reinterpret_cast<uint4 *>(wl)[q * GN + nn] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// head hidden-layer epilogue: D (64 columns of this lane) 2^-10 + bias -> tanh -> A hi (TMEM, A_COL) / A lo (shared)
__device__ __forceinline__ void lstm_head_epilogue(uint32_t lane_addr, const float *bias, elem_t *al, int r)
{
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint32_t v[16];
        tmem_ld16_issue(lane_addr + 16 * q, v);
        tmem_ld_wait(v);
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
            split2(tanhf(fmaf(__uint_as_float(v[2 * j]), LSTM_WUNSCALE, bias[16 * q + 2 * j])),
                   tanhf(fmaf(__uint_as_float(v[2 * j + 1]), LSTM_WUNSCALE, bias[16 * q + 2 * j + 1])), hi[j], lo[j]);
        reinterpret_cast<uint4 *>(al)[(2 * q) * TM + r] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        reinterpret_cast<uint4 *>(al)[(2 * q + 1) * TM + r] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
        tmem_st8(lane_addr + A_COL + 8 * q, hi);
    }
    tmem_st_wait();
}

// every thread's shared-memory and TMEM stores -> visible to the MMAs issued after this CTA barrier
__device__ __forceinline__ void cta_sync_for_mma()
{
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
}

// What the step does after the LSTM: LSTM_HEAD_MEAN is the deterministic clipped actor of rdv_lstm_policy_step;
// LSTM_HEAD_ACTOR_CRITIC is the collection step of rdv_lstm_actor_critic_step, where CTAs [0, half) run the actor's
// tile pairs with the sampled Gaussian head and CTAs [half, 2 half) the critic's (LstmCritic) with the value head.
enum LstmHead { LSTM_HEAD_MEAN = 0, LSTM_HEAD_ACTOR_CRITIC = 1 };

template <int HEAD> struct LstmExtra {};
template <> struct LstmExtra<LSTM_HEAD_ACTOR_CRITIC> {
    RdvLstmPolicy critic;                                // its w2, b2: value_net [1][64], [1]
    const float *h_in, *c_in;                            // the critic's state in / out
    float *h_out, *c_out;
    float *env_actions, *log_prob, *values;              // env_actions nullable
    const float *log_std;
    uint64_t seed;                                       // noise of env i: philox_normals(seed; env_offset + i, step)
    int64_t step_index, env_offset, half;
};

// W1 and W2 (ROWS outputs) of the head into the weight stage
template <int ROWS>
__device__ __forceinline__ void stage_head_w12(const RdvLstmPolicy &pi, LstmSmem &s, int t)
{
    WeightTile<LSTM_THREADS, H, H, H, H> w1;
    WeightTile<LSTM_THREADS, ROWS, H, N3, H> w2;
    w1.fetch(pi.w1, nullptr, t);
    w2.fetch(pi.w2, nullptr, t);
    w1.store(LSTM_WSCALE, s.wh, s.wl, t);
    w2.store(LSTM_WSCALE, s.wh + H * H, s.wl + H * H, t);
}

template <int HEAD>
__global__ void __launch_bounds__(LSTM_THREADS, 1)
lstm_step_kernel(RdvLstmPolicy pi, const float *obs, const uint8_t *start, const float *h_in, const float *c_in,
                 float *h_out, float *c_out, float *actions, int64_t n, int64_t ld, const LstmExtra<HEAD> x)
{
    extern __shared__ __align__(128) unsigned char raw[];
    LstmSmem &s = *reinterpret_cast<LstmSmem *>(raw);
    const int t = threadIdx.x, g = t / TM, r = t % TM;
    const uint32_t tmem_all = tile_cta_setup(s);
    const uint32_t tmem = tmem_all + (uint32_t)g * LSTM_TILE_COLS;
    const uint32_t lane_addr = tmem + ((uint32_t)(r & ~31) << 16);         // this warp's 32 TMEM lanes
    elem_t *al = s.al[g];
    uint64_t *bar = &s.mma_bar[g];
    uint32_t phase = 0;
    const int64_t tiles = (n + TM - 1) / TM, pairs = (tiles + LSTM_TILES - 1) / LSTM_TILES;
    unsigned first = blockIdx.x, stride = gridDim.x;
    bool critic = false;
    if constexpr (HEAD == LSTM_HEAD_ACTOR_CRITIC) {
        stride = (unsigned)x.half;
        critic = blockIdx.x >= stride;
        if (critic) {
            first -= stride;
            pi = x.critic;
            h_in = x.h_in;
            c_in = x.c_in;
            h_out = x.h_out;
            c_out = x.c_out;
        }
    }

    for (int64_t pair = first; pair < pairs; pair += stride) {
        const int64_t env = (pair * LSTM_TILES + g) * TM + r;
        const bool valid = env < n;
        const bool keep = valid && !(start && start[env]);                  // else h = c = 0 (episode start)
        // ---- A = [obs | 0 | h] ----
        {
            float v[32];
#pragma unroll
            for (int k = 0; k < 32; ++k)
                v[k] = k < RDV_OBS_DIM ? (valid ? fminf(60000.0f, fmaxf(-60000.0f, obs[env * RDV_OBS_DIM + k])) : 0.0f)
                                       : 0.0f;
            stage_a32(v, lane_addr + A_COL, al, r, 0);
#pragma unroll 1
            for (int b = 1; b < KA / 32; ++b) {
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = keep ? h_in[(int64_t)(32 * (b - 1) + e) * ld + env] : 0.0f;
                stage_a32(v, lane_addr + A_COL, al, r, b);
            }
            tmem_st_wait();
        }
        // ---- gates and cell update, HU hidden units at a time ----
#pragma unroll 1
        for (int c = 0; c < LH / HU; ++c) {
            stage_gate_chunk(pi, c, s.wh, s.wl, s.gb, t);
            cta_sync_for_mma();
            if (r == 0) issue_layer(tmem + A_COL, al, tmem, s.wh, s.wl, GN, KA / KSTEP, bar);
            float c_old[HU];
#pragma unroll
            for (int u = 0; u < HU; ++u) c_old[u] = keep ? c_in[(int64_t)(c * HU + u) * ld + env] : 0.0f;
            mbar_wait(bar, phase);
            phase ^= 1;
            tc_fence_after();
            uint32_t zi[16], zf[16], zg[16], zo[16];
            tmem_ld16_issue(lane_addr + 0 * HU, zi);
            tmem_ld16_issue(lane_addr + 1 * HU, zf);
            tmem_ld16_issue(lane_addr + 2 * HU, zg);
            tmem_ld16_issue(lane_addr + 3 * HU, zo);
            tmem_ld_wait(zi);
            tmem_ld_wait(zf);
            tmem_ld_wait(zg);
            tmem_ld_wait(zo);
#pragma unroll
            for (int u = 0; u < HU; ++u) {
                const float zi_u = fmaf(__uint_as_float(zi[u]), LSTM_WUNSCALE, s.gb[0 * HU + u]);
                const float zf_u = fmaf(__uint_as_float(zf[u]), LSTM_WUNSCALE, s.gb[1 * HU + u]);
                const float zg_u = fmaf(__uint_as_float(zg[u]), LSTM_WUNSCALE, s.gb[2 * HU + u]);
                const float zo_u = fmaf(__uint_as_float(zo[u]), LSTM_WUNSCALE, s.gb[3 * HU + u]);
                const float cn = sigmoidf_acc(zf_u) * c_old[u] + sigmoidf_acc(zi_u) * tanhf(zg_u);
                const float hn = sigmoidf_acc(zo_u) * tanhf(cn);
                if (valid) {
                    h_out[(int64_t)(c * HU + u) * ld + env] = hn;
                    c_out[(int64_t)(c * HU + u) * ld + env] = cn;
                }
            }
            // D drained and the stage read by both groups' MMAs before it is overwritten
            tc_fence_before();
            __syncthreads();
        }
        // ---- head: W0 and the biases into the (now free) stage, A = h' ----
        {
            WeightTile<LSTM_THREADS, H, LH, H, LH> w0;
            w0.fetch(pi.w0, nullptr, t);
            if (t < H) {
                s.b0[t] = __ldg(pi.b0 + t);
                s.b1[t] = __ldg(pi.b1 + t);
            }
            if (t < N3) s.b2[t] = t < (critic ? 1 : RDV_ACT_DIM) ? __ldg(pi.b2 + t) : 0.0f;
            w0.store(LSTM_WSCALE, s.wh, s.wl, t);
            float v[32];
#pragma unroll 1
            for (int b = 0; b < LH / 32; ++b) {
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = valid ? h_out[(int64_t)(32 * b + e) * ld + env] : 0.0f;
                stage_a32(v, lane_addr + A_COL, al, r, b);
            }
            tmem_st_wait();
        }
        cta_sync_for_mma();
        if (r == 0) issue_layer(tmem + A_COL, al, tmem, s.wh, s.wl, H, LH / KSTEP, bar);
        mbar_wait(bar, phase);
        phase ^= 1;
        tc_fence_after();
        lstm_head_epilogue(lane_addr, s.b0, al, r);
        cta_sync_for_mma();                                  // both groups are past their W0 MMAs
        if (critic)
            stage_head_w12<1>(pi, s, t);
        else
            stage_head_w12<RDV_ACT_DIM>(pi, s, t);
        cta_sync_for_mma();
        if (r == 0) issue_layer(tmem + A_COL, al, tmem, s.wh, s.wl, H, H / KSTEP, bar);
        mbar_wait(bar, phase);
        phase ^= 1;
        tc_fence_after();
        lstm_head_epilogue(lane_addr, s.b1, al, r);
        fence_async_smem();
        tc_fence_before();
        group_sync(g, TM);
        if (r == 0) {
            tc_fence_after();
            issue_layer(tmem + A_COL, al, tmem, s.wh + H * H, s.wl + H * H, N3, H / KSTEP, bar);
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        tc_fence_after();
        {
            uint32_t v[16];
            tmem_ld16_issue(lane_addr, v);
            tmem_ld_wait(v);
            if constexpr (HEAD == LSTM_HEAD_MEAN) {
                if (valid) {
#pragma unroll
                    for (int j = 0; j < RDV_ACT_DIM; ++j)
                        actions[env * RDV_ACT_DIM + j] =
                            fminf(1.0f, fmaxf(-1.0f, fmaf(__uint_as_float(v[j]), LSTM_WUNSCALE, s.b2[j])));
                }
            } else if (valid && critic) {
                x.values[env] = fmaf(__uint_as_float(v[0]), LSTM_WUNSCALE, s.b2[0]);
            } else if (valid) {                              // a ~ N(mean, exp(log_std)^2), as the fused rollout draws
                float z[RDV_ACT_DIM];
                philox_normals(x.seed, x.env_offset + env, x.step_index, z);
                float lp = 0.0f;
#pragma unroll
                for (int j = 0; j < RDV_ACT_DIM; ++j) {
                    const float ls = __ldg(x.log_std + j);
                    const float a = fmaf(expf(ls), z[j], fmaf(__uint_as_float(v[j]), LSTM_WUNSCALE, s.b2[j]));
                    actions[env * RDV_ACT_DIM + j] = a;
                    if (x.env_actions) x.env_actions[env * RDV_ACT_DIM + j] = fminf(1.0f, fmaxf(-1.0f, a));
                    lp += fmaf(-0.5f * z[j], z[j], -ls);
                }
                x.log_prob[env] = lp - 5.51363120f;         // 3 ln(2 pi)
            }
        }
        // the next pair restages the weights, biases and this group's A
        tc_fence_before();
        __syncthreads();
    }
    tile_teardown(tmem_all);
}

}  // namespace tc
}  // namespace rdv
