// On-device policy step (SURVEY.md section 8f-1): the reference evaluates its trained agents on the host,
// once per env step, inside utilities/misc.py:134-221 run_env:
//     q_values, hs = model(torch.Tensor(obs), torch.Tensor(hs));  actions = np.argmax(q_values, axis=1)
// with model = utilities/rnn_agent.py:5-29 RNNAgent (fc1 -> ReLU -> GRUCell | Linear+ReLU -> fc2) or
// utilities/rnn_ns_agent.py:5-36 RNNNSAgent (one RNNAgent per agent).  Here ONE kernel does that for every
// agent of every env and writes the int32 actions buffer that mrb_step consumes.
//
// Mapping: a warp owns 16 rows = one agent index in 16 consecutive envs (rows of one agent share a weight
// set, so non-shared agents cost nothing extra).  All three layers are FP16 m16n8k16 tensor-core MMAs with
// FP32 accumulation (FP16 keeps the same 11-bit significand as TF32 at twice the MMA rate and half the
// shared-memory bytes per flop - the first, TF32 m16n8k8 version of this kernel was bound by B-fragment
// shared-memory loads, profiles/r01_ncu_policy_tf32.txt).  The activations never leave registers: the
// accumulator fragments of two adjacent 16x8 output tiles ARE the A fragment of the next layer's 16x16
// k-tile (no shuffles), the hidden state is loaded once as A fragments, and fc2 is accumulated as the GRU
// produces h'.  Weights are rounded to FP16 and laid out in fragment order once, on the device (policy_pack_kernel, at
// mrb_policy_create and mrb_policy_load), so staging them is a linear cp.async copy and every B fragment pair is a single
// conflict-free 128-bit shared load; the GRU weights (6 H^2 halves, 197 KB for H = 128) stream through a
// double-buffered 2 x 12.3 KB window, one 8-unit column tile at a time.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

#include <cuda_fp16.h>

#include "common.cuh"
#include "policy_tc.cuh"
#include "policy_tc2.cuh"
#include "policy_f32.cuh"

namespace mrb {

constexpr int kPolicyWarps = 4;          // 64 envs of one agent per CTA share every staged weight tile
constexpr int kMaxKS1 = 4;               // fc1 input width <= 64 (k-steps of 16)
constexpr int kMaxAT = 3;                // n_actions <= 24

struct PolicyParams {
    const float *wpack;                  // packed weight sets (device)
    int64_t set_floats;                  // floats per set
    int64_t B;
    int32_t obs_dim, input_dim, n_actions, n_agents, obs_agent_id, non_shared;
    int32_t KS1, AT;                     // fc1 k-steps, fc2 column tiles
    int32_t szW1, szW2, head_floats;     // packed section sizes (32-bit words)
};

// two floats -> one .f16x2 register (lower column in the lower half)
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi)
{
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&h);
}
// D = A (16x16, row) * B (16x8, col) + D, FP16 inputs, FP32 accumulate
__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(float *dst_smem, const float *src)
{
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// sigma(x) = 1 / (1 + 2^(-x log2 e)) and tanh(x) = 2 sigma(2x) - 1 straight on the SFU (ex2.approx + rcp.approx, relative
// error ~1e-7: three orders below the FP16 rounding of the matmul operands), 4 - 5 instructions, no branches
__device__ __forceinline__ float ex2_(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoidf_(float x) { return rcp_(1.f + ex2_(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanhf_(float x) { return fmaf(2.f, rcp_(1.f + ex2_(-2.8853900817779268f * x)), -1.f); }

constexpr int kPolicyMinBlocks = 4;      // 128 registers, 16 warps per SM: measured 0.327 ms vs 0.344 (3) and 0.427 (2) for 262,144 agents
template <int H, bool RNN>
__global__ void __launch_bounds__(kPolicyWarps * 32, kPolicyMinBlocks)
policy_act_kernel(const PolicyParams p, const float *obs, float *hidden, int32_t *__restrict__ actions,
                  float *__restrict__ q_out, const uint8_t *__restrict__ fresh)
{
    extern __shared__ __align__(16) float sm[];
    constexpr int NT = H / 8, KS = H / 16, G = RNN ? 6 : 1;  // 8-column output tiles, 16-wide k-steps
    constexpr int CHUNK = G * KS * 64;                       // 32-bit words per column tile of the recurrent layer
    constexpr int NB = RNN ? 6 * H : H;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const int agent = blockIdx.y;
    const float *wimg = p.wpack + (size_t)(p.non_shared ? agent : 0) * p.set_floats;
    float *sW1 = sm, *sB1 = sW1 + p.szW1, *sBias = sB1 + H, *sW2 = sBias + NB, *sB2 = sW2 + p.szW2;
    float *sChunk = sm + p.head_floats;
    const float *gchunks = wimg + p.head_floats;

    for (int i = threadIdx.x * 4; i < p.head_floats; i += kPolicyWarps * 128) cp_async16(sm + i, wimg + i);
    cp_commit();
    for (int i = threadIdx.x * 4; i < CHUNK; i += kPolicyWarps * 128) cp_async16(sChunk + i, gchunks + i);
    cp_commit();

    const int N = p.n_agents, D = p.obs_dim;
    const int64_t e0 = (int64_t)blockIdx.x * (kPolicyWarps * 16) + warp * 16;
    const int64_t eA = e0 + g, eB = e0 + g + 8;
    const bool vA = eA < p.B, vB = eB < p.B;
    const bool zA = !vA || (fresh && fresh[eA]), zB = !vB || (fresh && fresh[eB]);     // rows that read as zero
    const int64_t rA = ((vA ? eA : 0) * N + agent), rB = ((vB ? eB : 0) * N + agent);
    const float *oA = obs + rA * D, *oB = obs + rB * D;
    float *hA_ptr = hidden + rA * H, *hB_ptr = hidden + rB * H;

    // ---- observation (+ one-hot agent id, misc.py:161-162) as A fragments: a0 = (row g, cols 2t, 2t+1),
    //      a1 = (row g+8, same cols), a2 / a3 = the same rows, cols 2t+8, 2t+9 of the 16-wide k-step
    uint32_t oa[kMaxKS1][4];
    auto in_val = [&](const float *o, bool zero, int c) -> float {
        const float v = o[c < D ? c : 0];                     // always in bounds; selected away below
        return c < D ? (zero ? 0.f : v) : ((p.obs_agent_id && c - D == agent) ? 1.f : 0.f);
    };
#pragma unroll
    for (int s = 0; s < kMaxKS1; s++) {
        if (s < p.KS1) {
            const int c = 16 * s + 2 * t;
            oa[s][0] = pack_h2(in_val(oA, zA, c), in_val(oA, zA, c + 1));
            oa[s][1] = pack_h2(in_val(oB, zB, c), in_val(oB, zB, c + 1));
            oa[s][2] = pack_h2(in_val(oA, zA, c + 8), in_val(oA, zA, c + 9));
            oa[s][3] = pack_h2(in_val(oB, zB, c + 8), in_val(oB, zB, c + 9));
        } else {
            oa[s][0] = oa[s][1] = oa[s][2] = oa[s][3] = 0u;
        }
    }
    // ---- hidden state as A fragments (GRU only)
    uint32_t ha[RNN ? KS : 1][4];
    if (RNN) {
        const float2 zero2 = make_float2(0.f, 0.f);
#pragma unroll
        for (int s = 0; s < KS; s++) {
            const int c = 16 * s + 2 * t;
            float2 a0 = *reinterpret_cast<const float2 *>(hA_ptr + c), a1 = *reinterpret_cast<const float2 *>(hB_ptr + c);
            float2 a2 = *reinterpret_cast<const float2 *>(hA_ptr + c + 8), a3 = *reinterpret_cast<const float2 *>(hB_ptr + c + 8);
            a0 = zA ? zero2 : a0; a1 = zB ? zero2 : a1; a2 = zA ? zero2 : a2; a3 = zB ? zero2 : a3;   // rows are always in bounds
            ha[s][0] = pack_h2(a0.x, a0.y); ha[s][1] = pack_h2(a1.x, a1.y);
            ha[s][2] = pack_h2(a2.x, a2.y); ha[s][3] = pack_h2(a3.x, a3.y);
        }
    }

    cp_wait<1>();                                            // head (W1, biases, W2) has landed
    __syncthreads();

    // ---- x = relu(fc1(obs))                                 rnn_agent.py:22
    // the accumulator fragments (rows g, g+8; cols 2t, 2t+1) of output tiles 2k and 2k+1 are exactly the A
    // fragment (a0, a1 | a2, a3) of k-step k of the next layer
    uint32_t xa[KS][4];
    {
        const uint2 *w1 = reinterpret_cast<const uint2 *>(sW1) + lane;
#pragma unroll
        for (int j = 0; j < NT; j++) {
            const float2 b = *reinterpret_cast<const float2 *>(sB1 + 8 * j + 2 * t);
            float acc[4] = {b.x, b.y, b.x, b.y};
#pragma unroll
            for (int s = 0; s < kMaxKS1; s++)
                if (s < p.KS1) {
                    const uint2 w = w1[(j * p.KS1 + s) * 32];
                    mma_f16(acc, oa[s], w.x, w.y);
                }
            xa[j >> 1][(j & 1) * 2] = pack_h2(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f));
            xa[j >> 1][(j & 1) * 2 + 1] = pack_h2(fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f));
        }
    }

    // ---- recurrent layer, one 8-unit column tile at a time; fc2 accumulated on the fly
    float qacc[kMaxAT][4];
#pragma unroll
    for (int jt = 0; jt < kMaxAT; jt++) {
        const float2 b = jt < p.AT ? *reinterpret_cast<const float2 *>(sB2 + 8 * jt + 2 * t) : make_float2(0.f, 0.f);
        qacc[jt][0] = b.x; qacc[jt][1] = b.y; qacc[jt][2] = b.x; qacc[jt][3] = b.y;
    }
    uint32_t hp[4] = {0u, 0u, 0u, 0u};                       // h' of the current pair of column tiles, A layout
#pragma unroll 1
    for (int j = 0; j < NT; j++) {
        if (j + 1 < NT) {
            float *dst = sChunk + ((j + 1) & 1) * CHUNK;
            const float *src = gchunks + (size_t)(j + 1) * CHUNK;
            for (int i = threadIdx.x * 4; i < CHUNK; i += kPolicyWarps * 128) cp_async16(dst + i, src + i);
        }
        cp_commit();
        cp_wait<1>();                                        // tile j has landed (tile j + 1 may be in flight)
        __syncthreads();
        const uint4 *c4 = reinterpret_cast<const uint4 *>(sChunk + (j & 1) * CHUNK) + lane;
        const int c0 = 8 * j + 2 * t;
        float hn[4];
        if (RNN) {
            // torch.nn.GRUCell: r = s(W_ir x + b_ir + W_hr h + b_hr), z likewise, n = tanh(W_in x + b_in + r (W_hn h + b_hn)),
            // h' = (1 - z) n + z h; weight_ih / weight_hh rows are the (r, z, n) gates in that order
            const float *bi = sBias, *bh = sBias + 3 * H;
            // old h of this tile in accumulator layout (issued before the MMAs so that the latency is hidden)
            float2 oldA = *reinterpret_cast<const float2 *>(hA_ptr + c0), oldB = *reinterpret_cast<const float2 *>(hB_ptr + c0);
            oldA = zA ? make_float2(0.f, 0.f) : oldA;
            oldB = zB ? make_float2(0.f, 0.f) : oldB;
            float ar[4], az[4], ai[4], ah[4];
            float ar2[4] = {0.f, 0.f, 0.f, 0.f}, az2[4] = {0.f, 0.f, 0.f, 0.f};     // separate chains for the h-side products
            {
                const float2 ir = *reinterpret_cast<const float2 *>(bi + c0), hr = *reinterpret_cast<const float2 *>(bh + c0);
                const float2 iz = *reinterpret_cast<const float2 *>(bi + H + c0), hz = *reinterpret_cast<const float2 *>(bh + H + c0);
                const float2 in = *reinterpret_cast<const float2 *>(bi + 2 * H + c0), hn2 = *reinterpret_cast<const float2 *>(bh + 2 * H + c0);
                ar[0] = ar[2] = ir.x + hr.x; ar[1] = ar[3] = ir.y + hr.y;
                az[0] = az[2] = iz.x + hz.x; az[1] = az[3] = iz.y + hz.y;
                ai[0] = ai[2] = in.x; ai[1] = ai[3] = in.y;
                ah[0] = ah[2] = hn2.x; ah[1] = ah[3] = hn2.y;
            }
#pragma unroll
            for (int sp = 0; sp < KS / 2; sp++) {
                uint4 w;
                w = c4[(0 * (KS / 2) + sp) * 32]; mma_f16(ar, xa[2 * sp], w.x, w.y); mma_f16(ar, xa[2 * sp + 1], w.z, w.w);
                w = c4[(1 * (KS / 2) + sp) * 32]; mma_f16(az, xa[2 * sp], w.x, w.y); mma_f16(az, xa[2 * sp + 1], w.z, w.w);
                w = c4[(2 * (KS / 2) + sp) * 32]; mma_f16(ai, xa[2 * sp], w.x, w.y); mma_f16(ai, xa[2 * sp + 1], w.z, w.w);
                w = c4[(3 * (KS / 2) + sp) * 32]; mma_f16(ar2, ha[2 * sp], w.x, w.y); mma_f16(ar2, ha[2 * sp + 1], w.z, w.w);
                w = c4[(4 * (KS / 2) + sp) * 32]; mma_f16(az2, ha[2 * sp], w.x, w.y); mma_f16(az2, ha[2 * sp + 1], w.z, w.w);
                w = c4[(5 * (KS / 2) + sp) * 32]; mma_f16(ah, ha[2 * sp], w.x, w.y); mma_f16(ah, ha[2 * sp + 1], w.z, w.w);
            }
            const float old[4] = {oldA.x, oldA.y, oldB.x, oldB.y};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const float r = sigmoidf_(ar[i] + ar2[i]), z = sigmoidf_(az[i] + az2[i]);
                const float n = tanhf_(ai[i] + r * ah[i]);
                hn[i] = (1.f - z) * n + z * old[i];
            }
        } else {
            // h = relu(rnn(x)) with rnn = nn.Linear                rnn_agent.py:26-27
            const float2 b = *reinterpret_cast<const float2 *>(sBias + c0);
            hn[0] = b.x; hn[1] = b.y; hn[2] = b.x; hn[3] = b.y;
#pragma unroll
            for (int sp = 0; sp < KS / 2; sp++) {
                const uint4 w = c4[sp * 32];
                mma_f16(hn, xa[2 * sp], w.x, w.y);
                mma_f16(hn, xa[2 * sp + 1], w.z, w.w);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) hn[i] = fmaxf(hn[i], 0.f);
        }
        if (vA) *reinterpret_cast<float2 *>(hA_ptr + c0) = make_float2(hn[0], hn[1]);
        if (vB) *reinterpret_cast<float2 *>(hB_ptr + c0) = make_float2(hn[2], hn[3]);
        // q += h'[:, tiles j-1, j] * fc2.weight[:, those columns]'   (every second tile)        rnn_agent.py:28
        if (!(j & 1)) {
            hp[0] = pack_h2(hn[0], hn[1]);
            hp[1] = pack_h2(hn[2], hn[3]);
        } else {
            hp[2] = pack_h2(hn[0], hn[1]);
            hp[3] = pack_h2(hn[2], hn[3]);
            const uint2 *w2 = reinterpret_cast<const uint2 *>(sW2) + lane;
#pragma unroll
            for (int jt = 0; jt < kMaxAT; jt++)
                if (jt < p.AT) {
                    const uint2 w = w2[(jt * KS + (j >> 1)) * 32];
                    mma_f16(qacc[jt], hp, w.x, w.y);
                }
        }
        __syncthreads();                                     // everyone is done with buffer j & 1
    }

    // ---- greedy action: first maximum, like np.argmax (misc.py:170)
    float bestA = -INFINITY, bestB = -INFINITY;
    int idxA = 0, idxB = 0;
#pragma unroll
    for (int jt = 0; jt < kMaxAT; jt++)
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int c = 8 * jt + 2 * t + k;
            if (jt < p.AT && c < p.n_actions) {
                if (qacc[jt][k] > bestA) { bestA = qacc[jt][k]; idxA = c; }
                if (qacc[jt][2 + k] > bestB) { bestB = qacc[jt][2 + k]; idxB = c; }
                if (q_out) {
                    if (vA) q_out[rA * p.n_actions + c] = qacc[jt][k];
                    if (vB) q_out[rB * p.n_actions + c] = qacc[jt][2 + k];
                }
            }
        }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
        const float ovA = __shfl_xor_sync(0xffffffffu, bestA, o), ovB = __shfl_xor_sync(0xffffffffu, bestB, o);
        const int oiA = __shfl_xor_sync(0xffffffffu, idxA, o), oiB = __shfl_xor_sync(0xffffffffu, idxB, o);
        if (ovA > bestA || (ovA == bestA && oiA < idxA)) { bestA = ovA; idxA = oiA; }
        if (ovB > bestB || (ovB == bestB && oiB < idxB)) { bestB = ovB; idxB = oiB; }
    }
    if (t == 0) {
        if (vA) actions[rA] = idxA;
        if (vB) actions[rB] = idxB;
    }
}

// ---- weight images, built on the device from the state_dict-order weights (mrb_policy_create, mrb_policy_load)
//
// B fragment word of W' (W torch layout [out][in]; rows >= rows_valid and columns >= cols_valid read as zero) for 8-column
// tile j, 16-wide k-step s, lane (g, t): half 0 is b0 = {W[r][16s+2t], W[r][16s+2t+1]}, half 1 is b1 = the same 8 columns
// on, r = row0 + 8j + g, each pair rounded to FP16 and packed low | high
__device__ __forceinline__ uint32_t frag_word(const float *W, int ld, int row0, int rows_valid, int cols_valid, int j, int s,
                                              int lane, int half)
{
    const int r = 8 * j + (lane >> 2), k = 16 * s + 2 * (lane & 3) + 8 * half;
    auto at = [&](int c) { return (r < rows_valid && c < cols_valid) ? W[(size_t)(row0 + r) * ld + c] : 0.f; };
    return pack_h2(at(k), at(k + 1));
}

// Word o of the image of one weight set (PolicyParams::set_floats words), in the order policy_act_kernel stages it:
//   head (head_floats words): W1 fragments [NT][KS1][32 lanes][b0, b1] | b1 [H] | biases (b_ih | b_hh, or b) [NB] |
//   W2 fragments [AT][KS][32][b0, b1] | b2 [AT * 8] (zero past n_actions);
//   then per 8-unit column tile j of the recurrent layer a chunk [G][KS / 2][32][4]: gate matrix gi (W_ir, W_iz, W_in,
//   W_hr, W_hz, W_hn; the Linear's W alone), k-step pair sp, lane, then (b0, b1) of k-step 2sp and of k-step 2sp + 1.
__device__ __forceinline__ uint32_t wpack_word(const WeightSet &w, const PolicyParams &p, int H, bool rnn, int64_t o)
{
    const int Din = p.input_dim, A = p.n_actions, KS = H / 16;
    if (o < p.szW1) {
        const int js = (int)(o / 64);
        return frag_word(w.fc1w, Din, 0, H, Din, js / p.KS1, js % p.KS1, (int)(o / 2) % 32, (int)(o & 1));
    }
    o -= p.szW1;
    if (o < H) return __float_as_uint(w.fc1b[o]);
    o -= H;
    const int NB = rnn ? 6 * H : H;
    if (o < NB) return __float_as_uint(o < 3 * H || !rnn ? w.bih[o] : w.bhh[o - 3 * H]);
    o -= NB;
    if (o < p.szW2) {
        const int js = (int)(o / 64);
        return frag_word(w.fc2w, H, 0, A, H, js / KS, js % KS, (int)(o / 2) % 32, (int)(o & 1));
    }
    o -= p.szW2;
    if (o < 8 * p.AT) return __float_as_uint(o < A ? w.fc2b[o] : 0.f);
    o -= 8 * p.AT;
    const int chunk = (rnn ? 6 : 1) * KS * 64, j = (int)(o / chunk), c = (int)(o % chunk);
    const int gi = (c / 128) / (KS / 2), sp = (c / 128) % (KS / 2), q = c % 4;
    const float *W = rnn && gi >= 3 ? w.whh : w.wih;
    return frag_word(W, H, rnn ? (gi % 3) * H : 0, H, H, j, 2 * sp + (q >> 1), (c / 4) % 32, q & 1);
}

// Every image a policy holds, back to back in one index space of 32-bit words: wpack, then tc2 (n_tc2 = 0 without one),
// then w32 (n_w32 = 0 unless accurate).  Each thread writes one word, every word of every image.
struct PackParams {
    const float *w;                      // state_dict-order weights (device), `per_set` floats per set
    int64_t per_set;
    int32_t H, Din, A, rnn;
    uint32_t *wpack, *tc2, *w32;
    int64_t n_wpack, n_tc2, n_w32;       // words per image, all sets
    int64_t tc2_set_words;
    int32_t dp;
    PolicyParams p;
    f32::Params32 p32;
};
constexpr int kPackThreads = 256;

__global__ void __launch_bounds__(kPackThreads) policy_pack_kernel(const PackParams k)
{
    int64_t i = (int64_t)blockIdx.x * kPackThreads + threadIdx.x;
    const bool rnn = k.rnn != 0;
    if (i < k.n_wpack) {
        const int64_t set = i / k.p.set_floats;
        k.wpack[i] = wpack_word(WeightSet(k.w + set * k.per_set, k.H, k.Din, k.A, rnn), k.p, k.H, rnn, i % k.p.set_floats);
        return;
    }
    i -= k.n_wpack;
    if (i < k.n_tc2) {
        const int64_t set = i / k.tc2_set_words;
        k.tc2[i] = tc2::image_word(WeightSet(k.w + set * k.per_set, k.H, k.Din, k.A, rnn), k.Din, k.A, k.dp, i % k.tc2_set_words);
        return;
    }
    i -= k.n_tc2;
    if (i < k.n_w32) {
        const int64_t set = i / k.p32.set_floats;
        k.w32[i] = __float_as_uint(f32::image_value(WeightSet(k.w + set * k.per_set, k.H, k.Din, k.A, rnn), k.p32, k.H, rnn,
                                                    i % k.p32.set_floats));
    }
}

}  // namespace mrb

// ------------------------------------------------------------------------------------------------ host side
using namespace mrb;

struct mrb_policy {
    mrb_policy_desc d;
    int device;
    int64_t num_weights;        // the count mrb_policy_create took (mrb_policy_load takes the same)
    float *wpack;
    uint8_t *tc2_img;           // persistent tcgen05 path (policy_tc2.cuh), NULL when the model does not fit it
    mrb::tc2::Params2 tcp2;
    size_t tc2_smem;
    int num_sms;
    PolicyParams p;
    size_t smem_bytes;
    float *w32;                 // float32 path (policy_f32.cuh), only when desc.accurate
    mrb::f32::Params32 p32;
    PackParams pack;            // policy_pack_kernel's arguments but the weights
    std::string err;
};

static std::string g_policy_create_error;
namespace mrb { void count_launch(); }       // capi.cu: the library-wide launch counter

static int pfail(mrb_policy *p, int code, const std::string &msg)
{
    if (p) p->err = msg; else g_policy_create_error = msg;
    return code;
}

// rebuilds every image of `pol` from the state_dict-order weights w (device): one launch on s
static cudaError_t launch_pack(const mrb_policy *pol, const float *w, cudaStream_t s)
{
    PackParams k = pol->pack;
    k.w = w;
    const int64_t words = k.n_wpack + k.n_tc2 + k.n_w32;
    policy_pack_kernel<<<(unsigned)((words + kPackThreads - 1) / kPackThreads), kPackThreads, 0, s>>>(k);
    return cudaGetLastError();
}

static void free_images(mrb_policy *pol)
{
    if (pol->wpack) cudaFree(pol->wpack);
    if (pol->tc2_img) cudaFree(pol->tc2_img);
    if (pol->w32) cudaFree(pol->w32);
    delete pol;
}

extern "C" const char *mrb_policy_last_error(const mrb_policy *p) { return p ? p->err.c_str() : g_policy_create_error.c_str(); }

extern "C" int mrb_policy_create(const mrb_policy_desc *desc, int device, const float *weights, int64_t num_weights,
                                 mrb_policy **out)
{
    if (!desc || !weights || !out) return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: null argument");
    if (desc->struct_size != (int32_t)sizeof(mrb_policy_desc))
        return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: mrb_policy_desc.struct_size does not match this library");
    const mrb_policy_desc &d = *desc;
    const int H = d.hidden_dim, Din = d.input_dim, A = d.n_actions, N = d.n_agents;
    if (H != 64 && H != 128) return pfail(nullptr, MRB_E_UNSUPPORTED, "mrb_policy_create: hidden_dim must be 64 or 128");
    if (A < 1 || A > 8 * kMaxAT) return pfail(nullptr, MRB_E_UNSUPPORTED, "mrb_policy_create: n_actions must be in [1, 24]");
    if (N < 1 || N > MRB_MAX_ROBOTS) return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: n_agents must be in [1, 32]");
    if (Din < 1 || Din > 16 * kMaxKS1) return pfail(nullptr, MRB_E_UNSUPPORTED, "mrb_policy_create: input_dim must be in [1, 64]");
    if (Din != d.obs_dim + (d.obs_agent_id ? N : 0))
        return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: input_dim must equal obs_dim (+ n_agents with obs_agent_id): "
                                         "these weights were trained on a different observation layout");
    const int sets = d.non_shared ? N : 1;
    const int64_t per_set = weight_set_floats(H, Din, A, d.use_rnn != 0);
    if (num_weights != per_set * sets)
        return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: weight count does not match the descriptor");
    int ndev = 0;
    cudaError_t st = cudaGetDeviceCount(&ndev);
    if (st != cudaSuccess || ndev == 0) return pfail(nullptr, MRB_E_CUDA, "mrb_policy_create: no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: bad device index");
    cudaDeviceProp prop;
    if ((st = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return pfail(nullptr, MRB_E_CUDA, cudaGetErrorString(st));
    if (prop.major != 10) return pfail(nullptr, MRB_E_UNSUPPORTED, "mrb_policy_create: kernels are built for sm_100a (B200) only");

    mrb_policy *pol = new (std::nothrow) mrb_policy();
    if (!pol) return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: out of host memory");
    pol->d = d;
    pol->device = device;
    pol->num_weights = num_weights;
    pol->wpack = nullptr;
    pol->tc2_img = nullptr;
    pol->w32 = nullptr;
    pol->num_sms = 0;

    // mma.sync path (policy_act_kernel, wpack_word)
    const int KS1 = (Din + 15) / 16, NT = H / 8, KS = H / 16, AT = (A + 7) / 8, G = d.use_rnn ? 6 : 1;
    const int szW1 = NT * KS1 * 64, szW2 = AT * KS * 64, NB = d.use_rnn ? 6 * H : H;
    const int head = szW1 + H + NB + szW2 + AT * 8;
    const int chunk = G * KS * 64;
    PolicyParams &p = pol->p;
    p.set_floats = head + (int64_t)NT * chunk; p.B = 0;
    p.obs_dim = d.obs_dim; p.input_dim = Din; p.n_actions = A; p.n_agents = N;
    p.obs_agent_id = d.obs_agent_id; p.non_shared = d.non_shared;
    p.KS1 = KS1; p.AT = AT; p.szW1 = szW1; p.szW2 = szW2; p.head_floats = head;
    pol->smem_bytes = sizeof(float) * ((size_t)head + 2 * (size_t)chunk);

    // persistent tcgen05 path (policy_tc2.cuh image_word)
    mrb::tc2::Params2 &tcp2 = pol->tcp2;
    std::memset(&tcp2, 0, sizeof(tcp2));
    const int dp = (Din + 15) & ~15;
    pol->tc2_smem = mrb::tc2::smem_bytes(dp, A);
    const bool use_tc2 = !d.accurate && H == 128 && d.use_rnn && dp <= mrb::tc::kMaxKp1 && A <= mrb::tc2::kMaxA && mrb::tc2::ring_depth(dp, A) >= 2;
    if (use_tc2) {
        const int headf = mrb::tc2::head_floats(dp, A);
        tcp2.set_bytes = 4LL * headf + (int64_t)mrb::tc2::kSlabsPerTile * mrb::tc2::kHalfSlabBytes;
        tcp2.obs_dim = d.obs_dim; tcp2.input_dim = Din; tcp2.n_actions = A; tcp2.n_agents = N;
        tcp2.obs_agent_id = d.obs_agent_id; tcp2.non_shared = d.non_shared; tcp2.dp = dp; tcp2.head_bytes = 4 * headf;
        tcp2.ring_off = mrb::tc2::ring_offset(dp, A); tcp2.ring = mrb::tc2::ring_depth(dp, A);
    }

    // float32 path (policy_f32.cuh image_value)
    mrb::f32::Params32 &p32 = pol->p32;
    std::memset(&p32, 0, sizeof(p32));
    if (d.accurate) {
        p32.set_floats = mrb::f32::image_floats(H, Din, A, d.use_rnn != 0, &p32);
        p32.obs_dim = d.obs_dim; p32.input_dim = Din; p32.n_actions = A; p32.n_agents = N;
        p32.obs_agent_id = d.obs_agent_id; p32.non_shared = d.non_shared;
    }

    PackParams &k = pol->pack;
    std::memset(&k, 0, sizeof(k));
    k.per_set = per_set; k.H = H; k.Din = Din; k.A = A; k.rnn = d.use_rnn != 0;
    k.n_wpack = p.set_floats * sets;
    k.n_tc2 = use_tc2 ? tcp2.set_bytes / 4 * sets : 0;
    k.n_w32 = d.accurate ? p32.set_floats * sets : 0;
    k.tc2_set_words = tcp2.set_bytes / 4; k.dp = dp;
    k.p = p; k.p32 = p32;

    // images, then the weights uploaded once to a temporary buffer that the pack kernel reads; synchronous
    float *wdev = nullptr;
    if ((st = cudaSetDevice(device)) != cudaSuccess ||
        (st = cudaMalloc(&pol->wpack, sizeof(float) * k.n_wpack)) != cudaSuccess ||
        (use_tc2 && (st = cudaMalloc(&pol->tc2_img, 4 * k.n_tc2)) != cudaSuccess) ||
        (use_tc2 && (st = cudaDeviceGetAttribute(&pol->num_sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) ||
        (d.accurate && (st = cudaMalloc(&pol->w32, sizeof(float) * k.n_w32)) != cudaSuccess) ||
        (st = cudaMalloc(&wdev, sizeof(float) * num_weights)) != cudaSuccess ||
        (st = cudaMemcpy(wdev, weights, sizeof(float) * num_weights, cudaMemcpyHostToDevice)) != cudaSuccess) {
        const std::string msg = std::string("mrb_policy_create: ") + cudaGetErrorString(st);
        if (wdev) cudaFree(wdev);
        free_images(pol);
        return pfail(nullptr, MRB_E_CUDA, msg);
    }
    k.wpack = reinterpret_cast<uint32_t *>(pol->wpack);
    k.tc2 = reinterpret_cast<uint32_t *>(pol->tc2_img);
    k.w32 = reinterpret_cast<uint32_t *>(pol->w32);
    p.wpack = pol->wpack;
    tcp2.img = pol->tc2_img;
    p32.w = pol->w32;
    if ((st = launch_pack(pol, wdev, 0)) != cudaSuccess || (st = cudaStreamSynchronize(0)) != cudaSuccess) {
        const std::string msg = std::string("mrb_policy_create: weight packing: ") + cudaGetErrorString(st);
        cudaFree(wdev);
        free_images(pol);
        return pfail(nullptr, MRB_E_CUDA, msg);
    }
    count_launch();
    cudaFree(wdev);
    *out = pol;
    return MRB_OK;
}

extern "C" int mrb_policy_load(mrb_policy *pol, const float *weights, int64_t num_weights, void *stream)
{
    if (!pol) return pfail(nullptr, MRB_E_ARG, "mrb_policy_load: null policy");
    if (!weights) return pfail(pol, MRB_E_ARG, "mrb_policy_load: null weights");
    if (num_weights != pol->num_weights)
        return pfail(pol, MRB_E_ARG, "mrb_policy_load: " + std::to_string(num_weights) + " weights given, the policy was created with " +
                                     std::to_string(pol->num_weights));
    if (((uintptr_t)weights & 3) != 0) return pfail(pol, MRB_E_ARG, "mrb_policy_load: weights must be 4-byte aligned");
    cudaPointerAttributes attr;
    cudaError_t st = cudaPointerGetAttributes(&attr, weights);
    if (st != cudaSuccess) {
        cudaGetLastError();
        return pfail(pol, MRB_E_ARG, std::string("mrb_policy_load: weights: ") + cudaGetErrorString(st));
    }
    if (attr.type != cudaMemoryTypeDevice || attr.device != pol->device)
        return pfail(pol, MRB_E_ARG, "mrb_policy_load: weights must be device memory of the policy's device " + std::to_string(pol->device));
    if ((st = cudaSetDevice(pol->device)) != cudaSuccess || (st = launch_pack(pol, weights, (cudaStream_t)stream)) != cudaSuccess)
        return pfail(pol, MRB_E_CUDA, std::string("mrb_policy_load: ") + cudaGetErrorString(st));
    count_launch();
    return MRB_OK;
}

extern "C" int mrb_policy_destroy(mrb_policy *p)
{
    if (!p) return MRB_E_ARG;
    cudaSetDevice(p->device);
    free_images(p);
    return MRB_OK;
}

template <int H, bool RNN>
static cudaError_t launch_policy(const mrb_policy *pol, const PolicyParams &p, const float *obs, float *hidden, int32_t *actions,
                                 float *q, const uint8_t *fresh, cudaStream_t s)
{
    cudaError_t st = cudaFuncSetAttribute(policy_act_kernel<H, RNN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pol->smem_bytes);
    if (st != cudaSuccess) return st;
    const dim3 grid((unsigned)((p.B + kPolicyWarps * 16 - 1) / (kPolicyWarps * 16)), (unsigned)p.n_agents);
    policy_act_kernel<H, RNN><<<grid, kPolicyWarps * 32, pol->smem_bytes, s>>>(p, obs, hidden, actions, q, fresh);
    return cudaGetLastError();
}

extern "C" int mrb_policy_act(mrb_policy *pol, int64_t num_envs, const float *obs, float *hidden, int32_t *actions,
                              float *q, const uint8_t *fresh, void *stream)
{
    if (!pol || !obs || !hidden || !actions || num_envs < 1) return pfail(pol, MRB_E_ARG, "mrb_policy_act: bad argument");
    // the tcgen05 kernel moves hidden rows as float4 (the mma.sync kernel as float2): one rule for every path, so that a
    // buffer that works with one model works with all of them
    if (((uintptr_t)hidden & 15) != 0)
        return pfail(pol, MRB_E_ARG, "mrb_policy_act: hidden must be 16-byte aligned (its kernels access it as float4)");
    cudaError_t st = cudaSetDevice(pol->device);
    if (st != cudaSuccess) return pfail(pol, MRB_E_CUDA, cudaGetErrorString(st));
    PolicyParams p = pol->p;
    p.B = num_envs;
    cudaStream_t s = (cudaStream_t)stream;
    if (pol->w32) {                         // float32 arithmetic (desc.accurate)
        mrb::f32::Params32 fp = pol->p32;
        fp.B = num_envs;
        const int H = pol->d.hidden_dim;
        const size_t smem = mrb::f32::smem_bytes(H, fp.input_dim, fp.n_actions);
        const dim3 grid((unsigned)((num_envs + mrb::f32::kRows - 1) / mrb::f32::kRows), (unsigned)fp.n_agents);
        auto launch32 = [&](auto kernel) -> cudaError_t {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            kernel<<<grid, H, smem, s>>>(fp, obs, hidden, actions, q, fresh);
            return cudaGetLastError();
        };
        const bool rnn32 = pol->d.use_rnn != 0;
        if (H == 128) st = rnn32 ? launch32(mrb::f32::policy_act_f32_kernel<128, true>) : launch32(mrb::f32::policy_act_f32_kernel<128, false>);
        else st = rnn32 ? launch32(mrb::f32::policy_act_f32_kernel<64, true>) : launch32(mrb::f32::policy_act_f32_kernel<64, false>);
        if (st != cudaSuccess) return pfail(pol, MRB_E_CUDA, std::string("policy kernel launch: ") + cudaGetErrorString(st));
        count_launch();
        return MRB_OK;
    }
    // MRB_POLICY_TC=0 forces the mma.sync kernel for models that the persistent tcgen05 kernel covers
    static const bool tc_off = [] { const char *e = std::getenv("MRB_POLICY_TC"); return e && e[0] == '0'; }();
    if (pol->tc2_img && !tc_off) {
        mrb::tc2::Params2 tp = pol->tcp2;
        tp.B = num_envs;
        const int N = tp.n_agents;
        tp.num_tiles = (int)((num_envs + mrb::tc::kRows - 1) / mrb::tc::kRows) * N;
        // one persistent CTA per SM; a multiple of n_agents so that a CTA only ever sees one agent index (per-agent
        // weight sets keep their head resident)
        int grid = pol->num_sms / N * N;
        if (grid < N) grid = N;
        if (grid > tp.num_tiles) grid = tp.num_tiles;
        auto launch = [&](auto kernel) -> cudaError_t {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pol->tc2_smem);
            if (e != cudaSuccess) return e;
            kernel<<<grid, mrb::tc2::kThreads2, pol->tc2_smem, s>>>(tp, obs, hidden, actions, q, fresh);
            return cudaGetLastError();
        };
        st = launch(mrb::tc2::policy_act_tc2_kernel);
        if (st != cudaSuccess) return pfail(pol, MRB_E_CUDA, std::string("policy kernel launch: ") + cudaGetErrorString(st));
        count_launch();
        return MRB_OK;
    }
    const bool rnn = pol->d.use_rnn != 0;
    if (pol->d.hidden_dim == 128) st = rnn ? launch_policy<128, true>(pol, p, obs, hidden, actions, q, fresh, s)
                                            : launch_policy<128, false>(pol, p, obs, hidden, actions, q, fresh, s);
    else st = rnn ? launch_policy<64, true>(pol, p, obs, hidden, actions, q, fresh, s)
                  : launch_policy<64, false>(pol, p, obs, hidden, actions, q, fresh, s);
    if (st != cudaSuccess) return pfail(pol, MRB_E_CUDA, std::string("policy kernel launch: ") + cudaGetErrorString(st));
    count_launch();
    return MRB_OK;
}
