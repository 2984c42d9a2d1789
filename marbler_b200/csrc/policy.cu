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
// produces h'.  Weights are rounded to FP16 and laid out in fragment order ONCE on the host
// (mrb_policy_create), so staging them is a linear cp.async copy and every B fragment pair is a single
// conflict-free 128-bit shared load; the GRU weights (6 H^2 halves, 197 KB for H = 128) stream through a
// double-buffered 2 x 12.3 KB window, one 8-unit column tile at a time.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

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

}  // namespace mrb

// ------------------------------------------------------------------------------------------------ host side
using namespace mrb;

struct mrb_policy {
    mrb_policy_desc d;
    int device;
    float *wpack;
    uint8_t *tc2_img;           // persistent tcgen05 path (policy_tc2.cuh), NULL when the model does not fit it
    mrb::tc2::Params2 tcp2;
    size_t tc2_smem;
    int num_sms;
    PolicyParams p;
    size_t smem_bytes;
    float *w32;                 // float32 path (policy_f32.cuh), only when desc.accurate
    mrb::f32::Params32 p32;
    std::string err;
};

static std::string g_policy_create_error;
namespace mrb { void count_launch(); }       // capi.cu: the library-wide launch counter

static int pfail(mrb_policy *p, int code, const std::string &msg)
{
    if (p) p->err = msg; else g_policy_create_error = msg;
    return code;
}

// B fragment of W' for 8-column tile j, 16-wide k-step s (W in torch layout [out][in]; rows >= rows_valid and
// columns >= cols_valid read as zero): lane (g, t) holds b0 = {W[r][16s+2t], W[r][16s+2t+1]} and
// b1 = {W[r][16s+2t+8], W[r][16s+2t+9]} with r = row0 + 8j + g, each pair rounded to FP16 and packed low | high
static uint32_t h2bits(float lo, float hi)
{
    const uint32_t a = __half_as_ushort(__float2half_rn(lo)), b = __half_as_ushort(__float2half_rn(hi));
    return a | (b << 16);
}
static void frag(const float *W, int ld, int row0, int rows_valid, int cols_valid, int j, int s, int lane, float &b0, float &b1)
{
    const int g = lane >> 2, t = lane & 3, r = 8 * j + g;
    auto at = [&](int k) { return (r < rows_valid && k < cols_valid) ? W[(size_t)(row0 + r) * ld + k] : 0.f; };
    const int k0 = 16 * s + 2 * t;
    const uint32_t u0 = h2bits(at(k0), at(k0 + 1)), u1 = h2bits(at(k0 + 8), at(k0 + 9));
    std::memcpy(&b0, &u0, 4);
    std::memcpy(&b1, &u1, 4);
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
    const int64_t per_set = (int64_t)H * Din + H + (d.use_rnn ? 2LL * 3 * H * H + 2 * 3 * H : (int64_t)H * H + H) + (int64_t)A * H + A;
    if (num_weights != per_set * sets)
        return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: weight count does not match the descriptor");
    int ndev = 0;
    cudaError_t st = cudaGetDeviceCount(&ndev);
    if (st != cudaSuccess || ndev == 0) return pfail(nullptr, MRB_E_CUDA, "mrb_policy_create: no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: bad device index");
    cudaDeviceProp prop;
    if ((st = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return pfail(nullptr, MRB_E_CUDA, cudaGetErrorString(st));
    if (prop.major != 10) return pfail(nullptr, MRB_E_UNSUPPORTED, "mrb_policy_create: kernels are built for sm_100a (B200) only");

    const int KS1 = (Din + 15) / 16, NT = H / 8, KS = H / 16, AT = (A + 7) / 8, G = d.use_rnn ? 6 : 1;
    const int szW1 = NT * KS1 * 64, szW2 = AT * KS * 64, NB = d.use_rnn ? 6 * H : H;
    const int head = szW1 + H + NB + szW2 + AT * 8;
    const int chunk = G * KS * 64;
    const int64_t set_floats = head + (int64_t)NT * chunk;
    std::vector<float> img((size_t)set_floats * sets, 0.f);
    for (int sidx = 0; sidx < sets; sidx++) {
        const float *w = weights + per_set * sidx;
        const float *fc1w = w, *fc1b = fc1w + (size_t)H * Din;
        const float *rw = fc1b + H;
        const float *wih = rw, *whh = nullptr, *bih = nullptr, *bhh = nullptr, *fc2w = nullptr;
        if (d.use_rnn) { whh = wih + (size_t)3 * H * H; bih = whh + (size_t)3 * H * H; bhh = bih + 3 * H; fc2w = bhh + 3 * H; }
        else { bih = wih + (size_t)H * H; fc2w = bih + H; }
        const float *fc2b = fc2w + (size_t)A * H;
        float *o = img.data() + (size_t)set_floats * sidx;
        float *oW1 = o, *oB1 = oW1 + szW1, *oBias = oB1 + H, *oW2 = oBias + NB, *oB2 = oW2 + szW2, *oCh = o + head;
        for (int j = 0; j < NT; j++)
            for (int s = 0; s < KS1; s++)
                for (int l = 0; l < 32; l++)
                    frag(fc1w, Din, 0, H, Din, j, s, l, oW1[((j * KS1 + s) * 32 + l) * 2], oW1[((j * KS1 + s) * 32 + l) * 2 + 1]);
        std::memcpy(oB1, fc1b, sizeof(float) * H);
        if (d.use_rnn) { std::memcpy(oBias, bih, sizeof(float) * 3 * H); std::memcpy(oBias + 3 * H, bhh, sizeof(float) * 3 * H); }
        else std::memcpy(oBias, bih, sizeof(float) * H);
        for (int jt = 0; jt < AT; jt++)
            for (int s = 0; s < KS; s++)
                for (int l = 0; l < 32; l++)
                    frag(fc2w, H, 0, A, H, jt, s, l, oW2[((jt * KS + s) * 32 + l) * 2], oW2[((jt * KS + s) * 32 + l) * 2 + 1]);
        for (int a = 0; a < A; a++) oB2[a] = fc2b[a];
        for (int j = 0; j < NT; j++)
            for (int gi = 0; gi < G; gi++) {
                const float *W = d.use_rnn ? (gi < 3 ? wih : whh) : wih;
                const int row0 = d.use_rnn ? (gi % 3) * H : 0;
                for (int sp = 0; sp < KS / 2; sp++)
                    for (int l = 0; l < 32; l++) {
                        float *q = oCh + (size_t)j * chunk + ((size_t)(gi * (KS / 2) + sp) * 32 + l) * 4;
                        frag(W, H, row0, H, H, j, 2 * sp, l, q[0], q[1]);
                        frag(W, H, row0, H, H, j, 2 * sp + 1, l, q[2], q[3]);
                    }
            }
    }
    // persistent tcgen05 path: head = W1 FP16 [128][dp + 8] | biases | W2 [A][128] as FP32 values rounded to FP16, then twelve
    // 64 x 128 FP16 half slabs in the order the kernel consumes them (pass, gate r / z / n, W_ih then W_hh)
    std::vector<uint8_t> tc2img;
    mrb::tc2::Params2 tcp2;
    std::memset(&tcp2, 0, sizeof(tcp2));
    const int dp = (Din + 15) & ~15;
    const size_t tc2_smem = mrb::tc2::smem_bytes(dp, A);
    const bool use_tc2 = !d.accurate && H == 128 && d.use_rnn && dp <= mrb::tc::kMaxKp1 && A <= mrb::tc2::kMaxA && mrb::tc2::ring_depth(dp, A) >= 2;
    // float32 path: transposed float32 copies of every matrix (policy_f32.cuh)
    std::vector<float> img32;
    mrb::f32::Params32 p32;
    std::memset(&p32, 0, sizeof(p32));
    if (d.accurate) {
        const int64_t sf = mrb::f32::image_floats(H, Din, A, d.use_rnn != 0, &p32);
        img32.assign((size_t)sf * sets, 0.f);
        for (int sidx = 0; sidx < sets; sidx++) {
            const float *w = weights + per_set * sidx;
            const float *fc1w = w, *fc1b = fc1w + (size_t)H * Din, *rw = fc1b + H;
            float *o = img32.data() + (size_t)sf * sidx;
            for (int u = 0; u < H; u++)
                for (int k = 0; k < Din; k++) o[(size_t)k * H + u] = fc1w[(size_t)u * Din + k];
            std::memcpy(o + p32.off_b1, fc1b, sizeof(float) * H);
            const float *fc2w;
            if (d.use_rnn) {
                const float *wih = rw, *whh = wih + (size_t)3 * H * H, *bih = whh + (size_t)3 * H * H, *bhh = bih + 3 * H;
                for (int g = 0; g < 3; g++)
                    for (int u = 0; u < H; u++)
                        for (int k = 0; k < H; k++) {
                            o[p32.off_wih + ((size_t)g * H + k) * H + u] = wih[((size_t)g * H + u) * H + k];
                            o[p32.off_whh + ((size_t)g * H + k) * H + u] = whh[((size_t)g * H + u) * H + k];
                        }
                std::memcpy(o + p32.off_bias, bih, sizeof(float) * 3 * H);
                std::memcpy(o + p32.off_bias + 3 * H, bhh, sizeof(float) * 3 * H);
                fc2w = bhh + 3 * H;
            } else {
                const float *wl = rw, *bl = wl + (size_t)H * H;
                for (int u = 0; u < H; u++)
                    for (int k = 0; k < H; k++) o[p32.off_wih + (size_t)k * H + u] = wl[(size_t)u * H + k];
                std::memcpy(o + p32.off_bias, bl, sizeof(float) * H);
                fc2w = bl + H;
            }
            std::memcpy(o + p32.off_w2, fc2w, sizeof(float) * (size_t)A * H);
            std::memcpy(o + p32.off_b2, fc2w + (size_t)A * H, sizeof(float) * A);
        }
        p32.set_floats = sf; p32.obs_dim = d.obs_dim; p32.input_dim = Din; p32.n_actions = A; p32.n_agents = N;
        p32.obs_agent_id = d.obs_agent_id; p32.non_shared = d.non_shared;
    }
    if (use_tc2) {
        const int headf = mrb::tc2::head_floats(dp, A);
        const int64_t setb = 4LL * headf + (int64_t)mrb::tc2::kSlabsPerTile * mrb::tc2::kHalfSlabBytes;
        tc2img.assign((size_t)setb * sets, 0);
        auto r16 = [](float v) { return __half2float(__float2half_rn(v)); };
        for (int sidx = 0; sidx < sets; sidx++) {
            const float *w = weights + per_set * sidx;
            const float *fc1w = w, *fc1b = fc1w + (size_t)H * Din, *wih = fc1b + H, *whh = wih + (size_t)3 * H * H;
            const float *bih = whh + (size_t)3 * H * H, *bhh = bih + 3 * H, *fc2w = bhh + 3 * H, *fc2b = fc2w + (size_t)A * H;
            uint8_t *o = tc2img.data() + (size_t)setb * sidx;
            float *hf = reinterpret_cast<float *>(o);
            __half *w1h = reinterpret_cast<__half *>(o);
            for (int u = 0; u < H; u++)
                for (int k = 0; k < Din; k++) w1h[(size_t)u * mrb::tc2::w1_stride(dp) + k] = __float2half_rn(fc1w[(size_t)u * Din + k]);
            float *bo = hf + mrb::tc2::head_bias(dp);
            std::memcpy(bo, fc1b, sizeof(float) * H);
            std::memcpy(bo + H, bih, sizeof(float) * 3 * H);
            std::memcpy(bo + 4 * H, bhh, sizeof(float) * 3 * H);
            for (int a = 0; a < A; a++) bo[7 * H + a] = fc2b[a];
            float *w2 = hf + mrb::tc2::head_w2(dp);
            for (int a = 0; a < A; a++)
                for (int k = 0; k < H; k++) w2[(size_t)a * H + k] = r16(fc2w[(size_t)a * H + k]);
            uint8_t *slabs = o + 4 * (size_t)headf;
            for (int pass = 0; pass < 2; pass++)
                for (int g = 0; g < 6; g++)
                    mrb::tc::pack_canonical(slabs + (size_t)(pass * 6 + g) * mrb::tc2::kHalfSlabBytes, (g & 1) ? whh : wih, H,
                                            (g >> 1) * H + pass * mrb::tc2::kHalf, mrb::tc2::kHalf, H, mrb::tc2::kHalf, H);
        }
        tcp2.set_bytes = setb; tcp2.obs_dim = d.obs_dim; tcp2.input_dim = Din; tcp2.n_actions = A; tcp2.n_agents = N;
        tcp2.obs_agent_id = d.obs_agent_id; tcp2.non_shared = d.non_shared; tcp2.dp = dp; tcp2.head_bytes = 4 * headf;
        tcp2.ring_off = mrb::tc2::ring_offset(dp, A); tcp2.ring = mrb::tc2::ring_depth(dp, A);
    }
    mrb_policy *pol = new (std::nothrow) mrb_policy();
    if (!pol) return pfail(nullptr, MRB_E_ARG, "mrb_policy_create: out of host memory");
    pol->d = d;
    pol->device = device;
    pol->wpack = nullptr;
    pol->tc2_img = nullptr;
    pol->tcp2 = tcp2;
    pol->tc2_smem = tc2_smem;
    pol->num_sms = 0;
    pol->w32 = nullptr;
    pol->p32 = p32;
    if ((st = cudaSetDevice(device)) != cudaSuccess || (st = cudaMalloc(&pol->wpack, img.size() * sizeof(float))) != cudaSuccess ||
        (st = cudaMemcpy(pol->wpack, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice)) != cudaSuccess) {
        const std::string msg = std::string("mrb_policy_create: ") + cudaGetErrorString(st);
        if (pol->wpack) cudaFree(pol->wpack);
        delete pol;
        return pfail(nullptr, MRB_E_CUDA, msg);
    }
    if (use_tc2) {
        if ((st = cudaMalloc(&pol->tc2_img, tc2img.size())) != cudaSuccess ||
            (st = cudaMemcpy(pol->tc2_img, tc2img.data(), tc2img.size(), cudaMemcpyHostToDevice)) != cudaSuccess ||
            (st = cudaDeviceGetAttribute(&pol->num_sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) {
            const std::string msg = std::string("mrb_policy_create: ") + cudaGetErrorString(st);
            if (pol->tc2_img) cudaFree(pol->tc2_img);
            cudaFree(pol->wpack);
            delete pol;
            return pfail(nullptr, MRB_E_CUDA, msg);
        }
        pol->tcp2.img = pol->tc2_img;
    }
    if (d.accurate) {
        if ((st = cudaMalloc(&pol->w32, img32.size() * sizeof(float))) != cudaSuccess ||
            (st = cudaMemcpy(pol->w32, img32.data(), img32.size() * sizeof(float), cudaMemcpyHostToDevice)) != cudaSuccess) {
            const std::string msg = std::string("mrb_policy_create: ") + cudaGetErrorString(st);
            if (pol->w32) cudaFree(pol->w32);
            cudaFree(pol->wpack);
            delete pol;
            return pfail(nullptr, MRB_E_CUDA, msg);
        }
        pol->p32.w = pol->w32;
    }
    PolicyParams &p = pol->p;
    p.wpack = pol->wpack; p.set_floats = set_floats; p.B = 0;
    p.obs_dim = d.obs_dim; p.input_dim = Din; p.n_actions = A; p.n_agents = N;
    p.obs_agent_id = d.obs_agent_id; p.non_shared = d.non_shared;
    p.KS1 = KS1; p.AT = AT; p.szW1 = szW1; p.szW2 = szW2; p.head_floats = head;
    pol->smem_bytes = sizeof(float) * ((size_t)head + 2 * (size_t)chunk);
    *out = pol;
    return MRB_OK;
}

extern "C" int mrb_policy_destroy(mrb_policy *p)
{
    if (!p) return MRB_E_ARG;
    cudaSetDevice(p->device);
    if (p->wpack) cudaFree(p->wpack);
    if (p->tc2_img) cudaFree(p->tc2_img);
    if (p->w32) cudaFree(p->w32);
    delete p;
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
