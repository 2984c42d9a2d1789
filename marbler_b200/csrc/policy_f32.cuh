// Float32 policy step: the same network as policy.cu / policy_tc2.cuh (utilities/rnn_agent.py:5-29 RNNAgent,
// utilities/rnn_ns_agent.py:5-36 RNNNSAgent, driven as utilities/misc.py:155-170 drives them) evaluated in the
// reference's own arithmetic - float32 operands, float32 FMA accumulation, expf / tanhf gates - instead of FP16
// tensor-core operands.  mrb_policy_desc.accurate = 1 selects it.  The tensor-core kernels agree with the reference
// to ~1e-3 |q| (FP16 rounding of weights and activations), which flips about one greedy decision in a thousand at
// near-ties; this kernel agrees to float32 rounding (different summation order only), so the greedy actions of the
// shipped checkpoints are the reference's.  It costs ~10x the tensor-core kernel and is meant for evaluation runs
// that have to reproduce the reference's action sequence, not for throughput.
//
// Mapping: blockIdx.y = agent (one weight set per CTA), blockIdx.x = a tile of RB consecutive envs; one thread per
// hidden unit.  A thread accumulates its unit's pre-activations for all RB rows (6 gates x RB accumulators), reading
// the weights from transposed copies (Wt[k][unit]: consecutive threads, consecutive addresses) and the activations
// of the RB rows as shared-memory broadcasts.
#pragma once
#include "common.cuh"

namespace mrb {
namespace f32 {

struct Params32 {
    const float *w;              // device image, `set_floats` per weight set (layout: offsets below)
    int64_t set_floats, B;
    int32_t obs_dim, input_dim, n_actions, n_agents, obs_agent_id, non_shared;
    int32_t off_b1, off_wih, off_whh, off_bias, off_w2, off_b2;      // W1t at 0
};

constexpr int kRows = 16;        // envs (rows of one agent) per CTA

// image of one weight set (floats): W1t [Din][H] | b1 [H] | Wih_t [3][H][H] (gate, k, unit) | Whh_t [3][H][H] |
// biases (b_ih [3H] | b_hh [3H], or b [H]) | W2 [A][H] | b2 [A];  without a GRU: Wih_t is W_t [H][H], no Whh_t
inline int64_t image_floats(int H, int Din, int A, bool rnn, Params32 *p)
{
    int64_t o = (int64_t)Din * H;
    if (p) p->off_b1 = (int32_t)o;
    o += H;
    if (p) p->off_wih = (int32_t)o;
    o += (int64_t)(rnn ? 3 : 1) * H * H;
    if (p) p->off_whh = (int32_t)o;
    if (rnn) o += 3LL * H * H;
    if (p) p->off_bias = (int32_t)o;
    o += rnn ? 6 * H : H;
    if (p) p->off_w2 = (int32_t)o;
    o += (int64_t)A * H;
    if (p) p->off_b2 = (int32_t)o;
    o += A;
    return o;
}

// float o of the image of one weight set (layout above), built on the device by policy_pack_kernel (policy.cu)
__device__ __forceinline__ float image_value(const WeightSet &w, const Params32 &p, int H, bool rnn, int64_t o)
{
    if (o < p.off_b1) return w.fc1w[(size_t)(o % H) * p.input_dim + o / H];
    if (o < p.off_wih) return w.fc1b[o - p.off_b1];
    if (o < p.off_bias) {                                           // (gate, k, unit) <- [gate * H + unit][k]
        const bool hh = o >= p.off_whh;
        const int64_t i = o - (hh ? p.off_whh : p.off_wih), g = i / ((int64_t)H * H), k = (i / H) % H, u = i % H;
        return (hh ? w.whh : w.wih)[(size_t)(g * H + u) * H + k];
    }
    if (o < p.off_w2) {
        const int i = (int)(o - p.off_bias);
        return rnn && i >= 3 * H ? w.bhh[i - 3 * H] : w.bih[i];
    }
    if (o < p.off_b2) return w.fc2w[o - p.off_w2];
    return w.fc2b[o - p.off_b2];
}

__device__ __forceinline__ float sigmoid_(float x) { return 1.f / (1.f + expf(-x)); }

template <int H, bool RNN>
__global__ void __launch_bounds__(H) policy_act_f32_kernel(const Params32 p, const float *__restrict__ obs, float *hidden,
                                                          int32_t *__restrict__ actions, float *__restrict__ q_out,
                                                          const uint8_t *__restrict__ fresh)
{
    constexpr int RB = kRows;
    extern __shared__ __align__(16) float sm[];
    const int Din = p.input_dim, D = p.obs_dim, N = p.n_agents, A = p.n_actions;
    const int DinP = (Din + 3) & ~3;
    float *s_in = sm;                        // [RB][DinP]
    float *s_x = s_in + RB * DinP;           // [RB][H]   relu(fc1)
    float *s_h = s_x + RB * H;               // [RB][H]   hidden state in
    float *s_hn = s_h + RB * H;              // [RB][H]   hidden state out
    float *s_q = s_hn + RB * H;              // [RB][A]
    const int u = threadIdx.x, agent = blockIdx.y;
    const int64_t e0 = (int64_t)blockIdx.x * RB;
    const float *w = p.w + (size_t)(p.non_shared ? agent : 0) * p.set_floats;

    // ---- inputs: observation (+ one-hot agent id, misc.py:161-162) and hidden state; rows past the end or flagged
    //      fresh (run_env re-zeroes hs and feeds reset()'s all-zero observation, misc.py:156,219) read as zero
    for (int i = u; i < RB * DinP; i += H) {
        const int r = i / DinP, c = i - r * DinP;
        const int64_t e = e0 + r;
        float v = 0.f;
        if (e < p.B && c < Din) {
            const bool z = fresh && fresh[e];
            if (c < D) v = z ? 0.f : obs[(e * N + agent) * D + c];
            else v = (p.obs_agent_id && c - D == agent) ? 1.f : 0.f;
        }
        s_in[i] = v;
    }
#pragma unroll
    for (int r = 0; r < RB; r++) {
        const int64_t e = e0 + r;
        float v = 0.f;
        if (e < p.B && !(fresh && fresh[e])) v = hidden[(e * N + agent) * H + u];
        s_h[r * H + u] = v;
    }
    __syncthreads();

    // ---- fc1 + ReLU (rnn_agent.py:22)
    {
        float acc[RB];
        const float b = w[p.off_b1 + u];
#pragma unroll
        for (int r = 0; r < RB; r++) acc[r] = 0.f;
        for (int k = 0; k < Din; k++) {
            const float wk = w[(size_t)k * H + u];
#pragma unroll
            for (int r = 0; r < RB; r++) acc[r] = fmaf(s_in[r * DinP + k], wk, acc[r]);
        }
#pragma unroll
        for (int r = 0; r < RB; r++) s_x[r * H + u] = fmaxf(acc[r] + b, 0.f);
    }
    __syncthreads();

    // ---- recurrent layer (rnn_agent.py:24-27): GRUCell, or Linear + ReLU
    if (RNN) {
        float ir[RB], iz[RB], in_[RB], hr[RB], hz[RB], hn[RB];
#pragma unroll
        for (int r = 0; r < RB; r++) { ir[r] = iz[r] = in_[r] = hr[r] = hz[r] = hn[r] = 0.f; }
        const float *wih = w + p.off_wih, *whh = w + p.off_whh;
        for (int k = 0; k < H; k += 4) {
            float wi[3][4], wh[3][4];
#pragma unroll
            for (int g = 0; g < 3; g++)
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    wi[g][j] = wih[((size_t)g * H + k + j) * H + u];
                    wh[g][j] = whh[((size_t)g * H + k + j) * H + u];
                }
#pragma unroll
            for (int r = 0; r < RB; r++) {
                const float4 xv = *reinterpret_cast<const float4 *>(s_x + r * H + k);
                const float4 hv = *reinterpret_cast<const float4 *>(s_h + r * H + k);
                const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, hs[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    ir[r] = fmaf(xs[j], wi[0][j], ir[r]); iz[r] = fmaf(xs[j], wi[1][j], iz[r]); in_[r] = fmaf(xs[j], wi[2][j], in_[r]);
                    hr[r] = fmaf(hs[j], wh[0][j], hr[r]); hz[r] = fmaf(hs[j], wh[1][j], hz[r]); hn[r] = fmaf(hs[j], wh[2][j], hn[r]);
                }
            }
        }
        const float *bias = w + p.off_bias;
        const float bir = bias[u], biz = bias[H + u], bin = bias[2 * H + u];
        const float bhr = bias[3 * H + u], bhz = bias[4 * H + u], bhn = bias[5 * H + u];
#pragma unroll
        for (int r = 0; r < RB; r++) {
            // torch.nn.GRUCell: r = s(W_ir x + b_ir + W_hr h + b_hr), z likewise, n = tanh(W_in x + b_in + r (W_hn h + b_hn)),
            // h' = (1 - z) n + z h
            const float rg = sigmoid_((ir[r] + bir) + (hr[r] + bhr));
            const float zg = sigmoid_((iz[r] + biz) + (hz[r] + bhz));
            const float ng = tanhf((in_[r] + bin) + rg * (hn[r] + bhn));
            const float hv = s_h[r * H + u];
            const float o = (1.f - zg) * ng + zg * hv;
            s_hn[r * H + u] = o;
            const int64_t e = e0 + r;
            if (e < p.B) hidden[(e * N + agent) * H + u] = o;
        }
    } else {
        float acc[RB];
#pragma unroll
        for (int r = 0; r < RB; r++) acc[r] = 0.f;
        const float *wl = w + p.off_wih;
        for (int k = 0; k < H; k++) {
            const float wk = wl[(size_t)k * H + u];
#pragma unroll
            for (int r = 0; r < RB; r++) acc[r] = fmaf(s_x[r * H + k], wk, acc[r]);
        }
        const float b = w[p.off_bias + u];
#pragma unroll
        for (int r = 0; r < RB; r++) {
            const float o = fmaxf(acc[r] + b, 0.f);
            s_hn[r * H + u] = o;
            const int64_t e = e0 + r;
            if (e < p.B) hidden[(e * N + agent) * H + u] = o;
        }
    }
    __syncthreads();

    // ---- fc2 (rnn_agent.py:28) and the greedy action (misc.py:170 np.argmax: first maximum)
    for (int i = u; i < RB * A; i += H) {
        const int r = i / A, a = i - r * A;
        const float *w2 = w + p.off_w2 + (size_t)a * H;
        float acc = 0.f;
        for (int k = 0; k < H; k++) acc = fmaf(s_hn[r * H + k], w2[k], acc);
        s_q[i] = acc + w[p.off_b2 + a];
    }
    __syncthreads();
    if (u < RB) {
        const int64_t e = e0 + u;
        if (e < p.B) {
            int best = 0;
            float bq = s_q[u * A];
            for (int a = 1; a < A; a++) {
                const float v = s_q[u * A + a];
                if (v > bq) { bq = v; best = a; }
            }
            actions[e * N + agent] = best;
            if (q_out)
                for (int a = 0; a < A; a++) q_out[(e * N + agent) * A + a] = s_q[u * A + a];
        }
    }
}

inline size_t smem_bytes(int H, int Din, int A)
{
    const int DinP = (Din + 3) & ~3;
    return sizeof(float) * ((size_t)kRows * DinP + 3 * (size_t)kRows * H + (size_t)kRows * A);
}

}  // namespace f32
}  // namespace mrb
