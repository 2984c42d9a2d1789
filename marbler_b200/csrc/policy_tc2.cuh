// Persistent, warp-specialised tcgen05 / TMEM policy step (hidden 128, GRUCell): the reference's RNNAgent forward
// (utilities/rnn_agent.py:21-29) + greedy argmax (utilities/misc.py:170).  Same arithmetic contract as
// policy_act_kernel (FP16 operands, FP32 accumulation, FP32 gates).
//
// policy_tc.cuh runs its phases one after another in a 4-warp CTA and is slower than the mma.sync kernel: 39 % of
// its stall samples sit in the staging of the hidden state, 22 % in the gate epilogue, < 5 % near the MMAs
// (profiles/r01_ncu_policy_tc_v1_*).  Here one CTA per SM loops over (128-env tile, agent) work items and four
// roles run concurrently, coupled only by mbarriers:
//
//   staging   8 warps  each warp owns 16 rows of the NEXT tile: coalesced global loads of obs / hidden -> FP16 operands
//                      in shared memory (UMMA canonical K-major layout), and fc1 + ReLU as warp-level
//                      mma.sync.m16n8k16 (K <= 64: 1 % of the flops; a tcgen05 fc1 would need a MMA -> epilogue -> MMA
//                      round trip per tile and TMEM columns that the two gate halves occupy); two activation buffers
//   loader    1 thread streams the GRU weights as twelve 64 x 128 FP16 half slabs per tile (cp.async.bulk, 1-D: the
//                      image holds them in the canonical layout, image_word) through a three-deep (two when shared memory is short) 16 KB ring
//   mma       1 thread per tile two half passes of 64 hidden units; a pass is 6 slabs x 8 tcgen05.mma (M 128, N 64,
//                      K 16) into one 256-column half of TMEM: r -> [0,64), z -> [64,128), W_in x -> [128,192),
//                      W_hn h -> [192,256); tcgen05.commit releases slabs, activation buffers and TMEM halves
//   epilogue  8 warps  two per TMEM lane quarter, each with half of a pass's 64 units; thread t of a quarter = tile row =
//                      TMEM lane: tcgen05.ld the four gate accumulators, gates on the SFU, h' -> global through a
//                      per-warp transpose tile, fc2 partial sums on the CUDA cores (A <= 8 actions), argmax after the
//                      second pass.  While it works on one TMEM half the MMAs of the next pass fill the other.
//
// The warps are laid out by warpgroups of four -- epilogue 0 .. 7 | issuer, loader, two idle | staging 12 .. 19 -- so that
// setmaxnreg can move registers from the issuer / loader group (40) and the staging warps (88) to the epilogue (128).
// Every wait on an mbarrier is bounded and traps instead of hanging the GPU.
#pragma once
#include "policy_tc.cuh"

namespace mrb {
namespace tc2 {

using namespace mrb::tc;

constexpr int kHalf = 64;                                  // hidden units per pass
constexpr int kHalfSlabBytes = kHalf * kH * 2;             // 16 KB
constexpr int kSlabsPerTile = 12;                          // 2 passes x (W_ir, W_hr, W_iz, W_hz, W_in, W_hn)
constexpr int kRingMax = 3;                               // weight-ring slots: 3 when they fit, else 2 (Params2::ring)
constexpr int kStageWarps = 8, kEpiWarps = 8;             // kEpiWarps / 4 epilogue warps share a TMEM lane quarter
constexpr int kColGroups = kEpiWarps / 4;                  // ... and split the 64 units of a pass between them
constexpr int kUnitsPerWarp = kHalf / kColGroups;
constexpr int kTileStride = 20;                            // floats per row of an epilogue exchange tile (16 + 4 pad)
// Warp layout by warpgroups of four (setmaxnreg moves registers between WHOLE warpgroups): epilogue warps 0 .. 7, then one
// warpgroup holding the MMA issuer, the weight loader and two idle warps, then the eight staging warps.  The kernel starts
// with 96 registers per thread (640 threads = 61,440 registers, and setmaxnreg only redistributes what the CTA was launched
// with: asking for more blocks forever); the middle warpgroup drops to 40 and the staging warps to 88, which lets the
// epilogue warps rise to 128 (8 x 4096 + 4 x 1280 + 8 x 2816 = 60,416).
constexpr int kMmaWarp = kEpiWarps, kLoadWarp = kEpiWarps + 1, kStageBase = kEpiWarps + 4;
constexpr int kThreads2 = (kStageBase + kStageWarps) * 32;        // 640
template <int R> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
template <int R> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }
constexpr int kMaxA = 8;                                  // fc2 runs on the CUDA cores of the epilogue warps

struct Params2 {
    const uint8_t *img;       // packed weight sets (device): head | 12 half slabs
    int64_t set_bytes;
    int64_t B;
    int32_t obs_dim, input_dim, n_actions, n_agents, obs_agent_id, non_shared;
    int32_t dp;               // input_dim rounded up to a multiple of 16 (fc1 k extent)
    int32_t head_bytes;       // W1 f16 [128][dp + 8] | b1 | b_ih | b_hh | b2 [32] | W2 f32 [n_actions][128] (FP16-rounded values)
    int32_t num_tiles;        // ceil(B / 128) * n_agents
    int32_t ring_off, ring;   // byte offset and depth of the weight ring (after everything else in shared memory)
};

// head offsets in floats; W1 rows are dp + 8 halves long: the 16-byte pad spreads the B-fragment loads over the banks
__host__ __device__ inline int w1_stride(int dp) { return dp + 8; }
__host__ __device__ inline int head_bias(int dp) { return kH * w1_stride(dp) / 2; }
__host__ __device__ inline int head_w2(int dp) { return head_bias(dp) + kBiasFloats; }
__host__ __device__ inline int head_floats(int dp, int n_actions) { return head_w2(dp) + n_actions * kH; }

struct Smem2 {
    static constexpr int act = 0;                                    // 2 x (x | h)
    static constexpr int act_stride = 2 * kActBytes;
    static constexpr int bars = act + 2 * act_stride;                // act_full[2] act_free[2] slab_full[3] slab_empty[3] tmem_full[2] tmem_free[2] head
    static constexpr int tmem_slot = bars + 16 * 8;
    static constexpr int head = tmem_slot + 64;
};
// after the head: one 32-row x 16-unit exchange tile per epilogue warp (old hidden state in, h' out, fc2 partial sums),
// one 16-row x (dp + 8) FP16 scratch per staging warp for the A fragments of fc1, then the weight ring
__host__ __device__ inline int scratch_halves(int dp) { return 16 * w1_stride(dp); }
__host__ inline int ring_offset(int dp, int n_actions)
{
    const size_t end = (size_t)Smem2::head + 4 * (size_t)head_floats(dp, n_actions) + 4 * (size_t)kEpiWarps * 32 * kTileStride +
                       2 * (size_t)kStageWarps * scratch_halves(dp);
    return (int)((end + 127) & ~(size_t)127);
}
// deepest ring that fits the 227 KB a CTA may use (0: the model does not fit this kernel)
__host__ inline int ring_depth(int dp, int n_actions)
{
    for (int r = kRingMax; r >= 2; r--)
        if ((size_t)ring_offset(dp, n_actions) + (size_t)r * kHalfSlabBytes <= 227 * 1024) return r;
    return 0;
}
__host__ inline size_t smem_bytes(int dp, int n_actions) { return (size_t)ring_offset(dp, n_actions) + (size_t)ring_depth(dp, n_actions) * kHalfSlabBytes; }

// Word o (4 bytes) of the image of one weight set, built on the device by policy_pack_kernel (policy.cu):
//   head (head_floats words): W1 FP16 [128][dp + 8] (columns >= input_dim zero) | b1 | b_ih | b_hh | b2 [32] (zero past
//   n_actions) | W2 [n_actions][128] as float32 values rounded to FP16;
//   then twelve 64 x 128 FP16 half slabs in the order the kernel consumes them: pass p, gate r / z / n, W_ih then W_hh
//   (slab 6p + g holds rows (g / 2) * 128 + 64p .. + 63 of (g odd ? W_hh : W_ih)), each in the canonical K-major layout
//   of policy_tc.cuh with LBO = 64 / 8 * 128 = 1,024 bytes: element (r, k) at byte (k / 8) 1024 + (r / 8) 128 + (r % 8) 16 + (k % 8) 2.
__device__ __forceinline__ uint32_t image_word(const WeightSet &w, int Din, int A, int dp, int64_t o)
{
    const int hb = head_bias(dp), hw = head_w2(dp), hf = head_floats(dp, A);
    if (o < hb) {                                                   // W1 row u, columns k, k + 1 (dp + 8 is even)
        const int ws = w1_stride(dp) / 2, u = (int)o / ws, k = 2 * ((int)o % ws);
        const float *row = w.fc1w + (size_t)u * Din;
        return h2(k < Din ? row[k] : 0.f, k + 1 < Din ? row[k + 1] : 0.f);
    }
    if (o < hw) {
        const int i = (int)o - hb;
        const float v = i < kH ? w.fc1b[i] : i < 4 * kH ? w.bih[i - kH] : i < 7 * kH ? w.bhh[i - 4 * kH]
                      : (i - 7 * kH < A ? w.fc2b[i - 7 * kH] : 0.f);
        return __float_as_uint(v);
    }
    if (o < hf) return __float_as_uint(__half2float(__float2half_rn(w.fc2w[o - hw])));
    const int64_t b = 4 * (o - hf);
    const int slab = (int)(b / kHalfSlabBytes), rem = (int)(b % kHalfSlabBytes), pass = slab / 6, g = slab % 6;
    constexpr int lbo = kHalf / 8 * 128;
    const int r = 8 * ((rem % lbo) / 128) + (rem % 128) / 16, k = 8 * (rem / lbo) + (rem % 16) / 2;
    const float *W = ((g & 1) ? w.whh : w.wih) + (size_t)((g >> 1) * kH + pass * kHalf + r) * kH + k;
    return h2(W[0], W[1]);
}
// D = A (16x16, row) * B (16x8, col) + D, FP16 inputs, FP32 accumulate
__device__ __forceinline__ void mma_m16n8k16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void tmem_ld8(uint32_t addr, float (&v)[8])
{
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(addr));
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// mbar_wait with a back-off: the waiting roles share their scheduler with the working ones, and a tight try_wait loop
// was 11 % of all issued instructions (ncu, first version of this kernel)
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(100);
        if (++spins > (1u << 20)) __trap();               // never hang the device on a protocol bug
    }
}
__device__ __forceinline__ void prefetch_l1(const void *ptr) { asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr)); }
__device__ __forceinline__ float round_f16(float v) { return __half2float(__float2half_rn(v)); }

__global__ void __launch_bounds__(kThreads2, 1)
policy_act_tc2_kernel(const Params2 p, const float *__restrict__ obs, float *hidden, int32_t *__restrict__ actions,
                      float *__restrict__ q_out, const uint8_t *__restrict__ fresh)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *sm = smem_raw;
    const uint32_t sbase = smem_u32(sm);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t bar0 = sbase + Smem2::bars;
    const uint32_t act_full = bar0, act_free = bar0 + 16, slab_full = bar0 + 32, slab_empty = bar0 + 56,
                   tmem_full = bar0 + 80, tmem_free = bar0 + 96, head_full = bar0 + 112;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(sm + Smem2::tmem_slot);
    const int N = p.n_agents, D = p.obs_dim, Din = p.input_dim, A = p.n_actions, Dp = p.dp;
    constexpr int AP = kMaxA;                                   // action accumulators per epilogue thread (>= A)
    const uint32_t ring = (uint32_t)p.ring;
    const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp == kEpiWarps) {                                    // the MMA warp owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < 2; i++) {
            mbar_init(act_full + 8 * i, kStageWarps * 32);
            mbar_init(act_free + 8 * i, 1);
            mbar_init(tmem_full + 8 * i, 1);
            mbar_init(tmem_free + 8 * i, kEpiWarps * 32);
        }
        for (int i = 0; i < kRingMax; i++) { mbar_init(slab_full + 8 * i, 1); mbar_init(slab_empty + 8 * i, 1); }
        mbar_init(head_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const float *headf = reinterpret_cast<const float *>(sm + Smem2::head);

    if (warp < kEpiWarps) {
        // ------------------------------------------------------------------------------------------ epilogue
        reg_inc<128>();
        const int quarter = warp & 3, cq = warp >> 2;       // TMEM lane quarter (rows 32 quarter ..); which kUnitsPerWarp units of a pass
        const int row = 32 * quarter + lane;
        const uint32_t lane_base = tmem + ((uint32_t)(32 * quarter) << 16);
        mbar_wait_sleep(head_full, 0);                      // biases and W2 (loaded once: a CTA sees one agent index)
        const float *bias = headf + head_bias(Dp), *W2 = headf + head_w2(Dp);
        const float *b_ih = bias + kH, *b_hh = bias + 4 * kH, *b2 = bias + 7 * kH;
        // per-warp exchange tile, 32 rows x 16 hidden units (row stride kTileStride floats: conflict-free both ways).
        // The old hidden state comes in and h' goes out through it, so that every global access of this role is a
        // run of 64 contiguous bytes per row -- with one thread per row the 16-byte pieces at a 512-byte stride cost
        // a third of the kernel (measured: 13 -> 9.5 us per tile without the stores)
        float *tile = const_cast<float *>(headf) + head_floats(Dp, A) + warp * (32 * kTileStride);
        const int tr = lane >> 2, tc4 = lane & 3;           // transposed access: rows 8 i + tr, floats 4 tc4 .. 4 tc4 + 3
        for (int n = 0; n < my_tiles; n++) {
            const int t = (int)blockIdx.x + n * (int)gridDim.x;
            const int agent = t % N;
            const int64_t e0 = (int64_t)(t / N) * kRows + 32 * quarter;      // env of this warp's first row
            const int64_t e = e0 + lane;
            const bool valid = e < p.B;
            const int my_zero = (!valid || (fresh && fresh[e])) ? 1 : 0;
            const int64_t grow = (valid ? e : 0) * N + agent;
            float qacc[AP];
#pragma unroll
            for (int a = 0; a < AP; a++) qacc[a] = 0.f;
            // rows this lane moves in the transposed phases
            int64_t trow[4];
            bool tvalid[4];
            int tzero[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int64_t er = e0 + 8 * i + tr;
                tvalid[i] = er < p.B;
                trow[i] = (tvalid[i] ? er : 0) * N + agent;
                tzero[i] = __shfl_sync(0xffffffffu, my_zero, 8 * i + tr);
            }
            constexpr int GP = kUnitsPerWarp / 16;          // 16-unit groups per pass
            // old hidden state of a group: loaded one group ahead, so that the L2 round trip runs under the gate math
            float4 ov[4];
#pragma unroll
            for (int i = 0; i < 4; i++) ov[i] = *reinterpret_cast<const float4 *>(hidden + trow[i] * kH + kUnitsPerWarp * cq + 4 * tc4);
#pragma unroll 1
            for (int gi = 0; gi < 2 * GP; gi++) {
                {
                    const int pass = gi / GP, G = gi % GP;
                    const int ub = pass * kHalf + kUnitsPerWarp * cq + 16 * G;       // first hidden unit of this group
                    __syncwarp();                           // the previous group's stores have read the tile
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        *reinterpret_cast<float4 *>(tile + (8 * i + tr) * kTileStride + 4 * tc4) = tzero[i] ? make_float4(0.f, 0.f, 0.f, 0.f) : ov[i];
                    if (gi + 1 < 2 * GP) {
                        const int ubn = ((gi + 1) / GP) * kHalf + kUnitsPerWarp * cq + 16 * ((gi + 1) % GP);
#pragma unroll
                        for (int i = 0; i < 4; i++) ov[i] = *reinterpret_cast<const float4 *>(hidden + trow[i] * kH + ubn + 4 * tc4);
                    }
                    if (G == 0) {
                        mbar_wait_sleep(tmem_full + 8 * pass, (uint32_t)(n & 1));
                        tc_fence_after();
                    }
                    __syncwarp();
                    const uint32_t tb = lane_base + 256 * pass + kUnitsPerWarp * cq + 16 * G;
#pragma unroll 1
                    for (int c = 0; c < 2; c++) {
                        const int u0 = ub + 8 * c;
                        float ar[8], az[8], ai[8], ah[8];
                        tmem_ld8(tb + 8 * c, ar);
                        tmem_ld8(tb + 64 + 8 * c, az);
                        tmem_ld8(tb + 128 + 8 * c, ai);
                        tmem_ld8(tb + 192 + 8 * c, ah);
                        float *mine = tile + lane * kTileStride + 8 * c;
                        const float4 o0 = *reinterpret_cast<const float4 *>(mine), o1 = *reinterpret_cast<const float4 *>(mine + 4);
                        const float old[8] = {o0.x, o0.y, o0.z, o0.w, o1.x, o1.y, o1.z, o1.w};
                        tmem_ld_wait();
                        float hn[8];
#pragma unroll
                        for (int i = 0; i < 8; i++) {
                            const int k = u0 + i;
                            const float r = sigm(ar[i] + b_ih[k] + b_hh[k]);
                            const float z = sigm(az[i] + b_ih[kH + k] + b_hh[kH + k]);
                            const float nn = tanh_(ai[i] + b_ih[2 * kH + k] + r * (ah[i] + b_hh[2 * kH + k]));
                            hn[i] = (1.f - z) * nn + z * old[i];
                        }
                        *reinterpret_cast<float4 *>(mine) = make_float4(hn[0], hn[1], hn[2], hn[3]);
                        *reinterpret_cast<float4 *>(mine + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
                        // fc2 partial sums (rnn_agent.py:28) with FP16-rounded operands, like the tensor-core kernels
#pragma unroll
                        for (int i = 0; i < 8; i++) hn[i] = round_f16(hn[i]);
#pragma unroll
                        for (int a = 0; a < AP; a++) {
                            if (a < A) {
                                const float4 *w = reinterpret_cast<const float4 *>(W2 + a * kH + u0);
                                const float4 w0 = w[0], w1 = w[1];
                                float s = qacc[a];
                                s = fmaf(hn[0], w0.x, s); s = fmaf(hn[1], w0.y, s); s = fmaf(hn[2], w0.z, s); s = fmaf(hn[3], w0.w, s);
                                s = fmaf(hn[4], w1.x, s); s = fmaf(hn[5], w1.y, s); s = fmaf(hn[6], w1.z, s); s = fmaf(hn[7], w1.w, s);
                                qacc[a] = s;
                            }
                        }
                    }
                    if (G == kUnitsPerWarp / 16 - 1) {
                        tc_fence_before();
                        mbar_arrive(tmem_free + 8 * pass);  // this half may be overwritten by the next tile's pass
                    }
                    __syncwarp();
                    // h' -> global, 64 contiguous bytes per row
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        if (tvalid[i])
                            *reinterpret_cast<float4 *>(hidden + trow[i] * kH + ub + 4 * tc4) =
                                *reinterpret_cast<const float4 *>(tile + (8 * i + tr) * kTileStride + 4 * tc4);
                }
            }
            // the warps of a row add their parts of fc2 (fixed order), the first one picks the action; the partial sums
            // travel through the sender's own tile (row r at tile + r * kTileStride)
            __syncwarp();
            if (cq > 0) {
#pragma unroll
                for (int a = 0; a < AP; a++) tile[lane * kTileStride + a] = qacc[a];
            }
            epi_sync();
            if (cq == 0) {
                float best = -INFINITY;
                int idx = 0;
#pragma unroll
                for (int a = 0; a < AP; a++) {
                    if (a < A) {
                        float qv = qacc[a];
#pragma unroll
                        for (int gI = 1; gI < kColGroups; gI++) qv += tile[gI * 4 * (32 * kTileStride) + lane * kTileStride + a];
                        qv += b2[a];
                        if (qv > best) { best = qv; idx = a; }  // first maximum, like np.argmax (misc.py:170)
                        if (q_out && valid) q_out[grow * A + a] = qv;
                    }
                }
                if (valid) actions[grow] = idx;
            }
            epi_sync();
        }
    } else if (warp < kStageBase) {
        reg_dec<40>();                                       // the whole warpgroup: issuer, loader, two idle warps
        if (warp == kMmaWarp) {
        // ------------------------------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc(kHalf);
            uint32_t q = 0;                                 // running slab counter
            for (int n = 0; n < my_tiles; n++) {
                const int b = n & 1;
                mbar_wait(act_full + 8 * b, (uint32_t)((n >> 1) & 1));
                tc_fence_after();
                const uint32_t xa = sbase + Smem2::act + b * Smem2::act_stride, ha = xa + kActBytes;
                for (int pass = 0; pass < 2; pass++) {
                    mbar_wait(tmem_free + 8 * pass, (uint32_t)((n & 1) ^ 1));
                    tc_fence_after();
                    for (int g = 0; g < 6; g++, q++) {
                        const uint32_t slot = q % ring;
                        mbar_wait(slab_full + 8 * slot, (q / ring) & 1);
                        tc_fence_after();
                        const uint32_t a_base = (g & 1) ? ha : xa;                          // even slabs multiply x, odd slabs h
                        const uint32_t d_col = 256u * pass + (g < 4 ? 64u * (g >> 1) : 64u * (g - 2));   // r, r, z, z, in, hn
                        const uint32_t acc0 = (g == 1 || g == 3) ? 1u : 0u;                 // the h side of r and z accumulates
                        for (int ks = 0; ks < kH / 16; ks++) {
                            const uint64_t ad = make_desc(a_base + ks * 2 * kActLBO, kActLBO, 128);
                            const uint64_t bd = make_desc(sbase + p.ring_off + slot * kHalfSlabBytes + ks * 2 * (kHalf / 8 * 128), kHalf / 8 * 128, 128);
                            umma(tmem + d_col, ad, bd, idesc, acc0 | (ks > 0));
                        }
                        tc_commit(slab_empty + 8 * slot);
                    }
                    tc_commit(tmem_full + 8 * pass);
                }
                tc_commit(act_free + 8 * b);                // both passes have read x and h of this buffer
            }
        }
        } else if (warp == kLoadWarp) {
        // ------------------------------------------------------------------------------------------ weight loader
        if (lane == 0) {
            const uint8_t *img0 = p.img + (size_t)(p.non_shared ? ((int)blockIdx.x % N) : 0) * p.set_bytes;
            mbar_expect_tx(head_full, (uint32_t)p.head_bytes);
            bulk_g2s(sbase + Smem2::head, img0, (uint32_t)p.head_bytes, head_full);
            uint32_t q = 0;
            for (int n = 0; n < my_tiles; n++) {
                const int t = (int)blockIdx.x + n * (int)gridDim.x;
                const uint8_t *img = p.img + (size_t)(p.non_shared ? (t % N) : 0) * p.set_bytes + p.head_bytes;
                for (int s = 0; s < kSlabsPerTile; s++, q++) {
                    const uint32_t slot = q % ring;
                    mbar_wait(slab_empty + 8 * slot, ((q / ring) & 1) ^ 1);
                    mbar_expect_tx(slab_full + 8 * slot, kHalfSlabBytes);
                    bulk_g2s(sbase + p.ring_off + slot * kHalfSlabBytes, img + (size_t)s * kHalfSlabBytes, kHalfSlabBytes, slab_full + 8 * slot);
                }
            }
        }
        }
    } else {
        // ------------------------------------------------------------------------------------------ staging + fc1
        reg_dec<88>();
        const int sw = warp - kStageBase;                    // this warp stages rows 16 sw .. 16 sw + 15 of every tile
        const int g = lane >> 2, tq = lane & 3;              // mma.sync fragment coordinates
        const int KS = w1_stride(Dp), nk = Dp >> 4;
        mbar_wait_sleep(head_full, 0);
        const __half *W1h = reinterpret_cast<const __half *>(headf);
        const float *b1 = headf + head_bias(Dp);
        __half *scr = reinterpret_cast<__half *>(const_cast<float *>(headf) + head_floats(Dp, A) + kEpiWarps * 32 * kTileStride) + sw * scratch_halves(Dp);
        for (int n = 0; n < my_tiles; n++) {
            const int t = (int)blockIdx.x + n * (int)gridDim.x;
            const int agent = t % N;
            const int b = n & 1;
            // lane r < 16 describes row 16 sw + r; the others mirror it
            const int64_t e = (int64_t)(t / N) * kRows + 16 * sw + (lane & 15);
            const bool valid = e < p.B;
            const int my_zero = (!valid || (fresh && fresh[e])) ? 1 : 0;
            const int64_t my_grow = (valid ? e : 0) * N + agent;
            // hidden state: one coalesced 512-byte row per load instruction, packed to FP16 as it arrives (this lane
            // keeps k = 4 lane .. 4 lane + 3 of each of the 16 rows)
            uint2 hp[16];
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const int64_t gr = __shfl_sync(0xffffffffu, my_grow, r);
                const int zr = __shfl_sync(0xffffffffu, my_zero, r);
                float4 v = *reinterpret_cast<const float4 *>(hidden + gr * kH + 4 * lane);
                if (zr) v = make_float4(0.f, 0.f, 0.f, 0.f);
                hp[r] = make_uint2(h2(v.x, v.y), h2(v.z, v.w));
            }
            // observation (+ one-hot agent id, misc.py:161-162) -> FP16 scratch [16][KS]; lane = input column.  All 16
            // row loads are issued before the first use (branch-free: a branch per row made the compiler wait for
            // each load in turn -- 12 us per tile in the first version of this role)
            __syncwarp();
#pragma unroll 1
            for (int k0 = 0; k0 < Dp; k0 += 32) {
                const int k = k0 + lane;
                const bool in_obs = k < D;
                const float idv = (k >= D && k < Din && p.obs_agent_id && k - D == agent) ? 1.f : 0.f;
                const int kc = in_obs ? k : 0;
                float ov[16];
#pragma unroll
                for (int r = 0; r < 16; r++) {
                    const int64_t gr = __shfl_sync(0xffffffffu, my_grow, r);
                    ov[r] = obs[gr * D + kc];
                }
#pragma unroll
                for (int r = 0; r < 16; r++) {
                    const int zr = __shfl_sync(0xffffffffu, my_zero, r);
                    const float v = in_obs ? (zr ? 0.f : ov[r]) : idv;
                    if (k < Dp) scr[r * KS + k] = __float2half_rn(v);
                }
            }
            __syncwarp();
            uint32_t af[4][4];                               // A fragments of the 16 x dp observation block
#pragma unroll
            for (int ks = 0; ks < 4; ks++)
                if (ks < nk) {
                    af[ks][0] = *reinterpret_cast<const uint32_t *>(scr + g * KS + 16 * ks + 2 * tq);
                    af[ks][1] = *reinterpret_cast<const uint32_t *>(scr + (g + 8) * KS + 16 * ks + 2 * tq);
                    af[ks][2] = *reinterpret_cast<const uint32_t *>(scr + g * KS + 16 * ks + 2 * tq + 8);
                    af[ks][3] = *reinterpret_cast<const uint32_t *>(scr + (g + 8) * KS + 16 * ks + 2 * tq + 8);
                }
            mbar_wait_sleep(act_free + 8 * b, (uint32_t)(((n >> 1) & 1) ^ 1));
            uint8_t *xa = sm + Smem2::act + b * Smem2::act_stride, *ha = xa + kActBytes;
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const int rr = 16 * sw + r;
                *reinterpret_cast<uint2 *>(ha + (lane >> 1) * kActLBO + (rr >> 3) * 128 + (rr & 7) * 16 + (lane & 1) * 8) = hp[r];
            }
            // x = relu(fc1(obs)) (rnn_agent.py:22): 16 column tiles of 8 units; c0 c1 = (row g, units 2 tq, 2 tq + 1),
            // c2 c3 = (row g + 8, same units)
            const uint32_t r_lo = (uint32_t)(((16 * sw + g) >> 3) * 128 + ((16 * sw + g) & 7) * 16 + 4 * tq);
            const uint32_t r_hi = (uint32_t)(((16 * sw + g + 8) >> 3) * 128 + ((16 * sw + g + 8) & 7) * 16 + 4 * tq);
#pragma unroll 4
            for (int nt = 0; nt < kH / 8; nt++) {
                const float bx = b1[8 * nt + 2 * tq], by = b1[8 * nt + 2 * tq + 1];
                float c[4] = {bx, by, bx, by};
                const __half *wrow = W1h + (8 * nt + g) * KS + 2 * tq;
#pragma unroll
                for (int ks = 0; ks < 4; ks++)
                    if (ks < nk)
                        mma_m16n8k16(c, af[ks], *reinterpret_cast<const uint32_t *>(wrow + 16 * ks),
                                     *reinterpret_cast<const uint32_t *>(wrow + 16 * ks + 8));
                *reinterpret_cast<uint32_t *>(xa + nt * kActLBO + r_lo) = h2(fmaxf(c[0], 0.f), fmaxf(c[1], 0.f));
                *reinterpret_cast<uint32_t *>(xa + nt * kActLBO + r_hi) = h2(fmaxf(c[2], 0.f), fmaxf(c[3], 0.f));
            }
            fence_async_smem();                             // generic-proxy stores -> visible to the tensor core's async proxy
            mbar_arrive(act_full + 8 * b);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

}  // namespace tc2
}  // namespace mrb
