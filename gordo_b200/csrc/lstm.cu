// LSTM autoencoder / forecast: KerasLSTMBaseEstimator.predict / .fit (gordo/machine/model/models.py:557-660)
// over the [3P] Keras LSTM cell the factories of lstm_autoencoder.py:77-102 build
// (gate order i,f,c,o; z = x.W + h.U + b; i,f,o = sigmoid; c~ = act(z_c); c = f*c + i*c~; h = o*act(c)).
//
// Windows are never materialised (models.py:713-793 builds [B,L,T] copies on the host): sequence b of
// a launch is window `seq_base + b` of its Machine, i.e. rows [start, start+L) of the Machine's
// sample matrix, scaled on the fly (MinMaxScaler.transform fused into the layer-0 operand load).
//
// Inference (this file: exact fp32; lstm_tc.cu: the tcgen05 pipeline):
//   lstm_step_fwd      one (layer, t): tiled GEMM [seq x (in+u)] x [(in+u) x 4u] with the gate
//                      non-linearities, cell update and h = o*act(c) fused in the epilogue
//   lstm_dense_out     yhat = out_act(h_last . Wd + bd)
// Training (KerasLSTMBaseEstimator.fit, J jobs per launch), split by what is sequential:
//   lstm_bgemm_tc[v]   everything that is not the recurrence -- x_t.W + b for all t, dz.W^T for all t,
//                      the weight gradients over (t, seq) -- as batched GEMMs on tcgen05 (kind::tf32,
//                      3xTF32 split: fp32-accurate); lstm_bgemm (CUDA cores) for small launches
//   lstm_rec_fwd/bwd   the recurrence of a whole layer in one launch: a thread-block cluster per job,
//                      U slices resident in shared memory, h_t / partial dh_rec exchanged through DSMEM
//   lstm_step_fwd / lstm_bwd_gates / lstm_nt   the per-time-step launch path, kept for layers wider than
//                      the cluster kernels take and as their parity reference (GB200_LSTM_REC=0)
//   Keras-form Adam, loss history on the device.
#include "common.cuh"
#include "ptx.cuh"
#include <vector>
#include <stdlib.h>

namespace {

constexpr int ST_SEQ = 32;      // sequences per CTA tile
constexpr int ST_UNITS = 16;    // units per CTA tile (x4 gates = 64 GEMM columns)
constexpr int ST_K = 32;        // K slab
constexpr int ST_THREADS = 256;

struct LayerDims { int in, u; int64_t w_off, u_off, b_off; };

struct LstmPlan {
    int n_layers, T_in, T_out, L, lookahead, out_act;
    LayerDims ld[GB200_MAX_LAYERS];
    int acts[GB200_MAX_LAYERS];
    int64_t dense_w_off, dense_b_off, n_params;
    int sum_u, max_u, max_in;
};

LstmPlan make_plan(const gb200_lstm_arch* a) {
    LstmPlan p{};
    p.n_layers = a->n_layers; p.T_in = a->n_features; p.T_out = a->n_features_out;
    p.L = a->lookback_window; p.lookahead = a->lookahead; p.out_act = a->out_act;
    int64_t off = 0; int in = a->n_features;
    for (int l = 0; l < a->n_layers; ++l) {
        const int u = a->units[l];
        p.ld[l].in = in; p.ld[l].u = u;
        p.ld[l].w_off = off; off += (int64_t)in * 4 * u;
        p.ld[l].u_off = off; off += (int64_t)u * 4 * u;
        p.ld[l].b_off = off; off += 4 * u;
        p.acts[l] = a->acts[l];
        p.sum_u += u; if (u > p.max_u) p.max_u = u; if (in > p.max_in) p.max_in = in;
        in = u;
    }
    p.dense_w_off = off; off += (int64_t)in * a->n_features_out;
    p.dense_b_off = off; off += a->n_features_out;
    p.n_params = off;
    return p;
}

__device__ __forceinline__ float sigmoidf_(float z) { return 1.0f / (1.0f + expf(-z)); }

// A group = one Machine (predict) or one fit job (training).  nb = sequences of the group in this launch.
struct GroupCtx {
    const int64_t* rows_lo;   // [G] first sample row of the group
    const int32_t* n_win;     // [G] windows of the group
    int seq_base;             // first window of this launch (same for all groups: lock-step)
    int cap;                  // max sequences per group in this launch
};
__device__ __forceinline__ int group_nb(const GroupCtx& g, int grp) {
    const int n = g.n_win[grp] - g.seq_base;
    return n < 0 ? 0 : (n > g.cap ? g.cap : n);
}

struct StepArgs {
    GroupCtx g;
    int in, u, act, t, layer;
    const float* params; int64_t n_params, w_off, u_off, b_off;     // per group: params + grp*n_params
    // layer input: layer 0 reads the sample matrix (scaled), others a [seq][in] slab
    const float* x; int T_in; const float* in_scale; const float* in_min;          // layer 0
    const float* xin; int64_t xin_seq_stride, xin_grp_stride;                      // layer > 0
    const float* h_prev; int64_t hprev_seq_stride, hprev_grp_stride;               // nullptr at t == 0
    float* h_out; int64_t hout_seq_stride, hout_grp_stride;
    const float* c_prev; int64_t cprev_seq_stride, cprev_grp_stride;               // nullptr at t == 0
    float* c_out; int64_t cout_seq_stride, cout_grp_stride;
    // optional caches for BPTT ([seq] x stride): gates i,f,g,o (4u) and act(c) (u)
    float* gates; int64_t gates_seq_stride, gates_grp_stride;
    float* actc; int64_t actc_seq_stride, actc_grp_stride;
    // training: `gates` already holds x_t.W + b for this (layer, t) (batched over all t by
    // lstm_bgemm_kernel); only the recurrent product h_{t-1}.U is left for this kernel
    int pre;
};

__global__ void __launch_bounds__(ST_THREADS)
lstm_step_fwd_kernel(const __grid_constant__ StepArgs a) {
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    const int s0 = blockIdx.x * ST_SEQ;
    if (s0 >= nb) return;
    const int u0 = blockIdx.y * ST_UNITS;
    const int u = a.u, in = a.pre ? 0 : a.in, K = (a.pre && !a.h_prev) ? 0 : in + u;
    const float* P = a.params + (size_t)grp * a.n_params;
    const float* W = P + a.w_off; const float* U = P + a.u_off; const float* bias = P + a.b_off;

    __shared__ float As[ST_SEQ][ST_K + 1];
    __shared__ __align__(16) float Ws[ST_K][ST_UNITS * 4];            // [k][unit][gate]

    const int tid = threadIdx.x;
    const int s_l = tid >> 3;                // sequence within tile (0..31)
    const int uj = (tid & 7) * 2;            // two units per thread
    float acc[2][4];
    #pragma unroll
    for (int q = 0; q < 2; ++q)
        #pragma unroll
        for (int gte = 0; gte < 4; ++gte) {
            const int uu = u0 + uj + q;
            float b0 = 0.0f;
            if (uu < u) {
                if (!a.pre) b0 = bias[gte * u + uu];
                else if (s0 + s_l < nb)
                    b0 = a.gates[(size_t)grp * a.gates_grp_stride + (size_t)(s0 + s_l) * a.gates_seq_stride + gte * u + uu];
            }
            acc[q][gte] = b0;
        }
    const int64_t row0 = a.layer == 0 ? a.g.rows_lo[grp] + a.g.seq_base + a.t : 0;
    const float* sc = (a.layer == 0 && a.in_scale) ? a.in_scale + (size_t)grp * a.T_in : nullptr;
    const float* mn = (a.layer == 0 && a.in_min) ? a.in_min + (size_t)grp * a.T_in : nullptr;

    for (int k0 = 0; k0 < K; k0 += ST_K) {
        // ---- A slab: [seq][k] = concat(x_t, h_{t-1})
        for (int i = tid; i < ST_SEQ * ST_K; i += ST_THREADS) {
            const int ss = i / ST_K, kk = i - ss * ST_K;
            const int s = s0 + ss, k = k0 + kk;
            float v = 0.0f;
            if (s < nb && k < K) {
                if (k < in) {
                    if (a.layer == 0) {
                        v = a.x[(row0 + s) * a.T_in + k];
                        if (sc) v = fmaf(v, sc[k], mn[k]);
                    } else {
                        v = a.xin[(size_t)grp * a.xin_grp_stride + (size_t)s * a.xin_seq_stride + k];
                    }
                } else if (a.h_prev) {
                    v = a.h_prev[(size_t)grp * a.hprev_grp_stride + (size_t)s * a.hprev_seq_stride + (k - in)];
                }
            }
            As[ss][kk] = v;
        }
        // ---- weight slab: rows k of [W;U], the 4 gate columns of 16 units
        for (int i = tid; i < ST_K * ST_UNITS * 4; i += ST_THREADS) {
            const int kk = i / (ST_UNITS * 4), r = i - kk * (ST_UNITS * 4);
            const int gte = r / ST_UNITS, ul = r - gte * ST_UNITS;          // consecutive threads: consecutive units
            const int k = k0 + kk, uu = u0 + ul;
            float v = 0.0f;
            if (k < K && uu < u) v = (k < in) ? W[(size_t)k * 4 * u + gte * u + uu] : U[(size_t)(k - in) * 4 * u + gte * u + uu];
            Ws[kk][ul * 4 + gte] = v;
        }
        __syncthreads();
        #pragma unroll 8
        for (int kk = 0; kk < ST_K; ++kk) {
            const float av = As[s_l][kk];
            const float4 w0 = *reinterpret_cast<const float4*>(&Ws[kk][uj * 4]);
            const float4 w1 = *reinterpret_cast<const float4*>(&Ws[kk][uj * 4 + 4]);
            acc[0][0] = fmaf(av, w0.x, acc[0][0]); acc[0][1] = fmaf(av, w0.y, acc[0][1]);
            acc[0][2] = fmaf(av, w0.z, acc[0][2]); acc[0][3] = fmaf(av, w0.w, acc[0][3]);
            acc[1][0] = fmaf(av, w1.x, acc[1][0]); acc[1][1] = fmaf(av, w1.y, acc[1][1]);
            acc[1][2] = fmaf(av, w1.z, acc[1][2]); acc[1][3] = fmaf(av, w1.w, acc[1][3]);
        }
        __syncthreads();
    }
    const int s = s0 + s_l;
    if (s >= nb) return;
    #pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int uu = u0 + uj + q;
        if (uu >= u) continue;
        const float ig = sigmoidf_(acc[q][0]), fg = sigmoidf_(acc[q][1]);
        const float gg = gb_act(a.act, acc[q][2]), og = sigmoidf_(acc[q][3]);
        const float cp = a.c_prev ? a.c_prev[(size_t)grp * a.cprev_grp_stride + (size_t)s * a.cprev_seq_stride + uu] : 0.0f;
        const float cn = fmaf(fg, cp, ig * gg);
        const float ac = gb_act(a.act, cn);
        a.c_out[(size_t)grp * a.cout_grp_stride + (size_t)s * a.cout_seq_stride + uu] = cn;
        a.h_out[(size_t)grp * a.hout_grp_stride + (size_t)s * a.hout_seq_stride + uu] = og * ac;
        if (a.gates) {
            float* gp = a.gates + (size_t)grp * a.gates_grp_stride + (size_t)s * a.gates_seq_stride;
            gp[uu] = ig; gp[u + uu] = fg; gp[2 * u + uu] = gg; gp[3 * u + uu] = og;
            a.actc[(size_t)grp * a.actc_grp_stride + (size_t)s * a.actc_seq_stride + uu] = ac;
        }
    }
}

struct DenseArgs {
    GroupCtx g;
    int u, T_out, act;
    const float* params; int64_t n_params, w_off, b_off;
    const float* h; int64_t h_seq_stride, h_grp_stride;
    float* out; const int64_t* out_row_off;      // predict: rows out_row_off[grp] + seq_base + s
    float* out_local; int64_t ol_seq_stride, ol_grp_stride;      // training: [grp][seq][T_out]
};

__global__ void lstm_dense_out_kernel(const __grid_constant__ DenseArgs a) {
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    const float* P = a.params + (size_t)grp * a.n_params;
    const float* Wd = P + a.w_off; const float* bd = P + a.b_off;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb * a.T_out; i += gridDim.x * blockDim.x) {
        const int s = i / a.T_out, n = i - s * a.T_out;
        const float* h = a.h + (size_t)grp * a.h_grp_stride + (size_t)s * a.h_seq_stride;
        float acc = bd[n];
        for (int k = 0; k < a.u; ++k) acc = fmaf(h[k], Wd[(size_t)k * a.T_out + n], acc);
        const float y = gb_act(a.act, acc);
        if (a.out) a.out[(a.out_row_off[grp] + a.g.seq_base + s) * a.T_out + n] = y;
        if (a.out_local) a.out_local[(size_t)grp * a.ol_grp_stride + (size_t)s * a.ol_seq_stride + n] = y;
    }
}

// ------------------------------------------------------------------------------------------ training
struct LossArgs {
    GroupCtx g;
    int u, T_out, act, L, lookahead;
    const float* params; int64_t n_params, w_off, b_off;
    const float* y; const float* yhat; int64_t yh_seq_stride, yh_grp_stride;
    const float* h_last; int64_t h_seq_stride, h_grp_stride;
    float* dzd; int64_t dzd_grp_stride;              // [grp][seq][T_out]  dLoss/dz_dense
    float* loss_sum;                                 // [grp] sum of squared errors of this step (atomic)
};

// dzd = 2/(nb*T_out) * (yhat - y) * out_act'(yhat); accumulates the squared error
__global__ void lstm_loss_kernel(const __grid_constant__ LossArgs a) {
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    if (nb == 0) return;
    const float inv = 2.0f / (float)(nb * a.T_out);
    float sq = 0.0f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb * a.T_out; i += gridDim.x * blockDim.x) {
        const int s = i / a.T_out, n = i - s * a.T_out;
        const float yh = a.yhat[(size_t)grp * a.yh_grp_stride + (size_t)s * a.yh_seq_stride + n];
        // target row of window (seq_base + s): start + L - 1 + lookahead (models.py:713-793)
        const int64_t row = a.g.rows_lo[grp] + a.g.seq_base + s + a.L - 1 + a.lookahead;
        const float d = yh - a.y[row * a.T_out + n];
        sq = fmaf(d, d, sq);
        float gr;
        switch (a.act) {
            case GB200_ACT_TANH: gr = 1.0f - yh * yh; break;
            case GB200_ACT_RELU: gr = yh > 0.0f ? 1.0f : 0.0f; break;
            case GB200_ACT_SIGMOID: gr = yh * (1.0f - yh); break;
            case GB200_ACT_ELU: gr = yh > 0.0f ? 1.0f : yh + 1.0f; break;
            case GB200_ACT_SOFTPLUS: gr = 1.0f - expf(-yh); break;
            default: gr = 1.0f;
        }
        a.dzd[(size_t)grp * a.dzd_grp_stride + (size_t)s * a.T_out + n] = inv * d * gr;
    }
    #pragma unroll
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(a.loss_sum + grp, sq);
}

// generic small reductions used by the backward pass -------------------------------------------------
// out[grp][s][k] (+)= sum_n A[grp][s][n] * B[grp][k][n]   (rows of B contiguous: "NT")
struct NTArgs {
    GroupCtx g;
    int N, Kout;
    const float* A; int64_t a_seq_stride, a_grp_stride;
    const float* B; int64_t b_row_stride, b_grp_stride;      // B row k at B + k*b_row_stride
    float* out; int64_t o_seq_stride, o_grp_stride;
    int accumulate;
};
__global__ void lstm_nt_kernel(const __grid_constant__ NTArgs a) {
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < nb * a.Kout; i += nwarps) {
        const int s = i / a.Kout, k = i - s * a.Kout;
        const float* ap = a.A + (size_t)grp * a.a_grp_stride + (size_t)s * a.a_seq_stride;
        const float* bp = a.B + (size_t)grp * a.b_grp_stride + (size_t)k * a.b_row_stride;
        float acc = 0.0f;
        for (int n = lane; n < a.N; n += 32) acc = fmaf(ap[n], bp[n], acc);
        #pragma unroll
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            float* op = a.out + (size_t)grp * a.o_grp_stride + (size_t)s * a.o_seq_stride + k;
            *op = a.accumulate ? *op + acc : acc;
        }
    }
}

struct BwdGateArgs {
    GroupCtx g;
    int u, act, t, L;
    const float* dh_above; int64_t da_seq_stride, da_grp_stride;   // dLoss/dh_t from the layer above (may be null)
    const float* dh_rec; int64_t dr_seq_stride, dr_grp_stride;     // from t+1 (null at t == L-1)
    float* dc; int64_t dc_seq_stride, dc_grp_stride;               // running dLoss/dc (in/out)
    const float* gates; int64_t g_seq_stride, g_grp_stride;        // i,f,g,o at t
    const float* actc; int64_t ac_seq_stride, ac_grp_stride;       // act(c_t)
    const float* c_t; int64_t ct_seq_stride, ct_grp_stride;
    const float* c_prev; int64_t cp_seq_stride, cp_grp_stride;     // null at t == 0
    float* dz; int64_t dz_seq_stride, dz_grp_stride;               // [seq][4u] out
};
__device__ __forceinline__ float act_grad_h(int code, float h) {
    switch (code) {
        case GB200_ACT_TANH: return 1.0f - h * h;
        case GB200_ACT_RELU: return h > 0.0f ? 1.0f : 0.0f;
        case GB200_ACT_SIGMOID: return h * (1.0f - h);
        case GB200_ACT_ELU: return h > 0.0f ? 1.0f : h + 1.0f;
        case GB200_ACT_SOFTPLUS: return 1.0f - expf(-h);
        default: return 1.0f;
    }
}
__global__ void lstm_bwd_gates_kernel(const __grid_constant__ BwdGateArgs a) {
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    const int u = a.u;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb * u; i += gridDim.x * blockDim.x) {
        const int s = i / u, j = i - s * u;
        float dh = 0.0f;
        if (a.dh_above) dh += a.dh_above[(size_t)grp * a.da_grp_stride + (size_t)s * a.da_seq_stride + j];
        if (a.dh_rec) dh += a.dh_rec[(size_t)grp * a.dr_grp_stride + (size_t)s * a.dr_seq_stride + j];
        const float* gp = a.gates + (size_t)grp * a.g_grp_stride + (size_t)s * a.g_seq_stride;
        const float ig = gp[j], fg = gp[u + j], gg = gp[2 * u + j], og = gp[3 * u + j];
        const float ac = a.actc[(size_t)grp * a.ac_grp_stride + (size_t)s * a.ac_seq_stride + j];
        const float cp = a.c_prev ? a.c_prev[(size_t)grp * a.cp_grp_stride + (size_t)s * a.cp_seq_stride + j] : 0.0f;
        float* dcp = a.dc + (size_t)grp * a.dc_grp_stride + (size_t)s * a.dc_seq_stride + j;
        const float dc_in = (a.t == a.L - 1) ? 0.0f : *dcp;
        const float d_o = dh * ac;
        const float dc = dc_in + dh * og * act_grad_h(a.act, ac);
        *dcp = dc * fg;
        float* dz = a.dz + (size_t)grp * a.dz_grp_stride + (size_t)s * a.dz_seq_stride;
        dz[j] = dc * gg * ig * (1.0f - ig);
        dz[u + j] = dc * cp * fg * (1.0f - fg);
        dz[2 * u + j] = dc * ig * act_grad_h(a.act, gg);
        dz[3 * u + j] = d_o * og * (1.0f - og);
    }
}

// g[grp][k][n] = sum over (t, s) of A_t[grp][s][k] * dZ_t[grp][s][n]; A is either the layer input
// sequence or the h_{t-1} sequence (zero at t == 0).  One thread per (k, n).
struct WgradArgs {
    GroupCtx g;
    int Kdim, N, L, layer, T_in, shift;      // shift = 1: A_t = seq[t-1] (recurrent weights)
    const float* x; const float* in_scale; const float* in_min;        // layer 0 input from the sample matrix
    const float* aseq; int64_t a_t_stride, a_seq_stride, a_grp_stride; // otherwise [t][seq][Kdim]
    const float* dz; int64_t dz_t_stride, dz_seq_stride, dz_grp_stride;
    float* grad; int64_t grad_grp_stride; int64_t grad_off;            // [Kdim][N] at grad + grad_off
    float* gbias; int64_t gbias_off;                                   // [N] (only when shift == 0 pass)
};
__global__ void lstm_wgrad_kernel(const __grid_constant__ WgradArgs a) {
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    const int total = a.Kdim * a.N + (a.gbias ? a.N : 0);
    const float* sc = (a.layer == 0 && a.x && a.in_scale) ? a.in_scale + (size_t)grp * a.T_in : nullptr;
    const float* mn = sc ? a.in_min + (size_t)grp * a.T_in : nullptr;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        float acc = 0.0f;
        if (i < a.Kdim * a.N) {
            const int k = i / a.N, n = i - k * a.N;
            for (int t = a.shift; t < a.L; ++t) {
                const float* dzp = a.dz + (size_t)grp * a.dz_grp_stride + (size_t)t * a.dz_t_stride + n;
                for (int s = 0; s < nb; ++s) {
                    float av;
                    if (a.x) {
                        av = a.x[(a.g.rows_lo[grp] + a.g.seq_base + s + t) * a.T_in + k];
                        if (sc) av = fmaf(av, sc[k], mn[k]);
                    } else {
                        av = a.aseq[(size_t)grp * a.a_grp_stride + (size_t)(t - a.shift) * a.a_t_stride + (size_t)s * a.a_seq_stride + k];
                    }
                    acc = fmaf(av, dzp[(size_t)s * a.dz_seq_stride], acc);
                }
            }
            a.grad[(size_t)grp * a.grad_grp_stride + a.grad_off + i] = acc;
        } else {
            const int n = i - a.Kdim * a.N;
            for (int t = 0; t < a.L; ++t)
                for (int s = 0; s < nb; ++s)
                    acc += a.dz[(size_t)grp * a.dz_grp_stride + (size_t)t * a.dz_t_stride + (size_t)s * a.dz_seq_stride + n];
            a.gbias[(size_t)grp * a.grad_grp_stride + a.gbias_off + n] = acc;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Batched fp32 GEMM over the (t, seq) composite dimension of a training step.  Sequence buffers are
// dense [t][seq][width] (row r = t*cap + seq), so everything that is not the recurrence itself is
// one GEMM per layer instead of one launch per time step:
//   comp == 0:  C[r][j]  = sum_k A(r,k) * B(k,j) (+ bias[j])      rows r composite, masked by seq < nb
//               (x.W for all t: NN;  dz.W^T -> dLoss/dx for all t: NT)
//   comp == 1:  C[i][j]  = sum_r A(r,i) * B(r,j)                   K composite: the weight gradients
// 64x64x16 tiles, 256 threads, 4x4 register micro-tile; operands may be "k-contiguous" (element (m,k)
// at P[m*ld + k]) or "m-contiguous" (P[k*ld + m]); one grid.z slice per fit job.
struct GemmArgs {
    GroupCtx g;
    int seq_dim;             // sequences per time step in the buffers (the fit's batch size)
    int M, N, K, comp;
    const float* A; int64_t a_grp; int lda, a_kcontig;
    const float* B; int64_t b_grp; int ldb, b_kcontig;
    float* C; int64_t c_grp; int ldc;
    const float* bias; int64_t bias_grp;
};
constexpr int GK = 16;

template <int BM, int BN>
__global__ void __launch_bounds__(256)
lstm_bgemm_kernel(const __grid_constant__ GemmArgs a) {
    constexpr int RM = BM / 64, RN = BN / 64;        // 4-wide chunks of the micro-tile (rows / cols)
    constexpr int EA = BM * GK / 256, EB = BN * GK / 256;
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    if (nb == 0) return;
    const int sd = a.seq_dim;
    const bool full = nb == sd;                      // no masking needed (every step but a job's last)
    const float* __restrict__ A = a.A + (size_t)grp * a.a_grp;
    const float* __restrict__ B = a.B + (size_t)grp * a.b_grp;
    float* C = a.C + (size_t)grp * a.c_grp;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    __shared__ __align__(16) float As[GK][BM + 4];
    __shared__ __align__(16) float Bs[GK][BN + 4];
    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;          // 16 x 16 threads
    float acc[RM * 4][RN * 4] = {};
    float ra[EA], rb[EB];
    // global -> registers for the K slab at k0: consecutive threads walk the operand's contiguous dimension
    auto fetch = [&](int k0) {
        #pragma unroll
        for (int e = 0; e < EA; ++e) {
            const int i = tid + e * 256;
            int mm, kk;
            if (a.a_kcontig) { kk = i & (GK - 1); mm = i / GK; } else { mm = i & (BM - 1); kk = i / BM; }
            const int m = m0 + mm, k = k0 + kk;
            float v = 0.0f;
            if (m < a.M && k < a.K && (full || ((a.comp ? k : m) % sd) < nb))
                v = a.a_kcontig ? A[(size_t)m * a.lda + k] : A[(size_t)k * a.lda + m];
            ra[e] = v;
        }
        #pragma unroll
        for (int e = 0; e < EB; ++e) {
            const int i = tid + e * 256;
            int nn, kk;
            if (a.b_kcontig) { kk = i & (GK - 1); nn = i / GK; } else { nn = i & (BN - 1); kk = i / BN; }
            const int n = n0 + nn, k = k0 + kk;
            float v = 0.0f;
            if (n < a.N && k < a.K && (full || !a.comp || (k % sd) < nb))
                v = a.b_kcontig ? B[(size_t)n * a.ldb + k] : B[(size_t)k * a.ldb + n];
            rb[e] = v;
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < a.K; k0 += GK) {
        #pragma unroll
        for (int e = 0; e < EA; ++e) {
            const int i = tid + e * 256;
            if (a.a_kcontig) As[i & (GK - 1)][i / GK] = ra[e]; else As[i / BM][i & (BM - 1)] = ra[e];
        }
        #pragma unroll
        for (int e = 0; e < EB; ++e) {
            const int i = tid + e * 256;
            if (a.b_kcontig) Bs[i & (GK - 1)][i / GK] = rb[e]; else Bs[i / BN][i & (BN - 1)] = rb[e];
        }
        __syncthreads();
        if (k0 + GK < a.K) fetch(k0 + GK);          // next slab's loads fly while this one is multiplied
        #pragma unroll
        for (int kk = 0; kk < GK; ++kk) {
            float ar[RM * 4], br[RN * 4];
            #pragma unroll
            for (int c = 0; c < RM; ++c) {
                const float4 t = *reinterpret_cast<const float4*>(&As[kk][c * 64 + ty * 4]);
                ar[c * 4] = t.x; ar[c * 4 + 1] = t.y; ar[c * 4 + 2] = t.z; ar[c * 4 + 3] = t.w;
            }
            #pragma unroll
            for (int c = 0; c < RN; ++c) {
                const float4 t = *reinterpret_cast<const float4*>(&Bs[kk][c * 64 + tx * 4]);
                br[c * 4] = t.x; br[c * 4 + 1] = t.y; br[c * 4 + 2] = t.z; br[c * 4 + 3] = t.w;
            }
            #pragma unroll
            for (int i = 0; i < RM * 4; ++i)
                #pragma unroll
                for (int j = 0; j < RN * 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
        }
        __syncthreads();
    }
    const float* bias = a.bias ? a.bias + (size_t)grp * a.bias_grp : nullptr;
    #pragma unroll
    for (int i = 0; i < RM * 4; ++i) {
        const int m = m0 + (i >> 2) * 64 + ty * 4 + (i & 3);
        if (m >= a.M || (!a.comp && !full && (m % sd) >= nb)) continue;
        #pragma unroll
        for (int j = 0; j < RN * 4; ++j) {
            const int n = n0 + (j >> 2) * 64 + tx * 4 + (j & 3);
            if (n < a.N) C[(size_t)m * a.ldc + n] = acc[i][j] + (bias ? bias[n] : 0.0f);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// The same batched GEMM on the tensor cores, fp32-accurate: every fp32 operand element x is split
// into hi = tf32(x) and lo = tf32(x - hi) while it is staged into shared memory (tcgen05 canonical
// K-major, no swizzle: [K/4][rows/8][8 rows][4 elements]) and the product is accumulated in tensor
// memory as A_hi.B_hi + A_hi.B_lo + A_lo.B_hi (tcgen05.mma kind::tf32, fp32 accumulate; the dropped
// lo.lo term is below 2^-21 relative).  One CTA = one 128 x 128 tile of C; two shared-memory stages
// of K = 32: the threads stage slab i+1 (global loads issued one slab ahead, into registers) while
// the MMAs of slab i run; a stage is reused when the tcgen05.commit of the MMAs that read it lands.
constexpr int TK = 16;                       // K per stage
constexpr int T_LBO = 2048 + 16;             // byte stride between K chunks of 4 (padded: bank spread)
constexpr int T_IMG = (TK / 4) * T_LBO;      // one operand image: 128 rows x TK
constexpr int T_STAGE = 4 * T_IMG;           // A_hi, A_lo, B_hi, B_lo
constexpr int TC_THREADS = 256;
constexpr int T_ELEMS = 128 * TK / TC_THREADS;   // elements per thread per operand per slab

// AK / BK: operand is k-contiguous (element (row, k) at P[row*ld + k]) or row-contiguous (P[k*ld + row]);
// COMP: the composite (t, seq) dimension is K (weight gradients) instead of the rows of A and C.
// Template parameters, so that the per-element index math of the staging loops folds to constants.
template <bool AK, bool BK, bool COMP>
__global__ void __launch_bounds__(TC_THREADS, 2)
lstm_bgemm_tc_kernel(const __grid_constant__ GemmArgs a) {
    using namespace gbptx;
    extern __shared__ __align__(128) uint8_t tsm[];
    __shared__ __align__(8) uint64_t done[2];
    __shared__ uint32_t s_tmem;
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    if (nb == 0) return;
    const int sd = a.seq_dim;
    const bool full = nb == sd;
    const float* __restrict__ A = a.A + (size_t)grp * a.a_grp;
    const float* __restrict__ B = a.B + (size_t)grp * a.b_grp;
    float* C = a.C + (size_t)grp * a.c_grp;
    const int m0 = blockIdx.y * 128, n0 = blockIdx.x * 128;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        mbar_init(&done[0], 1); mbar_init(&done[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(&s_tmem, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;

    // element i = tid + e * TC_THREADS of an operand: (row, kk) inside the 128 x TK slab, fixed for the K loop
    //   k-contiguous  : kk = i % TK, row = i / TK               (a warp reads 2 rows x 64 B)
    //   row-contiguous: 8 rows x 4 k per warp: row = 8 * ((i >> 5) & 15) + (i & 7), kk = 4 * (i >> 9) + ((i >> 3) & 3)
    //                   -- 32-byte global segments, and the 32 lanes of a shared store hit 32 different banks
    auto row_of = [&](bool kc, int e) { const int i = tid + e * TC_THREADS; return kc ? i / TK : 8 * ((i >> 5) & 15) + (i & 7); };
    auto kk_of = [&](bool kc, int e) { const int i = tid + e * TC_THREADS; return kc ? (i & (TK - 1)) : 4 * (i >> 9) + ((i >> 3) & 3); };
    float ra[T_ELEMS], rb[T_ELEMS];
    auto fetch = [&](int k0) {
        #pragma unroll
        for (int e = 0; e < T_ELEMS; ++e) {
            const int m = m0 + row_of(AK, e), k = k0 + kk_of(AK, e);
            float v = 0.0f;
            if (m < a.M && k < a.K && (full || ((COMP ? k : m) % sd) < nb))
                v = AK ? A[(size_t)m * a.lda + k] : A[(size_t)k * a.lda + m];
            ra[e] = v;
        }
        #pragma unroll
        for (int e = 0; e < T_ELEMS; ++e) {
            const int n = n0 + row_of(BK, e), k = k0 + kk_of(BK, e);
            float v = 0.0f;
            if (n < a.N && k < a.K && (full || !COMP || (k % sd) < nb))
                v = BK ? B[(size_t)n * a.ldb + k] : B[(size_t)k * a.ldb + n];
            rb[e] = v;
        }
    };
    auto put = [&](uint8_t* hi_img, uint8_t* lo_img, int row, int kk, float v) {
        const uint32_t off = (uint32_t)(kk >> 2) * T_LBO + (uint32_t)(row >> 3) * 128 + (uint32_t)(row & 7) * 16 + (uint32_t)(kk & 3) * 4;
        const uint32_t hi = f32_to_tf32(v);
        const uint32_t lo = f32_to_tf32(v - __uint_as_float(hi));
        *reinterpret_cast<uint32_t*>(hi_img + off) = hi;
        *reinterpret_cast<uint32_t*>(lo_img + off) = lo;
    };
    const uint32_t idesc = make_idesc_tf32(128, 128);
    const int nit = (a.K + TK - 1) / TK;
    fetch(0);
    for (int it = 0; it < nit; ++it) {
        const int s = it & 1;
        uint8_t* st = tsm + (size_t)s * T_STAGE;
        if (it >= 2) mbar_wait(&done[s], (uint32_t)((it >> 1) - 1) & 1u);      // the MMAs that read this stage are done
        #pragma unroll
        for (int e = 0; e < T_ELEMS; ++e) put(st, st + T_IMG, row_of(AK, e), kk_of(AK, e), ra[e]);
        #pragma unroll
        for (int e = 0; e < T_ELEMS; ++e) put(st + 2 * T_IMG, st + 3 * T_IMG, row_of(BK, e), kk_of(BK, e), rb[e]);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (it + 1 < nit) fetch((it + 1) * TK);        // next slab's global loads fly under the MMAs
        if (tid == 0) {
            tc_fence_after();
            const uint32_t ah = smem_u32(st), al = ah + T_IMG, bh = ah + 2 * T_IMG, bl = ah + 3 * T_IMG;
            #pragma unroll
            for (int ks = 0; ks < TK / 8; ++ks) {
                const uint32_t ko = (uint32_t)ks * 2 * T_LBO;             // K = 8 -> two chunks of 4
                const uint64_t dah = make_desc(ah + ko, T_LBO, 128), dal = make_desc(al + ko, T_LBO, 128);
                const uint64_t dbh = make_desc(bh + ko, T_LBO, 128), dbl = make_desc(bl + ko, T_LBO, 128);
                umma_tf32(tmem, dal, dbh, idesc, (it > 0 || ks > 0) ? 1u : 0u);    // small terms first
                umma_tf32(tmem, dah, dbl, idesc, 1u);
                umma_tf32(tmem, dah, dbh, idesc, 1u);
            }
            umma_commit(&done[s]);
        }
    }
    {
        const int last = nit - 1;
        mbar_wait(&done[last & 1], (uint32_t)(last >> 1) & 1u);       // a commit covers every earlier MMA of the thread
        tc_fence_after();
    }
    // ---- epilogue: warp w reads lanes (w & 3) * 32 .. +31 (its tensor-memory sub-partition) of the
    // column range (w >> 2) * (128 / (warps / 4)) .. of the accumulator
    constexpr int CW = 128 / (TC_THREADS / 128);         // columns per warp
    const float* bias = a.bias ? a.bias + (size_t)grp * a.bias_grp : nullptr;
    const int m = m0 + (warp & 3) * 32 + lane;
    const bool row_ok = m < a.M && (COMP || full || (m % sd) < nb);
    #pragma unroll 1
    for (int c = 0; c < CW / 16; ++c) {
        const int col0 = (warp >> 2) * CW + c * 16;
        float v[16];
        tmem_ld16(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col0, v);
        if (row_ok) {
            #pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int n = n0 + col0 + j;
                if (n < a.N) C[(size_t)m * a.ldc + n] = v[j] + (bias ? bias[n] : 0.0f);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

// Vector variant of the staging for GEMMs whose operands are both k-contiguous and 16-byte aligned
// (dz.W^T: every dLoss/dx GEMM): 4 consecutive k of a row are one 16-byte global load and one 16-byte
// core-matrix row of the K-major image.  Ragged edges and partial batches use guarded scalar loads.
// (For row-contiguous operands two alternatives were measured and dropped: MN-major images did not
// reproduce the K-major results, and an in-warp 4x4 shuffle transpose was slower than the scalar
// staging with its conflict-free lane mapping -- profiles/README.md r1g.)
constexpr int V_LBO_K = 2048 + 32;           // stride between K chunks of 4 (16 row groups x 128 B, padded: bank spread)
constexpr int V_IMG = (TK / 4) * V_LBO_K;
constexpr int V_STAGE = 4 * V_IMG;

__global__ void __launch_bounds__(TC_THREADS, 2)
lstm_bgemm_tcv_kernel(const __grid_constant__ GemmArgs a) {
    using namespace gbptx;
    extern __shared__ __align__(128) uint8_t tsm[];
    __shared__ __align__(8) uint64_t done[2];
    __shared__ uint32_t s_tmem;
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    if (nb == 0) return;
    const int sd = a.seq_dim;
    const bool full = nb == sd;
    const float* __restrict__ A = a.A + (size_t)grp * a.a_grp;
    const float* __restrict__ B = a.B + (size_t)grp * a.b_grp;
    float* C = a.C + (size_t)grp * a.c_grp;
    const int m0 = blockIdx.y * 128, n0 = blockIdx.x * 128;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        mbar_init(&done[0], 1); mbar_init(&done[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(&s_tmem, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;

    constexpr int UNITS = 128 * TK / 4 / TC_THREADS;        // 16-byte units per thread per operand per slab
    // unit i = tid + e * TC_THREADS: k chunk i & 3 of row i >> 2
    float4 ra[UNITS], rb[UNITS];
    auto fetch_op = [&](const float* __restrict__ P, int ld, int r0, int rows, bool rows_masked, int k0, float4* out) {
        #pragma unroll
        for (int e = 0; e < UNITS; ++e) {
            const int i = tid + e * TC_THREADS;
            const int row = r0 + (i >> 2), k = k0 + (i & 3) * 4;
            const bool row_ok = row < rows && (full || !rows_masked || (row % sd) < nb);
            if (row_ok && k + 3 < a.K) {
                out[e] = *reinterpret_cast<const float4*>(P + (size_t)row * ld + k);
            } else {
                float t[4];
                #pragma unroll
                for (int q = 0; q < 4; ++q) t[q] = (row_ok && k + q < a.K) ? P[(size_t)row * ld + k + q] : 0.0f;
                out[e] = make_float4(t[0], t[1], t[2], t[3]);
            }
        }
    };
    auto fetch = [&](int k0) {
        fetch_op(A, a.lda, m0, a.M, true, k0, ra);      // the (t, seq) mask lives on the rows of A
        fetch_op(B, a.ldb, n0, a.N, false, k0, rb);
    };
    auto put = [&](uint8_t* hi_img, uint8_t* lo_img, int e, const float4& v) {
        const int i = tid + e * TC_THREADS;
        const int row = i >> 2;
        const uint32_t off = (uint32_t)(i & 3) * V_LBO_K + (uint32_t)(row >> 3) * 128 + (uint32_t)(row & 7) * 16;
        uint4 hi, lo;
        hi.x = f32_to_tf32(v.x); hi.y = f32_to_tf32(v.y); hi.z = f32_to_tf32(v.z); hi.w = f32_to_tf32(v.w);
        lo.x = f32_to_tf32(v.x - __uint_as_float(hi.x)); lo.y = f32_to_tf32(v.y - __uint_as_float(hi.y));
        lo.z = f32_to_tf32(v.z - __uint_as_float(hi.z)); lo.w = f32_to_tf32(v.w - __uint_as_float(hi.w));
        *reinterpret_cast<uint4*>(hi_img + off) = hi;
        *reinterpret_cast<uint4*>(lo_img + off) = lo;
    };
    const uint32_t idesc = make_idesc_tf32(128, 128);
    const int nit = (a.K + TK - 1) / TK;
    fetch(0);
    for (int it = 0; it < nit; ++it) {
        const int s = it & 1;
        uint8_t* st = tsm + (size_t)s * V_STAGE;
        if (it >= 2) mbar_wait(&done[s], (uint32_t)((it >> 1) - 1) & 1u);
        #pragma unroll
        for (int e = 0; e < UNITS; ++e) put(st, st + V_IMG, e, ra[e]);
        #pragma unroll
        for (int e = 0; e < UNITS; ++e) put(st + 2 * V_IMG, st + 3 * V_IMG, e, rb[e]);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (it + 1 < nit) fetch((it + 1) * TK);
        if (tid == 0) {
            tc_fence_after();
            const uint32_t ah = smem_u32(st), al = ah + V_IMG, bh = ah + 2 * V_IMG, bl = ah + 3 * V_IMG;
            #pragma unroll
            for (int ks = 0; ks < TK / 8; ++ks) {
                const uint32_t ko = (uint32_t)ks * 2 * V_LBO_K;             // K = 8 -> two chunks of 4
                const uint64_t dah = make_desc(ah + ko, V_LBO_K, 128), dal = make_desc(al + ko, V_LBO_K, 128);
                const uint64_t dbh = make_desc(bh + ko, V_LBO_K, 128), dbl = make_desc(bl + ko, V_LBO_K, 128);
                umma_tf32(tmem, dal, dbh, idesc, (it > 0 || ks > 0) ? 1u : 0u);
                umma_tf32(tmem, dah, dbl, idesc, 1u);
                umma_tf32(tmem, dah, dbh, idesc, 1u);
            }
            umma_commit(&done[s]);
        }
    }
    {
        const int last = nit - 1;
        mbar_wait(&done[last & 1], (uint32_t)(last >> 1) & 1u);
        tc_fence_after();
    }
    constexpr int CW = 128 / (TC_THREADS / 128);
    const float* bias = a.bias ? a.bias + (size_t)grp * a.bias_grp : nullptr;
    const int m = m0 + (warp & 3) * 32 + lane;
    const bool row_ok = m < a.M && (full || (m % sd) < nb);
    #pragma unroll 1
    for (int c = 0; c < CW / 16; ++c) {
        const int col0 = (warp >> 2) * CW + c * 16;
        float v[16];
        tmem_ld16(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col0, v);
        if (row_ok) {
            #pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int n = n0 + col0 + j;
                if (n < a.N) C[(size_t)m * a.ldc + n] = v[j] + (bias ? bias[n] : 0.0f);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

// layer-0 operand of a training step, dense: xs[t][seq][k] = scale(x[rows_lo + seq_base + seq + t][k])
__global__ void lstm_gather_x_kernel(GroupCtx g, int B, int L, int T_in, const float* __restrict__ x,
                                     const float* __restrict__ in_scale, const float* __restrict__ in_min,
                                     float* __restrict__ xs, int64_t xs_grp) {
    const int grp = blockIdx.z;
    const int nb = group_nb(g, grp);
    const int64_t total = (int64_t)L * B * T_in;
    const float* sc = in_scale ? in_scale + (size_t)grp * T_in : nullptr;
    const float* mn = in_min ? in_min + (size_t)grp * T_in : nullptr;
    const int64_t row0 = g.rows_lo[grp] + g.seq_base;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(i % T_in);
        const int64_t r = i / T_in;
        const int s = (int)(r % B), t = (int)(r / B);
        float v = 0.0f;
        if (s < nb) { v = x[(row0 + s + t) * T_in + k]; if (sc) v = fmaf(v, sc[k], mn[k]); }
        xs[(size_t)grp * xs_grp + i] = v;
    }
}

// bias gradients: out[grp][n] = sum over rows r = (t, seq < nb) of dz[r][n]
__global__ void lstm_colsum_kernel(GroupCtx g, int B, int rows, int N, const float* __restrict__ dz, int64_t dz_grp,
                                   float* __restrict__ out, int64_t out_grp, int64_t out_off) {
    const int grp = blockIdx.z;
    const int nb = group_nb(g, grp);
    const int n = blockIdx.x * 32 + (threadIdx.x & 31);
    const int lane_r = threadIdx.x >> 5;                 // 8 row lanes
    __shared__ float part[8][33];
    float acc = 0.0f;
    if (n < N) {
        // four independent partial sums: the loads of a thread's 4 rows are in flight together (one dependent
        // add per load made this kernel 30 us for 400 KB: pure load latency)
        const float* base = dz + (size_t)grp * dz_grp + n;
        float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
        int r = lane_r;
        for (; r + 24 < rows; r += 32) {
            const float v0 = ((r % B) < nb) ? base[(size_t)r * N] : 0.0f;
            const float v1 = (((r + 8) % B) < nb) ? base[(size_t)(r + 8) * N] : 0.0f;
            const float v2 = (((r + 16) % B) < nb) ? base[(size_t)(r + 16) * N] : 0.0f;
            const float v3 = (((r + 24) % B) < nb) ? base[(size_t)(r + 24) * N] : 0.0f;
            a0 += v0; a1 += v1; a2 += v2; a3 += v3;
        }
        for (; r < rows; r += 8)
            if ((r % B) < nb) a0 += base[(size_t)r * N];
        acc = (a0 + a1) + (a2 + a3);
    }
    part[lane_r][threadIdx.x & 31] = acc;
    __syncthreads();
    if (lane_r == 0 && n < N) {
        for (int q = 1; q < 8; ++q) acc += part[q][threadIdx.x & 31];
        out[(size_t)grp * out_grp + out_off + n] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// The recurrence of a training step, persistent: ONE launch per layer walks all L time steps.
// A fit job is a thread-block cluster of CL CTAs; CTA c keeps the recurrent weights of its slice of
// units (all four gate columns) in shared memory for the whole sequence, so U is read once per layer
// per step instead of once per time step, and time steps are separated by a cluster barrier instead
// of a kernel launch.
//   forward : z_t = (x_t.W + b)  [already in `gates`, from lstm_bgemm_kernel]  + h_{t-1}.U[:, own columns];
//             gates, c_t, h_t for the own units; h_t is broadcast into every CTA's next h buffer (DSMEM).
//   backward: dz_t for the own units from dLoss/dh_t (from above + recurrent) and the cached gates;
//             partial dh_rec[s][j] = sum over OWN columns n of dz_t[s][n].U[j][n] for all units j, sent to
//             the CTA owning unit j, which adds the CL partials in rank order (deterministic).
struct RecArgs {
    GroupCtx g;
    int B, BP, L, u, act, us, nc, CL, width, NG, top;
    const float* params; int64_t n_params, u_off;
    float* gates; float* hs; float* cs; float* ac;      // [t][seq][4u] / [t][seq][u] caches, group stride gs
    const float* dH; float* dz;                         // backward: dLoss/dh from above [t][seq][u]; dz out [t][seq][4u]
    int64_t gs;
};
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_peer(const float* local, uint32_t rank, float v) {
    uint32_t addr;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(addr) : "r"((uint32_t)__cvta_generic_to_shared(local)), "r"(rank));
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
constexpr int REC_SG = 16;          // sequences per thread per pass of the small GEMMs

__global__ void lstm_rec_fwd_kernel(const __grid_constant__ RecArgs a) {
    extern __shared__ __align__(16) float rsm[];
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    if (nb == 0) return;                              // the whole cluster leaves together
    const int rank = (int)cluster_rank();
    const int u = a.u, us = a.us, nc = a.nc, B = a.B, BP = a.BP, CL = a.CL;
    const int tid = threadIdx.x, nthr = blockDim.x;
    float* Us = rsm;                                  // [u][nc]     own columns of U, column = gate*us + unit
    float* hb = Us + (size_t)u * nc;                  // [2][u][BP]  h_{t-1} / h_t, transposed (seq contiguous)
    float* zb = hb + (size_t)2 * u * BP;              // [nc][BP+1]  pre-activations of the own columns
    float* cst = zb + (size_t)nc * (BP + 1);          // [us][BP]    cell state
    const int j0 = rank * us, nu = max(0, min(us, u - j0));
    const float* U = a.params + (size_t)grp * a.n_params + a.u_off;
    for (int i = tid; i < u * nc; i += nthr) {
        const int k = i / nc, c = i - k * nc, gte = c / us, j = c - gte * us;
        Us[i] = j < nu ? U[(size_t)k * 4 * u + gte * u + j0 + j] : 0.0f;
    }
    for (int i = tid; i < 2 * u * BP; i += nthr) hb[i] = 0.0f;
    for (int i = tid; i < us * BP; i += nthr) cst[i] = 0.0f;
    __syncthreads();
    cluster_sync_all();                               // every CTA initialised before any peer writes into it
    float* gates = a.gates + (size_t)grp * a.gs;
    float* hs = a.hs + (size_t)grp * a.gs; float* cs = a.cs + (size_t)grp * a.gs; float* ac = a.ac + (size_t)grp * a.gs;
    const int col = tid % a.width, sg = tid / a.width;
    const int cg = col / us, cj = col - cg * us;
    for (int t = 0; t < a.L; ++t) {
        const float* hcur = hb + (size_t)(t & 1) * u * BP;
        float* hnext = hb + (size_t)((t + 1) & 1) * u * BP;
        // ---- phase A: z[col][s] = (x.W + b)[s][col] + sum_k h_{t-1}[s][k] * U[k][col]
        if (col < nc) {
            for (int sb = sg * REC_SG; sb < BP; sb += a.NG * REC_SG) {
                float acc[REC_SG];
                #pragma unroll
                for (int i = 0; i < REC_SG; ++i) {
                    const int sq = sb + i;
                    acc[i] = (sq < nb && cj < nu) ? gates[((size_t)t * B + sq) * 4 * u + cg * u + j0 + cj] : 0.0f;
                }
                if (t > 0) {
                    #pragma unroll 4
                    for (int k = 0; k < u; ++k) {
                        const float uv = Us[k * nc + col];
                        const float4* h4 = reinterpret_cast<const float4*>(hcur + (size_t)k * BP + sb);
                        #pragma unroll
                        for (int q = 0; q < REC_SG / 4; ++q) {
                            const float4 hv = h4[q];
                            acc[4 * q] = fmaf(hv.x, uv, acc[4 * q]); acc[4 * q + 1] = fmaf(hv.y, uv, acc[4 * q + 1]);
                            acc[4 * q + 2] = fmaf(hv.z, uv, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(hv.w, uv, acc[4 * q + 3]);
                        }
                    }
                }
                #pragma unroll
                for (int i = 0; i < REC_SG; ++i) zb[col * (BP + 1) + sb + i] = acc[i];
            }
        }
        __syncthreads();
        // ---- phase B: gates, cell update, h_t for the own units; h_t goes to every CTA of the cluster
        for (int e = tid; e < us * BP; e += nthr) {
            const int j = e / BP, sq = e - j * BP;
            if (j >= nu) continue;
            float hval = 0.0f;
            if (sq < nb) {
                const float ig = sigmoidf_(zb[(0 * us + j) * (BP + 1) + sq]), fg = sigmoidf_(zb[(1 * us + j) * (BP + 1) + sq]);
                const float gg = gb_act(a.act, zb[(2 * us + j) * (BP + 1) + sq]), og = sigmoidf_(zb[(3 * us + j) * (BP + 1) + sq]);
                const float cn = fmaf(fg, cst[e], ig * gg);
                const float acv = gb_act(a.act, cn);
                cst[e] = cn;
                hval = og * acv;
                const size_t r = (size_t)t * B + sq;
                float* gp = gates + r * 4 * u + j0 + j;
                gp[0] = ig; gp[u] = fg; gp[2 * u] = gg; gp[3 * u] = og;
                cs[r * u + j0 + j] = cn; ac[r * u + j0 + j] = acv; hs[r * u + j0 + j] = hval;
            }
            const float* dst = hnext + (size_t)(j0 + j) * BP + sq;
            for (int r = 0; r < CL; ++r) st_peer(dst, (uint32_t)r, hval);
        }
        cluster_sync_all();
    }
}

__global__ void lstm_rec_bwd_kernel(const __grid_constant__ RecArgs a) {
    extern __shared__ __align__(16) float rsm[];
    const int grp = blockIdx.z;
    const int nb = group_nb(a.g, grp);
    if (nb == 0) return;
    const int rank = (int)cluster_rank();
    const int u = a.u, us = a.us, nc = a.nc, B = a.B, BP = a.BP, CL = a.CL;
    const int tid = threadIdx.x, nthr = blockDim.x;
    float* UT = rsm;                                  // [nc][u]          U[j][own column n], n-major
    float* dzT = UT + (size_t)nc * u;                 // [nc][BP]         dz_t of the own columns, transposed
    float* recv = dzT + (size_t)nc * BP;              // [2][CL][us][BP]  partial dh_rec from every CTA
    float* dcs = recv + (size_t)2 * CL * us * BP;     // [us][BP]         running dLoss/dc
    const int j0 = rank * us, nu = max(0, min(us, u - j0));
    const float* U = a.params + (size_t)grp * a.n_params + a.u_off;
    for (int i = tid; i < nc * u; i += nthr) {
        const int n = i / u, j = i - n * u, gte = n / us, jl = n - gte * us;
        UT[i] = jl < nu ? U[(size_t)j * 4 * u + gte * u + j0 + jl] : 0.0f;
    }
    for (int i = tid; i < 2 * CL * us * BP; i += nthr) recv[i] = 0.0f;
    for (int i = tid; i < us * BP; i += nthr) dcs[i] = 0.0f;
    __syncthreads();
    cluster_sync_all();
    const float* gates = a.gates + (size_t)grp * a.gs;
    const float* cs = a.cs + (size_t)grp * a.gs; const float* ac = a.ac + (size_t)grp * a.gs;
    const float* dH = a.dH ? a.dH + (size_t)grp * a.gs : nullptr;
    float* dz = a.dz + (size_t)grp * a.gs;
    const int jc = tid % a.width, sg = tid / a.width;
    for (int it = 0; it < a.L; ++it) {
        const int t = a.L - 1 - it;
        // ---- phase E: dz_t of the own units
        for (int e = tid; e < us * BP; e += nthr) {
            const int jl = e / BP, sq = e - jl * BP;
            float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            if (jl < nu && sq < nb) {
                const size_t r = (size_t)t * B + sq;
                float dh = 0.0f;
                if (dH && (!a.top || t == a.L - 1)) dh += dH[r * u + j0 + jl];
                if (it > 0) {
                    const float* rp = recv + (size_t)((it - 1) & 1) * CL * us * BP + (size_t)jl * BP + sq;
                    float rec = 0.0f;
                    for (int q = 0; q < CL; ++q) rec += rp[(size_t)q * us * BP];
                    dh += rec;
                }
                const float* gp = gates + r * 4 * u + j0 + jl;
                const float ig = gp[0], fg = gp[u], gg = gp[2 * u], og = gp[3 * u];
                const float acv = ac[r * u + j0 + jl];
                const float cp = t > 0 ? cs[(r - B) * u + j0 + jl] : 0.0f;
                const float dc_in = it == 0 ? 0.0f : dcs[e];
                const float d_o = dh * acv;
                const float dc = dc_in + dh * og * act_grad_h(a.act, acv);
                dcs[e] = dc * fg;
                d0 = dc * gg * ig * (1.0f - ig);
                d1 = dc * cp * fg * (1.0f - fg);
                d2 = dc * ig * act_grad_h(a.act, gg);
                d3 = d_o * og * (1.0f - og);
                float* dp = dz + r * 4 * u + j0 + jl;
                dp[0] = d0; dp[u] = d1; dp[2 * u] = d2; dp[3 * u] = d3;
            }
            dzT[(0 * us + jl) * BP + sq] = d0; dzT[(1 * us + jl) * BP + sq] = d1;
            dzT[(2 * us + jl) * BP + sq] = d2; dzT[(3 * us + jl) * BP + sq] = d3;
        }
        __syncthreads();
        // ---- phase G: partial dh_rec[s][j] over the own columns, sent to the owner of unit j
        if (t > 0 && jc < u) {
            const int owner = jc / us, jl = jc - owner * us;
            for (int sb = sg * REC_SG; sb < BP; sb += a.NG * REC_SG) {
                float acc[REC_SG] = {};
                #pragma unroll 4
                for (int n = 0; n < nc; ++n) {
                    const float uv = UT[n * u + jc];
                    const float4* d4 = reinterpret_cast<const float4*>(dzT + (size_t)n * BP + sb);
                    #pragma unroll
                    for (int q = 0; q < REC_SG / 4; ++q) {
                        const float4 dv = d4[q];
                        acc[4 * q] = fmaf(dv.x, uv, acc[4 * q]); acc[4 * q + 1] = fmaf(dv.y, uv, acc[4 * q + 1]);
                        acc[4 * q + 2] = fmaf(dv.z, uv, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(dv.w, uv, acc[4 * q + 3]);
                    }
                }
                const float* dst = recv + ((size_t)(it & 1) * CL + rank) * us * BP + (size_t)jl * BP + sb;
                #pragma unroll
                for (int i = 0; i < REC_SG; ++i) st_peer(dst + i, (uint32_t)owner, acc[i]);
            }
        }
        cluster_sync_all();
    }
}

struct RecPlan { bool ok; int CL, us, nc, BP, width_f, ng_f, width_b, ng_b; size_t smem_f, smem_b; };
static RecPlan make_rec_plan_cl(int u, int B, int CL) {
    RecPlan r{};
    r.BP = (B + REC_SG - 1) / REC_SG * REC_SG;
    r.CL = CL;
    r.us = (u + r.CL - 1) / r.CL;
    r.nc = 4 * r.us;
    r.width_f = (r.nc + 31) / 32 * 32;
    r.width_b = (u + 31) / 32 * 32;
    const int passes = r.BP / REC_SG;
    r.ng_f = 512 / r.width_f < passes ? 512 / r.width_f : passes;
    r.ng_b = 512 / r.width_b < passes ? 512 / r.width_b : passes;
    r.smem_f = sizeof(float) * ((size_t)u * r.nc + (size_t)2 * u * r.BP + (size_t)r.nc * (r.BP + 1) + (size_t)r.us * r.BP);
    r.smem_b = sizeof(float) * ((size_t)r.nc * u + (size_t)r.nc * r.BP + (size_t)2 * r.CL * r.us * r.BP + (size_t)r.us * r.BP);
    r.ok = u <= 256 && r.ng_f >= 1 && r.ng_b >= 1 && r.smem_f <= 200 * 1024 && r.smem_b <= 200 * 1024;
    return r;
}
// Cluster size of the recurrence: a time step costs (B * u * 4u / CL) FMAs per CTA plus one cluster barrier + DSMEM
// hand-over.  The per-CTA FMA loop, not the barrier, is the longer part: measured on a 4-job fit (r2, lookback 16,
// profiles/README.md r2c) at 60 tags (u = 30-50) 1 / 2 / 4 / 8 CTAs per job = 388 / 264 / 206 / 174 ms, at 30 tags
// 208 (2-4 CTAs) vs 138 ms (8) -- so every layer with >= 3 units per CTA gets the full portable cluster of 8.
// The first size >= the rule whose slices fit in shared memory wins (large batches need more CTAs).
static RecPlan make_rec_plan(int u, int B) {
    int min_cl = u >= 24 ? 8 : (u >= 12 ? 4 : (u >= 6 ? 2 : 1));
    if (const char* e = getenv("GB200_LSTM_REC_CL")) {              // tuning knob: smallest cluster size to try
        const int v = atoi(e);
        if (v == 1 || v == 2 || v == 4 || v == 8) min_cl = v;
    }
    RecPlan r{};
    for (int cl = min_cl; cl <= 8; cl <<= 1) {
        r = make_rec_plan_cl(u, B, cl);
        if (r.ok) return r;
    }
    return r;
}
static int launch_rec(bool fwd, const RecPlan& rp, RecArgs& a, int J, cudaStream_t stream) {
    a.BP = rp.BP; a.us = rp.us; a.nc = rp.nc; a.CL = rp.CL;
    a.width = fwd ? rp.width_f : rp.width_b; a.NG = fwd ? rp.ng_f : rp.ng_b;
    const size_t smem = fwd ? rp.smem_f : rp.smem_b;
    auto* kern = fwd ? lstm_rec_fwd_kernel : lstm_rec_bwd_kernel;
    GB_CUDA_CHECK(gb_allow_max_smem(kern));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(rp.CL, 1, J); cfg.blockDim = dim3(a.width * a.NG, 1, 1);
    cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = rp.CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    GB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, a));
    return GB_OK;
}

struct AdamArgs {
    GroupCtx g; gb200_adam adam; int64_t n_params;
    float* params; const float* grad; float* mv; int64_t* tcount;
};
__global__ void lstm_adam_kernel(const __grid_constant__ AdamArgs a) {
    const int grp = blockIdx.z;
    if (group_nb(a.g, grp) == 0) return;               // this job has no batch in this step
    const float tf = (float)(a.tcount[grp] + 1);
    const float alpha = a.adam.lr * sqrtf(1.0f - powf(a.adam.beta_2, tf)) / (1.0f - powf(a.adam.beta_1, tf));
    float* P = a.params + (size_t)grp * a.n_params;
    const float* G = a.grad + (size_t)grp * a.n_params;
    float* M = a.mv + (size_t)grp * 2 * a.n_params; float* V = M + a.n_params;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_params; i += (int64_t)gridDim.x * blockDim.x) {
        const float gr = G[i];
        float m = M[i], v = V[i];
        m += (gr - m) * (1.0f - a.adam.beta_1);
        v += (gr * gr - v) * (1.0f - a.adam.beta_2);
        M[i] = m; V[i] = v;
        P[i] -= alpha * m / (sqrtf(v) + a.adam.epsilon);
    }
}
// Last kernel of an optimizer step.  `advance` > 0 moves every group's window cursor (first sample row, windows
// left) forward by one batch on the device.  The kernels of a step read their batch from that cursor, so a group
// whose windows have run out sees nb = 0 and takes no step: no loss, no Adam update, no step count.
__global__ void lstm_step_end_kernel(GroupCtx g, int n_groups, int64_t* tcount, const float* loss_sum,
                                     float* epoch_acc, int T_out, float* primer_loss, int advance,
                                     int64_t* rows_cur, int32_t* nwin_cur) {
    const int grp = blockIdx.x * blockDim.x + threadIdx.x;
    if (grp >= n_groups) return;
    const int nb = group_nb(g, grp);
    if (nb > 0) {
        tcount[grp] += 1;
        const float batch_loss = loss_sum[grp] / (float)(nb * T_out);
        if (primer_loss) primer_loss[grp] = batch_loss;
        else epoch_acc[grp] += batch_loss * nb;            // Keras: sample-weighted running mean
    }
    if (advance > 0) { rows_cur[grp] += advance; nwin_cur[grp] -= advance; }
}
__global__ void lstm_epoch_end_kernel(int n_groups, const int32_t* n_win, float* epoch_acc, float* hist, int epochs, int e) {
    const int grp = blockIdx.x * blockDim.x + threadIdx.x;
    if (grp >= n_groups) return;
    hist[(size_t)grp * epochs + e] = n_win[grp] > 0 ? epoch_acc[grp] / (float)n_win[grp] : NAN;
    epoch_acc[grp] = 0.0f;
}

inline int cdiv(int a, int b) { return (a + b - 1) / b; }
inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

int64_t gb200_lstm_param_count(const gb200_lstm_arch* a) {
    if (!a || a->n_layers < 1 || a->n_layers > GB200_MAX_LAYERS) return 0;
    return make_plan(a).n_params;
}

int64_t gb200_lstm_out_rows(const gb200_lstm_arch* a, int64_t n_rows) {
    if (!a) return 0;
    const int64_t n = n_rows - a->lookback_window + 1 - a->lookahead;
    return n > 0 ? n : 0;
}

// predict scratch: per layer two h buffers + one c buffer of [max_windows][u]
int64_t gb200_lstm_scratch_bytes(const gb200_lstm_arch* a, int64_t max_windows, int precision) {
    if (!a || a->n_layers < 1 || a->n_layers > GB200_MAX_LAYERS || max_windows < 1) return 0;
    if (precision == GB200_PREC_BF16_TC) return gb_lstm_tc_scratch_bytes(a, max_windows);
    const LstmPlan p = make_plan(a);
    return (int64_t)align256((size_t)3 * p.sum_u * max_windows * sizeof(float)) + 1024;
}

static int check_lstm_arch(const gb200_lstm_arch* a) {
    GB_REQUIRE(a != nullptr, "arch is NULL");
    GB_REQUIRE(a->n_layers >= 1 && a->n_layers <= GB200_MAX_LAYERS, "n_layers=%d out of range", a->n_layers);
    GB_REQUIRE(a->n_features >= 1 && a->n_features_out >= 1, "bad feature counts");
    GB_REQUIRE(a->lookback_window >= 1 && a->lookahead >= 0, "bad lookback_window / lookahead");
    for (int l = 0; l < a->n_layers; ++l) GB_REQUIRE(a->units[l] >= 1, "units[%d] must be >= 1", l);
    return GB_OK;
}

int gb200_lstm_predict(gb200_fleet* f, const gb200_lstm_arch* arch, int precision, const float* params,
                       const float* in_scale, const float* in_min, const float* x,
                       const int64_t* out_row_off, float* model_out,
                       void* scratch, int64_t scratch_bytes, void* stream_) {
    GB_REQUIRE(f != nullptr, "fleet is NULL");
    int rc = check_lstm_arch(arch); if (rc) return rc;
    GB_REQUIRE(params && x && out_row_off && model_out && scratch, "NULL argument");
    GB_REQUIRE((in_scale == nullptr) == (in_min == nullptr), "in_scale and in_min must be given together");
    GB_REQUIRE(precision == GB200_PREC_F32 || precision == GB200_PREC_BF16_TC, "unknown precision %d", precision);
    cudaStream_t stream = (cudaStream_t)stream_;
    if (precision == GB200_PREC_BF16_TC) {
        // host-side prefix of the per-Machine output rows (out_row_off is its device twin)
        std::vector<int64_t> off(f->n_machines + 1, 0);
        for (int m = 0; m < f->n_machines; ++m)
            off[m + 1] = off[m] + gb200_lstm_out_rows(arch, f->h_row_hi[m] - f->h_row_lo[m]);
        return gb_lstm_predict_tc(f, arch, params, in_scale, in_min, x, off.data(), model_out, scratch, scratch_bytes, stream);
    }
    const LstmPlan p = make_plan(arch);
    const int64_t cap64 = (scratch_bytes - 1024) / ((int64_t)3 * p.sum_u * sizeof(float));
    GB_REQUIRE(cap64 >= 1, "scratch too small (see gb200_lstm_scratch_bytes)");
    const int cap = (int)(cap64 > (1 << 22) ? (1 << 22) : cap64);
    float* base = (float*)scratch;
    // per Machine n_win lives on the device next to the schedule: build a tiny array in the scratch tail
    int32_t* d_nwin = (int32_t*)((char*)scratch + scratch_bytes - 1024);
    for (int m = 0; m < f->n_machines; ++m) {
        const int64_t rows = f->h_row_hi[m] - f->h_row_lo[m];
        const int64_t n_win = rows - p.L + 1 - p.lookahead;
        if (rows <= 0) continue;
        GB_REQUIRE(p.L < rows, "For KerasLSTMForecast lookback_window must be < size of X (machine %d)", m);
        if (n_win <= 0) continue;
        const int32_t nw32 = (int32_t)n_win;
        GB_CUDA_CHECK(cudaMemcpyAsync(d_nwin, &nw32, sizeof(int32_t), cudaMemcpyHostToDevice, stream));
        for (int64_t k0 = 0; k0 < n_win; k0 += cap) {
            const int nb = (int)((n_win - k0) < cap ? (n_win - k0) : cap);
            GroupCtx g{f->d_row_lo + m, d_nwin, (int)k0, cap};
            // state layout: for layer l: hA[cap][u], hB[cap][u], c[cap][u]
            size_t off = 0;
            float* hA[GB200_MAX_LAYERS]; float* hB[GB200_MAX_LAYERS]; float* cS[GB200_MAX_LAYERS];
            for (int l = 0; l < p.n_layers; ++l) {
                hA[l] = base + off; off += (size_t)cap * p.ld[l].u;
                hB[l] = base + off; off += (size_t)cap * p.ld[l].u;
                cS[l] = base + off; off += (size_t)cap * p.ld[l].u;
            }
            for (int t = 0; t < p.L; ++t) {
                for (int l = 0; l < p.n_layers; ++l) {
                    StepArgs a{};
                    a.g = g; a.in = p.ld[l].in; a.u = p.ld[l].u; a.act = p.acts[l]; a.t = t; a.layer = l;
                    a.params = params + (size_t)m * p.n_params; a.n_params = 0;
                    a.w_off = p.ld[l].w_off; a.u_off = p.ld[l].u_off; a.b_off = p.ld[l].b_off;
                    a.x = x; a.T_in = p.T_in;
                    a.in_scale = in_scale ? in_scale + (size_t)m * p.T_in : nullptr;
                    a.in_min = in_min ? in_min + (size_t)m * p.T_in : nullptr;
                    float* hcur = (t & 1) ? hB[l] : hA[l];
                    float* hprev = (t & 1) ? hA[l] : hB[l];
                    if (l > 0) { a.xin = (t & 1) ? hB[l - 1] : hA[l - 1]; a.xin_seq_stride = p.ld[l - 1].u; }
                    a.h_prev = t > 0 ? hprev : nullptr; a.hprev_seq_stride = a.u;
                    a.h_out = hcur; a.hout_seq_stride = a.u;
                    a.c_prev = t > 0 ? cS[l] : nullptr; a.cprev_seq_stride = a.u;
                    a.c_out = cS[l]; a.cout_seq_stride = a.u;
                    dim3 grid(cdiv(nb, ST_SEQ), cdiv(a.u, ST_UNITS), 1);
                    lstm_step_fwd_kernel<<<grid, ST_THREADS, 0, stream>>>(a);
                }
            }
            DenseArgs d{};
            d.g = g; d.u = p.ld[p.n_layers - 1].u; d.T_out = p.T_out; d.act = p.out_act;
            d.params = params + (size_t)m * p.n_params; d.n_params = 0; d.w_off = p.dense_w_off; d.b_off = p.dense_b_off;
            d.h = ((p.L - 1) & 1) ? hB[p.n_layers - 1] : hA[p.n_layers - 1]; d.h_seq_stride = d.u;
            d.out = model_out; d.out_row_off = out_row_off + m;
            int blocks = cdiv(nb * p.T_out, 256); if (blocks > 148 * 8) blocks = 148 * 8;
            lstm_dense_out_kernel<<<dim3(blocks, 1, 1), 256, 0, stream>>>(d);
            GB_CUDA_CHECK(cudaGetLastError());
        }
    }
    return GB_OK;
}

// ---- training scratch (per job): see the layout in gb200_lstm_fit
static size_t fit_floats_per_job(const LstmPlan& p, int B) {
    size_t n = 0;
    const size_t BL = (size_t)B * p.L;
    for (int l = 0; l < p.n_layers; ++l) {
        const size_t u = p.ld[l].u;
        n += BL * u * 3;            // hs, cs, act(c)
        n += BL * 4 * u * 2;        // gates, dz
        n += BL * u;                // dH (dLoss/dh_t delivered to this layer from above)
        n += (size_t)B * u * 2;     // dh_rec, dc
    }
    n += (size_t)B * p.T_out * 2;   // yhat, dzd
    n += BL * p.T_in;               // dense scaled layer-0 input [t][seq][T_in]
    n += (size_t)p.n_params * 3;    // grad, m, v
    return n + 64;
}

int64_t gb200_lstm_fit_scratch_bytes(const gb200_lstm_arch* a, int32_t n_jobs, int32_t batch_size) {
    if (!a || a->n_layers < 1 || a->n_layers > GB200_MAX_LAYERS || n_jobs < 1 || batch_size < 1) return 0;
    const LstmPlan p = make_plan(a);
    return (int64_t)align256(fit_floats_per_job(p, batch_size) * sizeof(float)) * n_jobs + 4096 + (int64_t)n_jobs * 64;
}

int gb200_lstm_fit(const gb200_lstm_arch* arch, const gb200_adam* adam, int32_t n_jobs,
                   const int64_t* job_rows_lo_host, const int64_t* job_rows_hi_host,
                   const float* in_scale, const float* in_min, const float* x, const float* y,
                   int32_t epochs, int32_t batch_size, float* params,
                   float* hist_loss, float* primer_loss,
                   void* scratch, int64_t scratch_bytes, void* stream_) {
    int rc = check_lstm_arch(arch); if (rc) return rc;
    GB_REQUIRE(adam && job_rows_lo_host && job_rows_hi_host && x && params && scratch, "NULL argument");
    GB_REQUIRE(n_jobs >= 1 && epochs >= 1 && batch_size >= 1, "bad n_jobs / epochs / batch_size");
    GB_REQUIRE((in_scale == nullptr) == (in_min == nullptr), "in_scale and in_min must be given together");
    GB_REQUIRE(y != nullptr || arch->n_features == arch->n_features_out, "y may alias x only when n_features == n_features_out");
    GB_REQUIRE(scratch_bytes >= gb200_lstm_fit_scratch_bytes(arch, n_jobs, batch_size), "scratch too small (see gb200_lstm_fit_scratch_bytes)");
    cudaStream_t stream = (cudaStream_t)stream_;
    const LstmPlan p = make_plan(arch);
    const int J = n_jobs, B = batch_size, L = p.L;
    const float* ysrc = y ? y : x;

    // ---- control block at the tail of the scratch: rows_lo[J] (i64), n_win[J] (i32), tcount[J] (i64), loss_sum[J], epoch_acc[J]
    char* tail = (char*)scratch + scratch_bytes - (4096 + (size_t)J * 64);
    int64_t* d_rows_lo = (int64_t*)tail;
    int64_t* d_tcount = d_rows_lo + J;
    int32_t* d_nwin = (int32_t*)(d_tcount + J);
    float* d_loss = (float*)(d_nwin + J);
    float* d_epoch = d_loss + J;
    int32_t* d_nwin_cur = (int32_t*)(d_epoch + J);                  // windows left from the cursor
    int64_t* d_rows_cur = (int64_t*)(tail + 4096 + (size_t)J * 48);  // cursor: first sample row of the next batch
    std::vector<int64_t> rows_lo(J); std::vector<int32_t> nwin(J); int max_win = 0;
    for (int j = 0; j < J; ++j) {
        const int64_t rows = job_rows_hi_host[j] - job_rows_lo_host[j];
        GB_REQUIRE(L < rows, "For KerasLSTMForecast lookback_window must be < size of X (job %d)", j);
        rows_lo[j] = job_rows_lo_host[j];
        const int64_t nw = rows - L + 1 - p.lookahead;
        nwin[j] = (int32_t)(nw > 0 ? nw : 0);
        if (nwin[j] > max_win) max_win = nwin[j];
    }
    GB_CUDA_CHECK(cudaMemcpyAsync(d_rows_lo, rows_lo.data(), sizeof(int64_t) * J, cudaMemcpyHostToDevice, stream));
    GB_CUDA_CHECK(cudaMemcpyAsync(d_nwin, nwin.data(), sizeof(int32_t) * J, cudaMemcpyHostToDevice, stream));
    GB_CUDA_CHECK(cudaMemsetAsync(d_tcount, 0, sizeof(int64_t) * J, stream));
    GB_CUDA_CHECK(cudaMemsetAsync(d_epoch, 0, sizeof(float) * J, stream));
    GB_CUDA_CHECK(cudaStreamSynchronize(stream));       // host vectors go out of scope safely; one-off

    const size_t per_job = align256(fit_floats_per_job(p, B) * sizeof(float)) / sizeof(float);
    float* S = (float*)scratch;
    // per-job layout offsets (floats)
    size_t o = 0;
    size_t hs_o[GB200_MAX_LAYERS], cs_o[GB200_MAX_LAYERS], ac_o[GB200_MAX_LAYERS], gt_o[GB200_MAX_LAYERS],
           dz_o[GB200_MAX_LAYERS], dH_o[GB200_MAX_LAYERS], dr_o[GB200_MAX_LAYERS], dc_o[GB200_MAX_LAYERS];
    const size_t BL = (size_t)B * L;
    for (int l = 0; l < p.n_layers; ++l) {
        const size_t u = p.ld[l].u;
        hs_o[l] = o; o += BL * u; cs_o[l] = o; o += BL * u; ac_o[l] = o; o += BL * u;
        gt_o[l] = o; o += BL * 4 * u; dz_o[l] = o; o += BL * 4 * u; dH_o[l] = o; o += BL * u;
        dr_o[l] = o; o += (size_t)B * u; dc_o[l] = o; o += (size_t)B * u;
    }
    const size_t yh_o = o; o += (size_t)B * p.T_out;
    const size_t dzd_o = o; o += (size_t)B * p.T_out;
    const size_t x0_o = o; o += BL * p.T_in;
    const size_t grad_o = o; o += p.n_params;
    const size_t mv_o = o; o += 2 * (size_t)p.n_params;
    for (int j = 0; j < J; ++j)
        GB_CUDA_CHECK(cudaMemsetAsync(S + (size_t)j * per_job + mv_o, 0, sizeof(float) * 2 * p.n_params, stream));
    const int64_t gs = (int64_t)per_job;            // group stride of everything in the scratch

    // the per-time-step launch path stays as the fallback for very wide layers (GB200_LSTM_REC=0 forces it)
    bool use_rec = true;
    { const char* e = getenv("GB200_LSTM_REC"); if (e && atoi(e) == 0) use_rec = false; }
    // batched GEMMs: tcgen05 3xTF32 (fp32-accurate) by default, GB200_LSTM_GEMM=simt for the CUDA-core kernel
    // GB200_LSTM_GEMM: "simt" CUDA-core GEMM only; "tc" / "tcs" force the tensor-core GEMM for every launch
    // (vector / scalar staging) -- the parity tests use these; default: tensor cores from 64 tiles up
    bool use_vec = true, use_tc_gemm = true, force_tc = false;
    if (const char* e = getenv("GB200_LSTM_GEMM")) {
        if (e[0] == 's') use_tc_gemm = false;
        else if (e[0] == 't') { force_tc = true; use_vec = !(e[1] == 'c' && e[2] == 's'); }
    }
    // sequence buffers are [t][seq][width]: t stride = B*width, seq stride = width
    // a step reads its batch position from the device cursor (d_rows_cur / d_nwin_cur), never from a host value
    auto run_step = [&](int cap, float* primer_out, int advance) -> int {
        GroupCtx g{d_rows_cur, d_nwin_cur, 0, cap};
        GB_CUDA_CHECK(cudaMemsetAsync(d_loss, 0, sizeof(float) * J, stream));
        // ---------------- forward with caches, layer by layer: the input projection x_t.W + b of ALL
        // time steps is one GEMM, the recurrence adds h_{t-1}.U step by step
        auto gemm = [&](int comp, int M, int N, int K, const float* A, int64_t a_grp, int lda, int a_kc,
                        const float* Bm, int64_t b_grp, int ldb, int b_kc, float* Cm, int64_t c_grp, int ldc,
                        const float* bias, int64_t bias_grp) -> int {
            GemmArgs ga{};
            ga.g = g; ga.seq_dim = B; ga.M = M; ga.N = N; ga.K = K; ga.comp = comp;
            ga.A = A; ga.a_grp = a_grp; ga.lda = lda; ga.a_kcontig = a_kc;
            ga.B = Bm; ga.b_grp = b_grp; ga.ldb = ldb; ga.b_kcontig = b_kc;
            ga.C = Cm; ga.c_grp = c_grp; ga.ldc = ldc; ga.bias = bias; ga.bias_grp = bias_grp;
            if (use_tc_gemm && (force_tc || (int64_t)cdiv(N, 128) * cdiv(M, 128) * J >= 64)) {      // enough 128x128 tiles to fill the GPU
                // 16-byte staging when both operands are k-contiguous and every row starts 16-byte aligned
                const bool vec = use_vec && !comp && a_kc && b_kc && lda % 4 == 0 && ldb % 4 == 0 && a_grp % 4 == 0 && b_grp % 4 == 0
                                 && (reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(Bm) & 15) == 0;
                if (vec) {
                    auto* kv = lstm_bgemm_tcv_kernel;
                    GB_CUDA_CHECK(cudaFuncSetAttribute(kv, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * V_STAGE));
                    kv<<<dim3(cdiv(N, 128), cdiv(M, 128), J), TC_THREADS, 2 * V_STAGE, stream>>>(ga);
                    return GB_OK;
                }
                auto* kern = comp ? lstm_bgemm_tc_kernel<false, false, true>
                           : (b_kc ? lstm_bgemm_tc_kernel<true, true, false> : lstm_bgemm_tc_kernel<true, false, false>);
                GB_REQUIRE(comp ? (!a_kc && !b_kc) : (a_kc != 0), "lstm gemm: operand layout combination not instantiated");
                GB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * T_STAGE));
                kern<<<dim3(cdiv(N, 128), cdiv(M, 128), J), TC_THREADS, 2 * T_STAGE, stream>>>(ga);
                return GB_OK;
            }
            // big tiles once they fill the GPU, small ones for a handful of jobs
            if ((int64_t)cdiv(N, 128) * cdiv(M, 128) * J >= 148)
                lstm_bgemm_kernel<128, 128><<<dim3(cdiv(N, 128), cdiv(M, 128), J), 256, 0, stream>>>(ga);
            else
                lstm_bgemm_kernel<64, 64><<<dim3(cdiv(N, 64), cdiv(M, 64), J), 256, 0, stream>>>(ga);
            return GB_OK;
        };
        {
            const int64_t tot = (int64_t)L * B * p.T_in;
            int blocks = (int)((tot + 255) / 256); if (blocks > 2048) blocks = 2048;
            lstm_gather_x_kernel<<<dim3(blocks, 1, J), 256, 0, stream>>>(g, B, L, p.T_in, x, in_scale, in_min, S + x0_o, gs);
        }
        for (int l = 0; l < p.n_layers; ++l) {
            const int u = p.ld[l].u, in = p.ld[l].in;
            const float* Ain = l == 0 ? S + x0_o : S + hs_o[l - 1];
            gemm(0, L * B, 4 * u, in, Ain, gs, in, 1, params + p.ld[l].w_off, p.n_params, 4 * u, 0,
                 S + gt_o[l], gs, 4 * u, params + p.ld[l].b_off, p.n_params);
            const RecPlan rp = make_rec_plan(u, B);
            if (rp.ok && use_rec) {
                RecArgs ra{};
                ra.g = g; ra.B = B; ra.L = L; ra.u = u; ra.act = p.acts[l];
                ra.params = params; ra.n_params = p.n_params; ra.u_off = p.ld[l].u_off;
                ra.gates = S + gt_o[l]; ra.hs = S + hs_o[l]; ra.cs = S + cs_o[l]; ra.ac = S + ac_o[l]; ra.gs = gs;
                rc = launch_rec(true, rp, ra, J, stream);
                if (rc) return rc;
                continue;
            }
            for (int t = 0; t < L; ++t) {
                StepArgs a{};
                a.g = g; a.in = in; a.u = u; a.act = p.acts[l]; a.t = t; a.layer = l; a.pre = 1;
                a.params = params; a.n_params = p.n_params;
                a.w_off = p.ld[l].w_off; a.u_off = p.ld[l].u_off; a.b_off = p.ld[l].b_off;
                a.T_in = p.T_in;
                a.h_prev = t > 0 ? S + hs_o[l] + (size_t)(t - 1) * B * u : nullptr; a.hprev_seq_stride = u; a.hprev_grp_stride = gs;
                a.h_out = S + hs_o[l] + (size_t)t * B * u; a.hout_seq_stride = u; a.hout_grp_stride = gs;
                a.c_prev = t > 0 ? S + cs_o[l] + (size_t)(t - 1) * B * u : nullptr; a.cprev_seq_stride = u; a.cprev_grp_stride = gs;
                a.c_out = S + cs_o[l] + (size_t)t * B * u; a.cout_seq_stride = u; a.cout_grp_stride = gs;
                a.gates = S + gt_o[l] + (size_t)t * B * 4 * u; a.gates_seq_stride = 4 * u; a.gates_grp_stride = gs;
                a.actc = S + ac_o[l] + (size_t)t * B * u; a.actc_seq_stride = u; a.actc_grp_stride = gs;
                lstm_step_fwd_kernel<<<dim3(cdiv(cap, ST_SEQ), cdiv(u, ST_UNITS), J), ST_THREADS, 0, stream>>>(a);
            }
        }
        const int ul = p.ld[p.n_layers - 1].u;
        const float* h_last = S + hs_o[p.n_layers - 1] + (size_t)(L - 1) * B * ul;
        {
            DenseArgs d{};
            d.g = g; d.u = ul; d.T_out = p.T_out; d.act = p.out_act;
            d.params = params; d.n_params = p.n_params; d.w_off = p.dense_w_off; d.b_off = p.dense_b_off;
            d.h = h_last; d.h_seq_stride = ul; d.h_grp_stride = gs;
            d.out_local = S + yh_o; d.ol_seq_stride = p.T_out; d.ol_grp_stride = gs;
            lstm_dense_out_kernel<<<dim3(cdiv(cap * p.T_out, 256), 1, J), 256, 0, stream>>>(d);
            LossArgs la{};
            la.g = g; la.u = ul; la.T_out = p.T_out; la.act = p.out_act; la.L = L; la.lookahead = p.lookahead;
            la.params = params; la.n_params = p.n_params; la.y = ysrc;
            la.yhat = S + yh_o; la.yh_seq_stride = p.T_out; la.yh_grp_stride = gs;
            la.dzd = S + dzd_o; la.dzd_grp_stride = gs; la.loss_sum = d_loss;
            lstm_loss_kernel<<<dim3(cdiv(cap * p.T_out, 256), 1, J), 256, 0, stream>>>(la);
        }
        // ---------------- backward: dense
        {
            // grad Wd[k][n] = sum_s h_last[s][k] * dzd[s][n]; grad bd[n] = sum_s dzd[s][n]  (L = 1 "time step")
            WgradArgs w{};
            w.g = g; w.Kdim = ul; w.N = p.T_out; w.L = 1; w.layer = 1; w.shift = 0;
            w.aseq = h_last; w.a_t_stride = 0; w.a_seq_stride = ul; w.a_grp_stride = gs;
            w.dz = S + dzd_o; w.dz_t_stride = 0; w.dz_seq_stride = p.T_out; w.dz_grp_stride = gs;
            w.grad = S + grad_o; w.grad_grp_stride = gs; w.grad_off = p.dense_w_off;
            w.gbias = S + grad_o; w.gbias_off = p.dense_b_off;
            lstm_wgrad_kernel<<<dim3(cdiv(ul * p.T_out + p.T_out, 256), 1, J), 256, 0, stream>>>(w);
            // dH of the last layer: zero everywhere except t = L-1 where it is dzd . Wd^T
            GB_CUDA_CHECK(cudaGetLastError());
            NTArgs n{};
            n.g = g; n.N = p.T_out; n.Kout = ul;
            n.A = S + dzd_o; n.a_seq_stride = p.T_out; n.a_grp_stride = gs;
            n.B = params + p.dense_w_off; n.b_row_stride = p.T_out; n.b_grp_stride = p.n_params;
            n.out = S + dH_o[p.n_layers - 1] + (size_t)(L - 1) * B * ul; n.o_seq_stride = ul; n.o_grp_stride = gs;
            lstm_nt_kernel<<<dim3(cdiv(cap * ul * 32, 256), 1, J), 256, 0, stream>>>(n);
        }
        // ---------------- backward: BPTT, top layer first.  Per time step only the recurrence
        // (gate derivatives, dh_rec = dz.U^T); dLoss/dx and the weight gradients are one GEMM per layer
        for (int l = p.n_layers - 1; l >= 0; --l) {
            const int u = p.ld[l].u, in = p.ld[l].in;
            const bool top = (l == p.n_layers - 1);
            const RecPlan rp = make_rec_plan(u, B);
            if (rp.ok && use_rec) {
                RecArgs ra{};
                ra.g = g; ra.B = B; ra.L = L; ra.u = u; ra.act = p.acts[l]; ra.top = top ? 1 : 0;
                ra.params = params; ra.n_params = p.n_params; ra.u_off = p.ld[l].u_off;
                ra.gates = S + gt_o[l]; ra.hs = S + hs_o[l]; ra.cs = S + cs_o[l]; ra.ac = S + ac_o[l]; ra.gs = gs;
                ra.dH = S + dH_o[l]; ra.dz = S + dz_o[l];
                rc = launch_rec(false, rp, ra, J, stream);
                if (rc) return rc;
            }
            for (int t = L - 1; t >= 0 && !(rp.ok && use_rec); --t) {
                BwdGateArgs b{};
                b.g = g; b.u = u; b.act = p.acts[l]; b.t = t; b.L = L;
                // the top layer only receives a gradient at t = L-1 (return_sequences=False)
                b.dh_above = (!top || t == L - 1) ? S + dH_o[l] + (size_t)t * B * u : nullptr; b.da_seq_stride = u; b.da_grp_stride = gs;
                b.dh_rec = t < L - 1 ? S + dr_o[l] : nullptr; b.dr_seq_stride = u; b.dr_grp_stride = gs;
                b.dc = S + dc_o[l]; b.dc_seq_stride = u; b.dc_grp_stride = gs;
                b.gates = S + gt_o[l] + (size_t)t * B * 4 * u; b.g_seq_stride = 4 * u; b.g_grp_stride = gs;
                b.actc = S + ac_o[l] + (size_t)t * B * u; b.ac_seq_stride = u; b.ac_grp_stride = gs;
                b.c_t = S + cs_o[l] + (size_t)t * B * u; b.ct_seq_stride = u; b.ct_grp_stride = gs;
                b.c_prev = t > 0 ? S + cs_o[l] + (size_t)(t - 1) * B * u : nullptr; b.cp_seq_stride = u; b.cp_grp_stride = gs;
                b.dz = S + dz_o[l] + (size_t)t * B * 4 * u; b.dz_seq_stride = 4 * u; b.dz_grp_stride = gs;
                lstm_bwd_gates_kernel<<<dim3(cdiv(cap * u, 256), 1, J), 256, 0, stream>>>(b);
                if (t > 0) {    // dh_rec[seq][j] = sum_n dz_t[seq][n] * U[j][n]  (needed by t-1): one warp per output
                    NTArgs n{};
                    n.g = g; n.N = 4 * u; n.Kout = u;
                    n.A = b.dz; n.a_seq_stride = 4 * u; n.a_grp_stride = gs;
                    n.B = params + p.ld[l].u_off; n.b_row_stride = 4 * u; n.b_grp_stride = p.n_params;
                    n.out = S + dr_o[l]; n.o_seq_stride = u; n.o_grp_stride = gs;
                    lstm_nt_kernel<<<dim3(cdiv(cap * u * 32, 256), 1, J), 256, 0, stream>>>(n);
                }
            }
            const float* Ain = l == 0 ? S + x0_o : S + hs_o[l - 1];
            if (l > 0)          // dLoss/dh of the layer below, all t: dz . W^T
                gemm(0, L * B, in, 4 * u, S + dz_o[l], gs, 4 * u, 1, params + p.ld[l].w_off, p.n_params, 4 * u, 1,
                     S + dH_o[l - 1], gs, in, nullptr, 0);
            // weight gradients: reductions over (t, seq) as GEMMs with the composite dimension as K
            gemm(1, in, 4 * u, L * B, Ain, gs, in, 0, S + dz_o[l], gs, 4 * u, 0,
                 S + grad_o + p.ld[l].w_off, gs, 4 * u, nullptr, 0);
            if (L > 1)
                gemm(1, u, 4 * u, (L - 1) * B, S + hs_o[l], gs, u, 0, S + dz_o[l] + (size_t)B * 4 * u, gs, 4 * u, 0,
                     S + grad_o + p.ld[l].u_off, gs, 4 * u, nullptr, 0);
            else        // lookback 1: no recurrent step, no gradient
                for (int j = 0; j < J; ++j)
                    GB_CUDA_CHECK(cudaMemsetAsync(S + (size_t)j * per_job + grad_o + p.ld[l].u_off, 0,
                                                  sizeof(float) * (size_t)u * 4 * u, stream));
            lstm_colsum_kernel<<<dim3(cdiv(4 * u, 32), 1, J), 256, 0, stream>>>(g, B, L * B, 4 * u, S + dz_o[l], gs,
                                                                               S + grad_o, gs, p.ld[l].b_off);
        }
        // ---------------- Adam
        AdamArgs ad{};
        ad.g = g; ad.adam = *adam; ad.n_params = p.n_params; ad.params = params;
        ad.grad = S + grad_o; ad.mv = S + mv_o; ad.tcount = d_tcount;
        // grad and mv live inside the per-job scratch: strides differ from n_params, so fix the bases
        // (kernel indexes grad + grp*n_params): launch per job instead
        for (int j = 0; j < J; ++j) {
            AdamArgs aj = ad;
            aj.g.rows_lo = d_rows_cur + j; aj.g.n_win = d_nwin_cur + j;      // the cursor: a finished job takes no step
            aj.params = params + (size_t)j * p.n_params; aj.grad = S + (size_t)j * per_job + grad_o;
            aj.mv = S + (size_t)j * per_job + mv_o; aj.tcount = d_tcount + j;
            int blocks = cdiv((int)((p.n_params + 255) / 256), 1); if (blocks > 148 * 4) blocks = 148 * 4;
            lstm_adam_kernel<<<dim3(blocks, 1, 1), 256, 0, stream>>>(aj);
        }
        lstm_step_end_kernel<<<cdiv(J, 128), 128, 0, stream>>>(g, J, d_tcount, d_loss, d_epoch, p.T_out, primer_out,
                                                              advance, d_rows_cur, d_nwin_cur);
        GB_CUDA_CHECK(cudaGetLastError());
        return GB_OK;
    };
    auto rewind = [&]() -> int {
        GB_CUDA_CHECK(cudaMemcpyAsync(d_rows_cur, d_rows_lo, sizeof(int64_t) * J, cudaMemcpyDeviceToDevice, stream));
        GB_CUDA_CHECK(cudaMemcpyAsync(d_nwin_cur, d_nwin, sizeof(int32_t) * J, cudaMemcpyDeviceToDevice, stream));
        return GB_OK;
    };

    // (1) primer: ONE Adam step on the first window alone (models.py:585-597)
    rc = rewind(); if (rc) return rc;
    rc = run_step(1, primer_loss ? primer_loss : d_epoch + 0 /*unused sink*/, 0);
    if (rc) return rc;
    if (!primer_loss) GB_CUDA_CHECK(cudaMemsetAsync(d_epoch, 0, sizeof(float) * J, stream));
    // (2) main fit: time-ordered batches, shuffle=False (models.py:599-615).  Every job runs the same number of steps,
    // enough for the job with the most windows; the device cursor stops the others once their windows run out.
    const int n_steps = (max_win + B - 1) / B;
    for (int e = 0; e < epochs; ++e) {
        rc = rewind(); if (rc) return rc;
        for (int s = 0; s < n_steps; ++s) {
            rc = run_step(B, nullptr, B);
            if (rc) return rc;
        }
        if (hist_loss) lstm_epoch_end_kernel<<<cdiv(J, 128), 128, 0, stream>>>(J, d_nwin, d_epoch, hist_loss, epochs, e);
        else GB_CUDA_CHECK(cudaMemsetAsync(d_epoch, 0, sizeof(float) * J, stream));
    }
    GB_CUDA_CHECK(cudaGetLastError());
    return GB_OK;
}

}  // extern "C"
