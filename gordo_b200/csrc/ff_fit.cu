// ff_fit: Keras Model.fit for many independent small autoencoders, one CTA per fit job.
//
// Replaces models.py:243-287 -> scikeras -> [3P] keras Model.fit (SURVEY.md §8 a3): float32
// mini-batch SGD with Keras-form Adam, loss = MSE + L1 activity terms, History loss/accuracy.
// The optimizer steps of one job are strictly sequential (ceil(N/batch) dependent steps per
// epoch), so parallelism comes from jobs: a CTA keeps its job's weights and both Adam moments in
// shared memory for the whole fit (T=50 hourglass: 3 x 9 497 x 4 B = 114 KB) and walks the
// mini-batches; CV folds and the final fit of every Machine are separate jobs of one launch.
//
// Per step (phases separated by __syncthreads):
//   gather  : h0[k][b] = x[row_b][k]*scale+min            (rows given by the permutation)
//   forward : h_{l+1}[n][b] = act(b_l[n] + sum_k h_l[k][b] W_l[k][n])
//   loss    : D_L[b][n] = dLoss/dz_L, MSE / accuracy / L1 sums
//   deltas  : l = L-1..1:  D_l = (D_{l+1} . W_l^T + l1 sign(h_l)) act'(h_l)     (every D_l kept)
//   update  : one barrier-free sweep over all layers: g = sum_b h_l[k][b] D_{l+1}[n][b] -> Adam update of W_l[k][n], b_l[n]
// Layouts: h and D feature-major [w][Bs], Bs a multiple of 4: a thread owns 4 consecutive samples of
// one feature (forward, backward A) or one weight (backward B), reads activations / deltas as 16-byte
// words along the batch and a weight once per 4 FMAs; samples past the batch end carry zero deltas.
#include "common.cuh"

namespace {

constexpr int FIT_THREADS = 512;

struct FitArgs {
    gb200_ff_arch arch;
    gb200_adam adam;
    const int64_t* lo; const int64_t* hi; const int32_t* scale_slot;
    const float* in_scale; const float* in_min;
    const float* x; const float* y;
    const int64_t* perm_off; const int32_t* perm_pool;
    int epochs, batch, l1_mean;
    float* params; float* adam_mv; int64_t* adam_t;
    float* hist_loss; float* hist_acc;
    int64_t n_params;
    int state_in_smem;      // 2: W,m,v in smem  1: W in smem  0: all global
    int h_floats;           // sum_l w_l * Bs
    int Bs;                 // sample stride of h and D (multiple of 4: 16-byte reads along the batch)
    int Bq;                 // 4-sample groups per batch
    const int32_t* order;   // CTA -> job, longest job first
    float* scratch;         // HG: per-job activations + deltas in global memory (2 * h_floats floats each)
};

// Jobs differ in length (CV folds of 1/4, 2/4, 3/4 of the rows next to full final fits) and CTAs are
// dispatched in index order: hand out the longest jobs first so the last wave is made of short ones.
__global__ void fit_order_kernel(int n_jobs, const int64_t* __restrict__ lo, const int64_t* __restrict__ hi,
                                 int32_t* __restrict__ order) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_jobs) return;
    const int64_t mine = hi[j] - lo[j];
    int rank = 0;
    for (int i = 0; i < n_jobs; ++i) {
        const int64_t other = hi[i] - lo[i];
        rank += (other > mine) || (other == mine && i < j);
    }
    order[rank] = j;
}

// act' from the OUTPUT h alone (tanh 1-h^2, sigmoid h(1-h), relu/elu via sign of h,
// softplus sigma(z) = 1 - exp(-h))
__device__ __forceinline__ float act_grad_from_h(int code, float h) {
    switch (code) {
        case GB200_ACT_TANH:     return 1.0f - h * h;
        case GB200_ACT_RELU:     return h > 0.0f ? 1.0f : 0.0f;
        case GB200_ACT_SIGMOID:  return h * (1.0f - h);
        case GB200_ACT_ELU:      return h > 0.0f ? 1.0f : h + 1.0f;
        case GB200_ACT_SOFTPLUS: return 1.0f - expf(-h);
        default:                 return 1.0f;
    }
}

__device__ __forceinline__ float block_sum(float v, float* red) {
    #pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = 0.0f;
    #pragma unroll
    for (int i = 0; i < FIT_THREADS / 32; ++i) s += red[i];
    return s;
}

// STATE: where W / Adam m, v live (2: all in shared memory, 1: W only, 0: global).  A template
// parameter so that the compiler knows the address space: plain LDS/STS with 32-bit addressing
// instead of generic loads in every inner loop.
// BQ: 4-sample groups per batch when known at compile time (8 = Keras' default batch of 32), else 0.
// HG: the batch's activations and deltas do not fit in shared memory next to nothing else (wide default
// topologies such as 256-128-64, or batch_size 128 with > 60 tags): they live in a per-job global scratch
// (L1/L2 resident: a few hundred KB) and shared memory only holds W when that fits.  Same arithmetic,
// same order of operations; __syncthreads() orders the global accesses of the block as it does the shared ones.
template <int STATE, int BQ, bool HG = false>
__global__ void __launch_bounds__(FIT_THREADS, 1)
ff_fit_kernel(const __grid_constant__ FitArgs a) {
    extern __shared__ __align__(16) float smem[];
    __shared__ float red[FIT_THREADS / 32];
    __shared__ int s_argmax_hits;

    const int job = a.order ? a.order[blockIdx.x] : blockIdx.x, tid = threadIdx.x;
    const int L = a.arch.n_layers;
    const int T_in = a.arch.widths[0], T_out = a.arch.widths[L];
    const int B = a.batch;
    const int Bq = BQ ? BQ : a.Bq, Bs = BQ ? 4 * BQ + 4 : a.Bs;
    const int64_t P = a.n_params;

    float* hbuf = HG ? a.scratch + (size_t)job * 2 * a.h_floats : smem;      // all layer activations of the batch
    float* Dall = hbuf + a.h_floats;                  // dLoss/dz of every layer, laid out like hbuf
    float* st = HG ? smem : Dall + a.h_floats;        // optional on-chip W / m / v
    float* gW = a.params + (size_t)job * P;
    float* gM = a.adam_mv + (size_t)job * 2 * P;
    float* gV = gM + P;
    float* W = STATE >= 1 ? st : gW;
    float* Mo = STATE >= 2 ? st + P : gM;
    float* Vo = STATE >= 2 ? st + 2 * P : gV;
    if (STATE >= 1) for (int64_t i = tid; i < P; i += FIT_THREADS) W[i] = gW[i];
    if (STATE >= 2) for (int64_t i = tid; i < P; i += FIT_THREADS) { Mo[i] = gM[i]; Vo[i] = gV[i]; }

    const int64_t r_lo = a.lo[job];
    const int n = (int)(a.hi[job] - r_lo);
    const int slot = a.scale_slot ? a.scale_slot[job] : job;
    const float* sc = a.in_scale ? a.in_scale + (size_t)slot * T_in : nullptr;
    const float* mn = a.in_min ? a.in_min + (size_t)slot * T_in : nullptr;
    const float* ysrc = a.y ? a.y : a.x;
    const int32_t* perm = a.perm_pool ? a.perm_pool + a.perm_off[job] : nullptr;
    int64_t t = a.adam_t ? a.adam_t[job] : 0;
    const float b1 = a.adam.beta_1, b2 = a.adam.beta_2, eps = a.adam.epsilon, lr = a.adam.lr;
    __syncthreads();

    for (int e = 0; e < a.epochs; ++e) {
        double loss_acc = 0.0; int hits_acc = 0;          // meaningful in thread 0 only
        for (int s0 = 0; s0 < n; s0 += B) {
            const int nb = min(B, n - s0);
            // ---- gather + MinMax scale
            for (int i = tid; i < nb * T_in; i += FIT_THREADS) {
                const int b = i / T_in, k = i - b * T_in;
                const int64_t r = r_lo + (perm ? perm[(int64_t)e * n + s0 + b] : s0 + b);
                float v = a.x[r * T_in + k];
                if (sc) v = fmaf(v, sc[k], mn[k]);
                hbuf[k * Bs + b] = v;
            }
            // samples past the end of a short batch: zero inputs keep every activation finite
            for (int i = tid; i < (4 * Bq - nb) * T_in; i += FIT_THREADS) {
                const int b = nb + i / T_in, k = i % T_in;
                hbuf[k * Bs + b] = 0.0f;
            }
            if (tid == 0) s_argmax_hits = 0;
            __syncthreads();
            // ---- forward: a thread owns one output feature for 4 consecutive samples, so a weight is
            // read once per 4 FMAs and the activations come as one 16-byte read
            float l1_sum = 0.0f;
            {
                int ho = 0; int po = 0;
                for (int l = 0; l < L; ++l) {
                    const int win = a.arch.widths[l], wout = a.arch.widths[l + 1];
                    const int code = a.arch.acts[l];
                    const float* Wl = W + po; const float* bl = Wl + win * wout;
                    const float* hin = hbuf + ho; float* hout = hbuf + ho + win * Bs;
                    const float c1 = a.arch.l1[l];
                    for (int i = tid; i < wout * Bq; i += FIT_THREADS) {
                        const int nn = i / Bq, b4 = (i - nn * Bq) * 4;
                        const float bias = bl[nn];
                        float a0 = bias, a1 = bias, a2 = bias, a3 = bias;
                        const float* wp = Wl + nn; const float* hp = hin + b4;
                        #pragma unroll 4
                        for (int k = 0; k < win; ++k, wp += wout, hp += Bs) {
                            const float w = *wp;
                            const float4 h4 = *reinterpret_cast<const float4*>(hp);
                            a0 = fmaf(h4.x, w, a0); a1 = fmaf(h4.y, w, a1); a2 = fmaf(h4.z, w, a2); a3 = fmaf(h4.w, w, a3);
                        }
                        float4 o;
                        o.x = gb_act(code, a0); o.y = gb_act(code, a1); o.z = gb_act(code, a2); o.w = gb_act(code, a3);
                        *reinterpret_cast<float4*>(hout + nn * Bs + b4) = o;
                        if (c1 != 0.0f) {
                            if (b4 < nb) l1_sum += c1 * fabsf(o.x);
                            if (b4 + 1 < nb) l1_sum += c1 * fabsf(o.y);
                            if (b4 + 2 < nb) l1_sum += c1 * fabsf(o.z);
                            if (b4 + 3 < nb) l1_sum += c1 * fabsf(o.w);
                        }
                    }
                    ho += win * Bs; po += win * wout + wout;
                    __syncthreads();
                }
            }
            // ---- loss, dLoss/dz_L, accuracy
            int hoffs[GB200_MAX_LAYERS + 1]; int poffs[GB200_MAX_LAYERS];
            {
                int ho = 0, po = 0;
                for (int l = 0; l < L; ++l) {
                    hoffs[l] = ho; poffs[l] = po;
                    ho += a.arch.widths[l] * Bs; po += a.arch.widths[l] * a.arch.widths[l + 1] + a.arch.widths[l + 1];
                }
                hoffs[L] = ho;
            }
            const float* hL = hbuf + hoffs[L];
            float* DL = Dall + hoffs[L];
            float sq = 0.0f;
            {
                const float inv = 2.0f / (float)(nb * T_out);
                const int code = a.arch.acts[L - 1];
                const float cL = a.arch.l1[L - 1] * (a.l1_mean ? 1.0f / (float)nb : 1.0f);
                // D is feature-major like h ([n][Bs]); samples past nb carry zeros so that the
                // batch reductions below can run over whole 4-sample groups
                for (int i = tid; i < 4 * Bq * T_out; i += FIT_THREADS) {
                    const int b = i / T_out, nn = i - b * T_out;
                    float dv = 0.0f;
                    if (b < nb) {
                        const int64_t r = r_lo + (perm ? perm[(int64_t)e * n + s0 + b] : s0 + b);
                        const float yh = hL[nn * Bs + b];
                        const float diff = yh - ysrc[r * T_out + nn];
                        sq = fmaf(diff, diff, sq);
                        float dh = inv * diff;
                        if (cL != 0.0f) dh += cL * (yh > 0.0f ? 1.0f : (yh < 0.0f ? -1.0f : 0.0f));
                        dv = dh * act_grad_from_h(code, yh);
                    }
                    DL[nn * Bs + b] = dv;
                }
                if (a.hist_acc) {
                    // Keras 'accuracy' on a float [B,T] target = categorical accuracy; binary at T_out == 1
                    for (int b = tid; b < nb; b += FIT_THREADS) {
                        const int64_t r = r_lo + (perm ? perm[(int64_t)e * n + s0 + b] : s0 + b);
                        int hit;
                        if (T_out == 1) {
                            hit = ((hL[b] > 0.5f ? 1.0f : 0.0f) == ysrc[r]) ? 1 : 0;
                        } else {
                            int ay = 0, ap = 0; float by = ysrc[r * T_out], bp = hL[b];
                            for (int j = 1; j < T_out; ++j) {
                                const float vy = ysrc[r * T_out + j], vp = hL[j * Bs + b];
                                if (vy > by) { by = vy; ay = j; }
                                if (vp > bp) { bp = vp; ap = j; }
                            }
                            hit = ay == ap;
                        }
                        if (hit) atomicAdd(&s_argmax_hits, 1);
                    }
                }
            }
            if (a.hist_loss) {
                const float tot_sq = block_sum(sq, red);
                const float tot_l1 = block_sum(l1_sum, red);
                if (tid == 0) {
                    const float batch_loss = tot_sq / (float)(nb * T_out) + (a.l1_mean ? tot_l1 / (float)nb : tot_l1);
                    loss_acc += (double)batch_loss * nb;
                    hits_acc += s_argmax_hits;
                }
            } else {
                __syncthreads();
            }
            // ---- Adam step size (Keras: alpha = lr*sqrt(1-b2^t)/(1-b1^t), eps outside)
            t += 1;
            const float tf = (float)t;
            const float alpha = lr * sqrtf(1.0f - powf(b2, tf)) / (1.0f - powf(b1, tf));
            const float l1_scale = a.l1_mean ? 1.0f / (float)nb : 1.0f;
            // ---- backward, deltas first: D_l = (D_{l+1} . W_l^T + l1 sign(h_l)) act'(h_l) for l = L-1 .. 1,
            // every delta kept (one slot per activation) and every W still the forward pass's
            for (int l = L - 1; l >= 1; --l) {
                const int win = a.arch.widths[l], wout = a.arch.widths[l + 1];
                const float* Wl = W + poffs[l];
                const float* hin = hbuf + hoffs[l];
                const float* Dcur = Dall + hoffs[l + 1];
                float* Dnext = Dall + hoffs[l];
                const int pcode = a.arch.acts[l - 1];
                const float c1 = a.arch.l1[l - 1] * l1_scale;
                for (int i = tid; i < win * Bq; i += FIT_THREADS) {
                    const int k = i / Bq, b4 = (i - k * Bq) * 4;
                    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
                    const float* wp = Wl + k * wout; const float* dq = Dcur + b4;
                    #pragma unroll 4
                    for (int nn = 0; nn < wout; ++nn, ++wp, dq += Bs) {
                        const float w = *wp;
                        const float4 d4 = *reinterpret_cast<const float4*>(dq);
                        a0 = fmaf(d4.x, w, a0); a1 = fmaf(d4.y, w, a1); a2 = fmaf(d4.z, w, a2); a3 = fmaf(d4.w, w, a3);
                    }
                    const float4 h4 = *reinterpret_cast<const float4*>(hin + k * Bs + b4);
                    const float hv[4] = {h4.x, h4.y, h4.z, h4.w};
                    float av[4] = {a0, a1, a2, a3};
                    #pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float acc = av[q];
                        if (c1 != 0.0f) acc += c1 * (hv[q] > 0.0f ? 1.0f : (hv[q] < 0.0f ? -1.0f : 0.0f));
                        av[q] = b4 + q < nb ? acc * act_grad_from_h(pcode, hv[q]) : 0.0f;
                    }
                    *reinterpret_cast<float4*>(Dnext + k * Bs + b4) = make_float4(av[0], av[1], av[2], av[3]);
                }
                __syncthreads();
            }
            // ---- then ONE sweep over all weights of all layers: gradient (sum over the batch, 4 samples per
            // 16-byte read) and Adam update in place.  No barrier between layers: nothing read here is written here.
            for (int l = 0; l < L; ++l) {
                const int win = a.arch.widths[l], wout = a.arch.widths[l + 1];
                float* Wl = W + poffs[l];
                const float* hin = hbuf + hoffs[l];
                const float* Dcur = Dall + hoffs[l + 1];
                const int n_w = win * wout;
                auto adam_update = [&](int i, float g) {
                    const int p = poffs[l] + i;
                    float m = Mo[p], v = Vo[p];
                    m += (g - m) * (1.0f - b1);
                    v += (g * g - v) * (1.0f - b2);
                    Mo[p] = m; Vo[p] = v;
                    Wl[i] -= alpha * m / (sqrtf(v) + eps);
                };
                {
                    // weight (k, nn) of item i, advanced without a division per item
                    int k = tid / wout, nn = tid - k * wout;
                    const int dk = FIT_THREADS / wout, dn = FIT_THREADS - dk * wout;
                    for (int i = tid; i < n_w; i += FIT_THREADS) {
                        const float4* hp = reinterpret_cast<const float4*>(hin + k * Bs);
                        const float4* dp = reinterpret_cast<const float4*>(Dcur + nn * Bs);
                        float g = 0.0f;
            #define GB_FIT_DOT4(q) { const float4 h4 = hp[q], d4 = dp[q]; \
                g = fmaf(h4.x, d4.x, g); g = fmaf(h4.y, d4.y, g); g = fmaf(h4.z, d4.z, g); g = fmaf(h4.w, d4.w, g); }
                        if constexpr (BQ > 0) {
                            #pragma unroll
                            for (int q = 0; q < BQ; ++q) GB_FIT_DOT4(q)
                        } else {
                            for (int q = 0; q < Bq; ++q) GB_FIT_DOT4(q)
                        }
            #undef GB_FIT_DOT4
                        adam_update(i, g);
                        nn += dn; k += dk;
                        if (nn >= wout) { nn -= wout; ++k; }
                    }
                }
                for (int nn = tid; nn < wout; nn += FIT_THREADS) {
                    const float4* dp = reinterpret_cast<const float4*>(Dcur + nn * Bs);
                    float g = 0.0f;
                    for (int q = 0; q < Bq; ++q) { const float4 d4 = dp[q]; g += d4.x; g += d4.y; g += d4.z; g += d4.w; }
                    adam_update(n_w + nn, g);
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            if (a.hist_loss) a.hist_loss[(size_t)job * a.epochs + e] = n > 0 ? (float)(loss_acc / n) : NAN;
            if (a.hist_acc) a.hist_acc[(size_t)job * a.epochs + e] = n > 0 ? (float)hits_acc / (float)n : NAN;
        }
    }
    __syncthreads();
    if (STATE >= 1) for (int64_t i = tid; i < P; i += FIT_THREADS) gW[i] = W[i];
    if (STATE >= 2) for (int64_t i = tid; i < P; i += FIT_THREADS) { gM[i] = Mo[i]; gV[i] = Vo[i]; }
    if (tid == 0 && a.adam_t) a.adam_t[job] = t;
}

}  // namespace

int gb_launch_ff_fit(const gb200_ff_arch* arch, const gb200_adam* adam, int n_jobs,
                     const int64_t* lo, const int64_t* hi, const int32_t* scale_slot,
                     const float* in_scale, const float* in_min, const float* x, const float* y,
                     const int64_t* perm_off, const int32_t* perm_pool, int epochs, int batch_size,
                     int l1_mean, float* params, float* adam_mv, int64_t* adam_t, float* hist_loss,
                     float* hist_acc, cudaStream_t stream) {
    if (n_jobs <= 0) return GB_OK;
    FitArgs a{};
    a.arch = *arch; a.adam = *adam;
    a.lo = lo; a.hi = hi; a.scale_slot = scale_slot; a.in_scale = in_scale; a.in_min = in_min;
    a.x = x; a.y = y; a.perm_off = perm_off; a.perm_pool = perm_pool;
    a.epochs = epochs; a.batch = batch_size; a.l1_mean = l1_mean;
    a.params = params; a.adam_mv = adam_mv; a.adam_t = adam_t; a.hist_loss = hist_loss; a.hist_acc = hist_acc;
    a.n_params = gb200_ff_param_count(arch);
    int sum_w = 0;
    for (int l = 0; l <= arch->n_layers; ++l) sum_w += arch->widths[l];
    a.Bq = (batch_size + 3) / 4;
    a.Bs = 4 * a.Bq + 4;            // 16-byte rows; +4 keeps the 8 row groups of a warp on distinct banks
    a.h_floats = sum_w * a.Bs;
    const size_t cap = 227 * 1024 - 256;
    GB_REQUIRE(a.n_params < (1ll << 30), "ff_fit: topology too large");
    int32_t* order = nullptr;
    if (n_jobs > 1) {
        GB_CUDA_CHECK(cudaMallocAsync(&order, sizeof(int32_t) * n_jobs, stream));
        fit_order_kernel<<<(n_jobs + 127) / 128, 128, 0, stream>>>(n_jobs, lo, hi, order);
    }
    a.order = order;
    size_t base = 2 * (size_t)a.h_floats * sizeof(float);      // activations + one delta slot per activation
    const bool hg = base > cap;         // the batch's activations go to a global scratch (see the HG note)
    float* scratch = nullptr;
    if (hg) {
        GB_REQUIRE((size_t)n_jobs * base < (64ull << 30), "ff_fit: batch_size %d x widths need too much scratch", batch_size);
        GB_CUDA_CHECK(cudaMallocAsync(&scratch, (size_t)n_jobs * base, stream));
        base = 0;
    }
    a.scratch = scratch;
    const size_t pbytes = (size_t)a.n_params * sizeof(float);
    a.state_in_smem = base + 3 * pbytes <= cap ? 2 : (base + pbytes <= cap ? 1 : 0);
    const size_t smem = base + (a.state_in_smem == 2 ? 3 * pbytes : a.state_in_smem == 1 ? pbytes : 0);
    auto* kern = hg ? (a.state_in_smem == 2 ? ff_fit_kernel<2, 0, true> : a.state_in_smem == 1 ? ff_fit_kernel<1, 0, true>
                                                                                                 : ff_fit_kernel<0, 0, true>)
               : a.state_in_smem == 2 ? (a.Bq == 8 ? ff_fit_kernel<2, 8> : ff_fit_kernel<2, 0>)
               : a.state_in_smem == 1 ? ff_fit_kernel<1, 0> : ff_fit_kernel<0, 0>;
    GB_CUDA_CHECK(gb_allow_max_smem(kern));
    kern<<<n_jobs, FIT_THREADS, smem, stream>>>(a);
    cudaError_t le = cudaGetLastError();
    if (order) cudaFreeAsync(order, stream);
    if (scratch) cudaFreeAsync(scratch, stream);
    GB_CUDA_CHECK(le);
    return GB_OK;
}
