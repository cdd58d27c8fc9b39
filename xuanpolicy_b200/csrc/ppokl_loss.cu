// ppokl_loss.cu — the PPO-KL minibatch loss of the native update on the packed minibatch rows, forward + backward w.r.t.
// the network outputs in one launch, with the adaptive KL coefficient (ppokl_learner.py:21-61).
//
//     L = -mean(ratio * adv) + kl_coef * mean KL(new || old) - ent_coef * mean H + vf_coef * mean (v - R)^2
//     ratio = exp(log_prob(act) - old_dist.log_prob(act))
// for the two heads the packed 32-byte records serve: 2 logits (CartPole-v1) or one Gaussian dimension with a shared
// log-std (Pendulum-v1).  Closed forms as in dist_loss.cu (which keeps the general shapes).
//
// Inputs per sample: the gathered {act, old_logp, adv, ret} float4 of xb_gather_records, the forward's head outputs and v,
// and the old-distribution pair {z0, z1} / {mu, std} read straight from the rollout's [T][N][2] array at the sample's
// buffer row (one 8-byte load: the 32-byte record stays the one layout every PPO gather kernel reads).  The old log-prob
// is taken from that pair, like the reference's `old_dist.log_prob(act)`; the record's lane is not read.
// HBM bytes per sample (Categorical): 8 index + 16 scalars + 8 old pair + 8 logits + 4 v read, 8 dlogits + 4 dv written.
//
// Reductions: warp shuffle -> per-CTA partials -> the last CTA (ticket) adds them in CTA order: deterministic, nothing to
// zero beforehand.  The same CTA, once every CTA has read the coefficient, records it (kl_used) and, given `adapt`,
// adapts it from this launch's KL (x2 above 1.5 target, /2 below 0.5 target, clip [0.1, 20]): the next update reads the
// new value, this one used the old.  Env-sharded, the KL that drives the decision is the global one: the launch writes its
// KL sum to kl_sum_out and xb_ppokl_kl_adapt follows the exchange.
#include "common.cuh"

namespace xb {

constexpr int kKlBlock = 256;
constexpr int kKlMaxGrid = kNumSMs * 8;
constexpr int kKlSlots = 7;   // {surrogate, (v-R)^2, entropy, v, -, KL, dL/dlogstd}
constexpr float kKlHalfLog2Pi = 0.9189385332046727f;

__device__ double g_kl_partials[kKlMaxGrid * kKlSlots];
__device__ unsigned int g_kl_ticket;

struct PpoklArgs {
    const int64_t* idx;
    int64_t B, T, N;
    const float4* scal;
    const float2* old_dist;
    const float* act_out;
    const float* logstd;
    const float* v_pred;
    const double* adv_stats;
    double inv_adv_count;
    float vf_coef, ent_coef, inv_batch;
    float* kl_coef;
    float* kl_used;
    float target_kl;
    int adapt;
    double inv_kl_count;
    double* kl_sum_out;
    float* dact;
    float* dv;
    double* dlogstd;
    double* scalars;
};

__device__ __forceinline__ void kl_adapt_store(float* kl_coef, float* kl_used, double kl_sum, double inv_count,
                                               float target_kl) {
    const float k0 = *kl_coef;
    if (kl_used) *kl_used = k0;
    const float kl = (float)(kl_sum * inv_count);
    float k = k0;
    if (kl > target_kl * 1.5f)
        k = k * 2.0f;
    else if (kl < target_kl * 0.5f)
        k = k / 2.0f;
    *kl_coef = fminf(fmaxf(k, 0.1f), 20.0f);
}

template <bool GAUSS>
__global__ void __launch_bounds__(kKlBlock) ppokl_loss_packed_kernel(PpoklArgs c) {
    __shared__ double smem[kKlSlots * 32];
    __shared__ bool is_last;
    float nmean = 0.0f, ndenom = 1.0f;
    if (c.adv_stats) {      // the advantage normalisation of the PPO-Clip loss kernels (ppo_loss.cu load_adv_norm)
        const double mean = c.adv_stats[0] * c.inv_adv_count;
        const double var = c.adv_stats[1] * c.inv_adv_count - mean * mean;
        nmean = (float)mean;
        ndenom = (float)sqrt(var > 0.0 ? var : 0.0) + 1e-8f;
    }
    const float kl_w = *c.kl_coef * c.inv_batch;   // (A = 1 for the Gaussian head: the mean over B*A is over B)
    const float ge = c.ent_coef * c.inv_batch;
    float ls = 0.0f, sd = 1.0f, inv_var = 1.0f, Hg = 0.0f;
    if (GAUSS) {
        ls = c.logstd[0];
        sd = expf(ls);
        inv_var = 1.0f / (sd * sd);
        Hg = 0.5f + kKlHalfLog2Pi + ls;
    }
    double acc[kKlSlots] = {0, 0, 0, 0, 0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < c.B; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = c.idx[i];
        const int64_t env = k / c.T;
        const int64_t row = (k - env * c.T) * c.N + env;
        const float4 sc = __ldg(c.scal + i);
        const float2 od = __ldg(c.old_dist + row);
        float adv = sc.z;
        if (c.adv_stats) adv = (adv - nmean) / ndenom;
        float logp, old_logp, H, KL;
        float g0 = 0.0f, g1 = 0.0f, gls = 0.0f;
        if (!GAUSS) {
            const float2 z = __ldg(reinterpret_cast<const float2*>(c.act_out) + i);
            const int a = (int)sc.x;
            const float zmax = fmaxf(z.x, z.y), omax = fmaxf(od.x, od.y);
            const float lse = zmax + logf(expf(z.x - zmax) + expf(z.y - zmax));
            const float lso = omax + logf(expf(od.x - omax) + expf(od.y - omax));
            const float lp0 = z.x - lse, lp1 = z.y - lse, lq0 = od.x - lso, lq1 = od.y - lso;
            const float p0 = expf(lp0), p1 = expf(lp1);
            H = -(p0 * lp0) - p1 * lp1;
            KL = p0 * (lp0 - lq0) + p1 * (lp1 - lq1);
            logp = a ? lp1 : lp0;
            old_logp = a ? lq1 : lq0;
            const float ratio = expf(logp - old_logp);
            const float dlogp = -c.inv_batch * adv * ratio;
            // softmax pair: dL/dz1 = -dL/dz0 (every term depends on the logits through the softmax only)
            g0 = dlogp * ((a == 0 ? 1.0f : 0.0f) - p0) + ge * p0 * (lp0 + H) + kl_w * p0 * ((lp0 - lq0) - KL);
            acc[0] += (double)(ratio * adv);
        } else {
            const float m = c.act_out[i], x = sc.x, mo = od.x, so = od.y;
            const float diff = x - m;
            logp = -(diff * diff) * (0.5f * inv_var) - ls - kKlHalfLog2Pi;
            const float d_old = x - mo;
            old_logp = -(d_old * d_old) * (0.5f * (1.0f / (so * so))) - logf(so) - kKlHalfLog2Pi;
            const float r = sd / so;
            const float s_ratio = r * r;
            const float dm = m - mo;
            const float t1 = (dm / so) * (dm / so);
            KL = 0.5f * (s_ratio + t1 - 1.0f - logf(s_ratio));
            H = Hg;
            const float ratio = expf(logp - old_logp);
            const float dlogp = -c.inv_batch * adv * ratio;
            g0 = dlogp * diff * inv_var + kl_w * (dm * (1.0f / (so * so)));
            gls = dlogp * (diff * diff * inv_var - 1.0f);
            acc[6] += (double)gls - (double)ge + (double)(kl_w * (s_ratio - 1.0f));
            acc[0] += (double)(ratio * adv);
        }
        const float v = c.v_pred[i];
        const float verr = v - sc.w;
        c.dv[i] = c.vf_coef * c.inv_batch * 2.0f * verr;
        if (!GAUSS) {
            g1 = -g0;
            reinterpret_cast<float2*>(c.dact)[i] = make_float2(g0, g1);
        } else {
            c.dact[i] = g0;
        }
        acc[1] += (double)(verr * verr);
        acc[2] += (double)H;
        acc[3] += (double)v;
        acc[5] += (double)KL;
    }
    block_sum<kKlSlots>(acc, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < kKlSlots; ++k) g_kl_partials[blockIdx.x * kKlSlots + k] = acc[k];
        __threadfence();
        is_last = (atomicAdd(&g_kl_ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    __shared__ double tot[kKlSlots];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int k = warp; k < kKlSlots; k += kKlBlock / 32) {   // one warp per output, CTA partials added in a fixed order
        double s = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) s += g_kl_partials[b * kKlSlots + k];
        s = warp_sum(s);
        if (lane == 0) tot[k] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < 6; ++k) c.scalars[k] = k == 4 ? 0.0 : tot[k];
        c.scalars[6] = 0.0;
        c.scalars[7] = 0.0;
        if (GAUSS) c.dlogstd[0] = tot[6];
        if (c.kl_sum_out) *c.kl_sum_out = tot[5];
        if (c.adapt)
            kl_adapt_store(c.kl_coef, c.kl_used, tot[5], c.inv_kl_count, c.target_kl);
        else if (c.kl_used)
            *c.kl_used = *c.kl_coef;
        g_kl_ticket = 0u;
    }
}

__global__ void ppokl_kl_adapt_kernel(const double* __restrict__ kl_sum, float* kl_coef, float* kl_used, float target_kl,
                                      double inv_count) {
    kl_adapt_store(kl_coef, kl_used, *kl_sum, inv_count, target_kl);
}

}  // namespace xb

using namespace xb;

extern "C" int xb_ppokl_loss_packed(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* scal,
                                    const float* old_dist, const float* act_out, const float* logstd, int gaussian,
                                    const float* v_pred, const double* adv_stats, int64_t adv_count, float vf_coef,
                                    float ent_coef, float inv_batch, float* kl_coef, float* kl_used, float target_kl,
                                    int adapt, int64_t kl_count, double* kl_sum_out, float* dact, float* dv, double* dlogstd,
                                    double* scalars, xb_stream_t stream) {
    if (B <= 0 || T <= 0 || N <= 0 || !idx || !scal || !old_dist || !act_out || !v_pred || !kl_coef || !dact || !dv ||
        !scalars)
        return XB_E_BADARG;
    if (((uintptr_t)scal & 15u) || ((uintptr_t)old_dist & 7u) || (!gaussian && (((uintptr_t)act_out | (uintptr_t)dact) & 7u)))
        return XB_E_BADARG;
    if (gaussian && (!logstd || !dlogstd)) return XB_E_BADARG;
    if (adv_stats && adv_count <= 0) return XB_E_BADARG;
    if (adapt && kl_count <= 0) return XB_E_BADARG;
    PpoklArgs c{idx, B, T, N, (const float4*)scal, (const float2*)old_dist, act_out, logstd, v_pred, adv_stats,
                adv_stats ? 1.0 / (double)adv_count : 0.0, vf_coef, ent_coef, inv_batch, kl_coef, kl_used, target_kl,
                adapt, kl_count > 0 ? 1.0 / (double)kl_count : 0.0, kl_sum_out, dact, dv, dlogstd, scalars};
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = grid_for(B, kKlBlock, 8);
    if (grid > kKlMaxGrid) return XB_E_UNSUPPORTED;
    if (gaussian)
        ppokl_loss_packed_kernel<true><<<grid, kKlBlock, 0, s>>>(c);
    else
        ppokl_loss_packed_kernel<false><<<grid, kKlBlock, 0, s>>>(c);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_ppokl_kl_adapt(const double* kl_sum, float* kl_coef, float* kl_used, float target_kl, int64_t count,
                                 xb_stream_t stream) {
    if (!kl_sum || !kl_coef || count <= 0) return XB_E_BADARG;
    ppokl_kl_adapt_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(kl_sum, kl_coef, kl_used, target_kl, 1.0 / (double)count);
    XB_LAUNCH_CHECK();
    return 0;
}
