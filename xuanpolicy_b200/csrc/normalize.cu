// normalize.cu — device-side RunningMeanStd + observation / reward normalisation (SURVEY.md §8 row f1).
//
// Replaces, on the per-step path of PPOCLIP_Agent.train (ppoclip_agent.py:63-64,68,87-92):
//     RunningMeanStd.update / update_from_moments      xuance/common/statistic_tools.py:63-112  (Chan merge)
//     Agent._process_observation / _process_reward     xuance/torch/agents/agent.py:104-123
//     the per-env discounted-return tracker            ppoclip_agent.py:87,91-92
// State per normaliser: fp64 [2*D+1] = mean[D], var[D], count, with mean/var rounded to float32 after every
// merge (the reference keeps them as float32 arrays, statistic_tools.py:46-47).
//
// Per step: `moments` (column sums over the env batch, deterministic last-block finish) -> [optional NCCL
// all-reduce of the 2*D+1 sums across ranks: the analogue of mpi_mean, statistic_tools.py:6-17] ->
// `rms_normalize` (every thread re-derives the merged statistics — a handful of flops — and normalises its
// row; one thread publishes the merged state into the OTHER state buffer, so readers never race the writer).
#include "common.cuh"
#include "normalize.cuh"

namespace xb {

constexpr int kNormBlock = 256;
constexpr int kNormMaxGrid = kNumSMs * 8;

// rows of D = 4 * V floats: sums[0, D) = sum x_d, sums[D, 2D) = sum x_d^2, sums[2D] = N
template <int V>
__global__ void __launch_bounds__(kNormBlock)
    moments_kernel(const float4* __restrict__ x, int64_t N, double* __restrict__ sums, double* __restrict__ ws) {
    constexpr int D = 4 * V, K = 2 * D;
    __shared__ double smem[K * 32];
    __shared__ bool is_last;
    double a[K];
#pragma unroll
    for (int k = 0; k < K; ++k) a[k] = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float4 q = x[i * V + v];
            a[4 * v + 0] += q.x; a[4 * v + 1] += q.y; a[4 * v + 2] += q.z; a[4 * v + 3] += q.w;
            a[D + 4 * v + 0] += (double)q.x * q.x; a[D + 4 * v + 1] += (double)q.y * q.y;
            a[D + 4 * v + 2] += (double)q.z * q.z; a[D + 4 * v + 3] += (double)q.w * q.w;
        }
    }
    block_sum<K>(a, smem);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws);
    double* partials = ws + 8;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) partials[K * blockIdx.x + k] = a[k];
        __threadfence();
        is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double t[K];
#pragma unroll
        for (int k = 0; k < K; ++k) t[k] = 0.0;
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
#pragma unroll
            for (int k = 0; k < K; ++k) t[k] += partials[K * b + k];
        }
        block_sum<K>(t, smem);
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < K; ++k) sums[k] = t[k];
            sums[K] = (double)N;
            *ticket = 0u;
        }
    }
}

__global__ void __launch_bounds__(kNormBlock)
    rms_normalize_kernel(const float4* __restrict__ x, int dim, const double* __restrict__ sums,
                         const double* __restrict__ state_in, double* __restrict__ state_out, float clip,
                         float4* __restrict__ out, int64_t N, int64_t n_merged_rows) {
    // rows [0, n_merged_rows) are normalised with the MERGED statistics, the rest with state_in as it is
    float mean[4], den[4], mean_old[4], den_old[4];
    const double b_count = n_merged_rows > 0 ? sums[8] : 0.0, count = state_in[8];
    double new_count = count;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        mean[d] = mean_old[d] = 0.0f;
        den[d] = den_old[d] = 1.0f;
        if (d < dim) {
            float nm = (float)state_in[d], nv = (float)state_in[4 + d];
            mean_old[d] = nm;
            den_old[d] = sqrtf(nv) + 1e-8f;
            if (b_count > 0.0) {
                const double bm = sums[d] / b_count;
                double bv = sums[4 + d] / b_count - bm * bm;   // np.square(np.std(x, axis=0))
                bv = bv > 0.0 ? bv : 0.0;
                chan_merge((float)state_in[d], (float)state_in[4 + d], count, (float)bm, (float)bv, b_count, nm, nv, new_count);
            }
            mean[d] = nm;
            den[d] = sqrtf(nv) + 1e-8f;
            if (blockIdx.x == 0 && threadIdx.x == 0) {
                state_out[d] = (double)nm;
                state_out[4 + d] = (double)nv;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) state_out[8] = new_count;
    const float keep[4] = {dim > 0 ? 1.0f : 0.0f, dim > 1 ? 1.0f : 0.0f, dim > 2 ? 1.0f : 0.0f, dim > 3 ? 1.0f : 0.0f};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = x[i];
        const bool nw = i < n_merged_rows;
        float4 o;   // (obs - mean) / (std + EPS), clipped  (agent.py:112-113)
        o.x = keep[0] * fminf(fmaxf((v.x - (nw ? mean[0] : mean_old[0])) / (nw ? den[0] : den_old[0]), -clip), clip);
        o.y = keep[1] * fminf(fmaxf((v.y - (nw ? mean[1] : mean_old[1])) / (nw ? den[1] : den_old[1]), -clip), clip);
        o.z = keep[2] * fminf(fmaxf((v.z - (nw ? mean[2] : mean_old[2])) / (nw ? den[2] : den_old[2]), -clip), clip);
        o.w = keep[3] * fminf(fmaxf((v.w - (nw ? mean[3] : mean_old[3])) / (nw ? den[3] : den_old[3]), -clip), clip);
        out[i] = o;
    }
}

// returns = (1 - term) * gamma * returns + rew ; finished envs contribute (R, R^2, 1) and restart at 0.
// fp64 like the reference: `(1 - terminals) * self.gamma * self.returns + rewards` promotes to float64
// (int64 array x python float), and ret_rms then evolves in float64 (ppoclip_agent.py:87,91).
__global__ void __launch_bounds__(kNormBlock)
    returns_track_kernel(double* __restrict__ returns, const float* __restrict__ rew, const uint8_t* __restrict__ term,
                         const uint8_t* __restrict__ trunc, double gamma, int mask_terminal, double* __restrict__ sums,
                         double* __restrict__ ws, int64_t N) {
    __shared__ double smem[3 * 32];
    __shared__ bool is_last;
    double a[3] = {0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const bool tm = term[i] != 0, tr = trunc[i] != 0;
        // PPO: (1 - terminals) * gamma * returns + rewards (ppoclip_agent.py:87); A2C: gamma * returns + rewards (a2c_agent.py:85)
        double R = ((tm && mask_terminal) ? 0.0 : 1.0) * gamma * returns[i] + (double)rew[i];
        if (tm || tr) {
            a[0] += R;
            a[1] += R * R;
            a[2] += 1.0;
            R = 0.0;
        }
        returns[i] = R;
    }
    block_sum<3>(a, smem);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws);
    double* partials = ws + 8;
    if (threadIdx.x == 0) {
        for (int k = 0; k < 3; ++k) partials[3 * blockIdx.x + k] = a[k];
        __threadfence();
        is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double t[3] = {0, 0, 0};
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
            for (int k = 0; k < 3; ++k) t[k] += partials[3 * b + k];
        block_sum<3>(t, smem);
        if (threadIdx.x == 0) {
            for (int k = 0; k < 3; ++k) sums[k] = t[k];
            *ticket = 0u;
        }
    }
}

// state = (mean, var, count); sums = (sum R, sum R^2, n finished).  rew_std = clip(sqrt(var), 0.1, 100) (agent.py:120)
__global__ void rms_merge_scalar_kernel(const double* __restrict__ sums, double* __restrict__ state, float* __restrict__ rew_std) {
    const double n = sums[2];
    if (n > 0.0) {
        const double bm = sums[0] / n;
        double bv = sums[1] / n - bm * bm;
        bv = bv > 0.0 ? bv : 0.0;
        const double count = state[2], tot = count + n, delta = bm - state[0];   // Chan merge in fp64
        const double m2 = state[1] * count + bv * n + delta * delta * count * n / tot;
        state[0] = state[0] + delta * n / tot;
        state[1] = m2 / tot;
        state[2] = tot;
    }
    if (rew_std) *rew_std = (float)fmin(fmax(sqrt(state[1]), 0.1), 100.0);
}

// ---- pieces of the fused-statistics rollout path (normalize.cuh) as launches of their own ----------------------------
// out[i] = normalise(x[i]) with `state_new` for rows [0, n_new_rows) and `state_old` for the rest; V float4s per row.
template <int V>
__global__ void __launch_bounds__(kNormBlock)
    rms_apply_kernel(const float4* __restrict__ x, int dim, const double* __restrict__ state_new,
                     const double* __restrict__ state_old, int64_t n_new_rows, float clip, float4* __restrict__ out, int64_t N) {
    constexpr int D = 4 * V;
    float mn[D], dn[D], mo[D], dO[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        mn[d] = mo[d] = 0.f;
        dn[d] = dO[d] = 1.f;
        if (d < dim) {
            norm_coeffs(state_new, D, d, mn[d], dn[d]);
            norm_coeffs(state_old, D, d, mo[d], dO[d]);
        }
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const bool nw = i < n_new_rows;
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float4 q = x[i * V + v];
            const float in[4] = {q.x, q.y, q.z, q.w};
            float o[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int d = 4 * v + k;
                o[k] = d < dim ? norm_apply(in[k], nw ? mn[d] : mo[d], nw ? dn[d] : dO[d], clip) : 0.f;
            }
            out[i * V + v] = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

// state_out = state_in merged with the batch moments of rows x[0, N): `obs_rms.update(obs)` as one launch (used once, for
// the very first observations; afterwards the fused rollout step carries the merge).
template <int V>
__global__ void __launch_bounds__(kNormBlock)
    rms_update_rows_kernel(const float4* __restrict__ x, int64_t N, StepStats s) {
    constexpr int D = 4 * V;
    __shared__ double smem[(2 * D + 3) * 32];
    __shared__ bool flag;
    double acc[2 * D + 3];
#pragma unroll
    for (int k = 0; k < 2 * D + 3; ++k) acc[k] = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float4 q = x[i * V + v];
            const float in[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                acc[4 * v + k] += (double)in[k];
                acc[D + 4 * v + k] += (double)in[k] * (double)in[k];
            }
        }
    }
    step_stats_finish<D>(s, acc, N, smem, &flag);
}

// env-sharded form: `sums` [2D + 4] = the cross-rank totals (sum x[D], sum x^2[D], N, sum R, sum R^2, n finished) of one step
__global__ void rms_merge_sums_kernel(const double* __restrict__ sums, int D, const double* __restrict__ obs_state_in,
                                      double* __restrict__ obs_state_out, int dim, double* __restrict__ ret_state,
                                      float* __restrict__ rew_std) {
    merge_step_sums(sums, D, obs_state_in, obs_state_out, dim, ret_state, rew_std, threadIdx.x);
}

}  // namespace xb

using namespace xb;

extern "C" int xb_rms_merge_sums(const double* sums, int n, const double* obs_state_in, double* obs_state_out, int dim,
                                 double* ret_state, float* rew_std, xb_stream_t stream) {
    if (n != 12 && n != 20) return XB_E_BADARG;          // 2D + 4 sums of D = 4 or 8 floats per row
    const int D = (n - 4) / 2;
    if (!sums || (!obs_state_in && !ret_state) || (obs_state_in && (!obs_state_out || obs_state_in == obs_state_out || dim < 1 || dim > D)) ||
        (ret_state && !rew_std))
        return XB_E_BADARG;
    rms_merge_sums_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(sums, D, obs_state_in, obs_state_out, dim, ret_state, rew_std);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_rms_apply(const float* x, int row_floats, int dim, const double* state_new, const double* state_old,
                            int64_t n_new_rows, float clip, float* out, int64_t N, xb_stream_t stream) {
    if (N <= 0 || !x || !state_new || !state_old || !out || dim < 1 || dim > row_floats || n_new_rows < 0) return XB_E_BADARG;
    if (row_floats != 4 && row_floats != 8) return XB_E_UNSUPPORTED;
    const int grid = grid_for(N, kNormBlock, 2);
    cudaStream_t s = (cudaStream_t)stream;
    if (row_floats == 4)
        rms_apply_kernel<1><<<grid, kNormBlock, 0, s>>>((const float4*)x, dim, state_new, state_old, n_new_rows, clip, (float4*)out, N);
    else
        rms_apply_kernel<2><<<grid, kNormBlock, 0, s>>>((const float4*)x, dim, state_new, state_old, n_new_rows, clip, (float4*)out, N);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_rms_update_rows(const float* x, int row_floats, int dim, int64_t N, const double* state_in, double* state_out,
                                  double* partials, uint32_t* ticket, xb_stream_t stream) {
    if (N <= 0 || !x || !state_in || !state_out || state_in == state_out || !partials || !ticket || dim < 1 || dim > row_floats)
        return XB_E_BADARG;
    if (row_floats != 4 && row_floats != 8) return XB_E_UNSUPPORTED;
    StepStats st{};
    st.obs_state_in = state_in;
    st.obs_state_out = state_out;
    st.dim = dim;
    st.partials = partials;
    st.ticket = ticket;
    st.sums_out = nullptr;
    const int grid = grid_for(N, kNormBlock, 1);
    cudaStream_t s = (cudaStream_t)stream;
    if (row_floats == 4) rms_update_rows_kernel<1><<<grid, kNormBlock, 0, s>>>((const float4*)x, N, st);
    else rms_update_rows_kernel<2><<<grid, kNormBlock, 0, s>>>((const float4*)x, N, st);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_moments4(const float* x, int row_floats, double* sums, double* workspace, int64_t N, xb_stream_t stream) {
    if (N <= 0 || !x || !sums || !workspace || (row_floats != 4 && row_floats != 8)) return XB_E_BADARG;
    const int grid = grid_for(N, kNormBlock, 2);
    cudaStream_t s = (cudaStream_t)stream;
    if (row_floats == 4) moments_kernel<1><<<grid, kNormBlock, 0, s>>>((const float4*)x, N, sums, workspace);
    else moments_kernel<2><<<grid, kNormBlock, 0, s>>>((const float4*)x, N, sums, workspace);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_rms_normalize(const float* x, int dim, const double* sums, const double* state_in, double* state_out,
                                float clip, float* out, int64_t N, int64_t n_merged_rows, xb_stream_t stream) {
    if (N <= 0 || dim < 1 || dim > 4 || !x || !state_in || !state_out || !out || state_in == state_out ||
        n_merged_rows < 0 || n_merged_rows > N || (n_merged_rows > 0 && !sums))
        return XB_E_BADARG;
    rms_normalize_kernel<<<grid_for(N, kNormBlock, 2), kNormBlock, 0, (cudaStream_t)stream>>>(
        (const float4*)x, dim, sums, state_in, state_out, clip, (float4*)out, N, n_merged_rows);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_returns_track(double* returns, const float* rew, const uint8_t* term, const uint8_t* trunc, double gamma,
                                int mask_terminal, double* sums, double* workspace, int64_t N, xb_stream_t stream) {
    if (N <= 0 || !returns || !rew || !term || !trunc || !sums || !workspace) return XB_E_BADARG;
    returns_track_kernel<<<grid_for(N, kNormBlock, 2), kNormBlock, 0, (cudaStream_t)stream>>>(returns, rew, term, trunc, gamma,
                                                                                              mask_terminal, sums, workspace, N);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_rms_merge_scalar(const double* sums, double* state, float* rew_std, xb_stream_t stream) {
    if (!sums || !state) return XB_E_BADARG;
    rms_merge_scalar_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sums, state, rew_std);
    XB_LAUNCH_CHECK();
    return 0;
}
