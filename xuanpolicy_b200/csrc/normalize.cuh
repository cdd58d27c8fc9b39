// normalize.cuh — device-side RunningMeanStd pieces shared by normalize.cu, env_classic.cu (fused rollout step) and
// dense_tc.cu (rollout forward from raw observations).
//
// Reference: RunningMeanStd.update / update_from_moments  xuance/common/statistic_tools.py:63-112 (Chan merge)
//            Agent._process_observation / _process_reward xuance/torch/agents/agent.py:104-123
//            the per-env discounted-return tracker        ppoclip_agent.py:87,91-92
// State of an observation normaliser: fp64 [2*D + 1] = mean[D], var[D], count, D = floats per observation ROW (4, or 8
// for wide rows); mean / var hold float32 values (the reference keeps float32 arrays, statistic_tools.py:46-47).
// State of the return normaliser: fp64 [3] = mean, var, count (it evolves in float64 in the reference, see normalize.cu).
#pragma once
#include "common.cuh"

namespace xb {

constexpr float kNormEps = 1e-8f;   // EPS of xuance/torch/agents/agent.py

// Chan et al. merge, in float32 like numpy does with float32 arrays and weak python scalars.
__device__ __forceinline__ void chan_merge(float mean, float var, double count, float b_mean, float b_var,
                                           double b_count, float& new_mean, float& new_var, double& new_count) {
    const double tot = count + b_count;
    const float fc = (float)count, fb = (float)b_count, ft = (float)tot;
    const float delta = b_mean - mean;
    new_mean = mean + delta * fb / ft;
    const float m_a = var * fc, m_b = b_var * fb;
    const float m2 = m_a + m_b + delta * delta * fc * fb / ft;
    new_var = m2 / ft;
    new_count = tot;
}

// np.clip((obs - mean) / (std + EPS), -clip, clip)   (agent.py:112-113), float32 like the reference's arrays
__device__ __forceinline__ float norm_apply(float v, float mean, float den, float clip) {
    return fminf(fmaxf((v - mean) / den, -clip), clip);
}
__device__ __forceinline__ void norm_coeffs(const double* __restrict__ state, int D, int d, float& mean, float& den) {
    mean = (float)state[d];
    den = sqrtf((float)state[D + d]) + kNormEps;
}

// ---- statistics carried by the fused rollout step (env_classic.cu) ---------------------------------------------------
// One launch per vector step also (a) merges the NEXT observations' batch moments into the observation normaliser
// (`obs_rms.update(obs)` of the following loop iteration, ppoclip_agent.py:62), (b) advances the per-env return tracker and
// merges the finished episodes' returns into the return normaliser (:87-92), publishing the reward divisor of the next
// step.  Per-CTA partial sums -> ticket -> the last CTA adds them in CTA order (deterministic) and publishes.
struct StepStats {
    const double* obs_state_in;   // nullable: S_t, read by every thread (normalises the stored observation)
    double* obs_state_out;        // S_{t+1} = S_t merged with the next observations' moments (a different buffer)
    int dim;                      // observation floats (<= 4 * row float4s)
    float obs_clip;
    double* ret_state;            // nullable: (mean, var, count) of the return normaliser
    float* rew_std;               // in: divisor of this step's rewards; out: clip(sqrt(var), 0.1, 100) for the next step
    double* returns;              // per-env discounted-return tracker (fp64 [N])
    double gamma;
    int mask_terminal;            // PPO drops the running return on a terminal (:87); A2C does not (a2c_agent.py:85)
    double* partials;             // scratch [grid][kStepStatSlots]
    unsigned int* ticket;         // scratch, self-resetting
    double* sums_out;             // nullable (env-sharded form): the last CTA writes THIS RANK's totals [2D + 4] = sum x[D],
                                  // sum x^2[D], N, (sum R, sum R^2, n finished) there instead of merging; the ranks' sums are
                                  // then exchanged (peer_comm.cu) and merged by xb_rms_merge_sums
#ifdef XB_STEP_TS
    unsigned long long* ts;
#endif
};
constexpr int kStepStatSlots = 20;   // 8 sums + 8 sums of squares + (sum R, sum R^2, n finished) + pad

// Merges batch sums into the two normalisers (threads 0..D-1 of one warp): observation state_in -> state_out (Chan, float32,
// statistic_tools.py:101-112) from this thread's (sum x_d, sum x_d^2) over n rows; return state in place (fp64, thread 0) from
// (sum R, sum R^2, n_ret), publishing the reward divisor clip(sqrt(var), 0.1, 100) (agent.py:119-120).
template <int D>
__device__ __forceinline__ void merge_step_stats(const double* obs_state_in, double* obs_state_out, int dim, double* ret_state,
                                                 float* rew_std, double sum_d, double sumsq_d, double n, double r_sum,
                                                 double r_sumsq, double r_n, int tid) {
    if (tid < D && obs_state_in) {
        const int d = tid;
        float nm = (float)obs_state_in[d], nv = (float)obs_state_in[D + d];
        double new_count = obs_state_in[2 * D];
        if (d < dim) {
            const double bm = sum_d / n;
            double bv = sumsq_d / n - bm * bm;            // np.square(np.std(x, axis=0))
            bv = bv > 0.0 ? bv : 0.0;
            chan_merge(nm, nv, obs_state_in[2 * D], (float)bm, (float)bv, n, nm, nv, new_count);
        }
        obs_state_out[d] = (double)nm;
        obs_state_out[D + d] = (double)nv;
        if (d == 0) obs_state_out[2 * D] = obs_state_in[2 * D] + n;
    }
    if (tid == 0 && ret_state) {
        if (r_n > 0.0) {
            const double bm = r_sum / r_n;
            double bv = r_sumsq / r_n - bm * bm;
            bv = bv > 0.0 ? bv : 0.0;
            const double count = ret_state[2], tot = count + r_n, delta = bm - ret_state[0];   // Chan merge in fp64
            const double m2 = ret_state[1] * count + bv * r_n + delta * delta * count * r_n / tot;
            ret_state[0] = ret_state[0] + delta * r_n / tot;
            ret_state[1] = m2 / tot;
            ret_state[2] = tot;
        }
        *rew_std = (float)fmin(fmax(sqrt(ret_state[1]), 0.1), 100.0);     // agent.py:120
    }
}

// merge_step_stats from the cross-rank totals of one step in the StepStats::sums_out layout [2D + 4] = sum x[D], sum x^2[D], N,
// sum R, sum R^2, n finished, for D = 4 or 8 floats per observation row (threads 0..31 of one warp).
__device__ __forceinline__ void merge_step_sums(const double* sums, int D, const double* obs_state_in, double* obs_state_out, int dim,
                                                double* ret_state, float* rew_std, int tid) {
    const int d = tid < D ? tid : 0;
    if (D == 8)
        merge_step_stats<8>(obs_state_in, obs_state_out, dim, ret_state, rew_std, sums[d], sums[8 + d], sums[16], sums[17], sums[18],
                            sums[19], tid);
    else
        merge_step_stats<4>(obs_state_in, obs_state_out, dim, ret_state, rew_std, sums[d], sums[4 + d], sums[8], sums[9], sums[10],
                            sums[11], tid);
}

// Sum of 32 doubles in shared memory, read in an order rotated by `rot` (lanes that walk rows 256 B apart then never share a
// bank) and added as four independent chains: a fixed association order, a quarter of the dependent-add latency.
__device__ __forceinline__ double row_sum32(const double* row, int rot) {
    double a[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
#pragma unroll
        for (int q = 0; q < 4; ++q) a[q] += row[(j + q + rot) & 31];
    }
    return (a[0] + a[1]) + (a[2] + a[3]);
}

// ticket increment with release + acquire semantics at device scope: the partial sums stored before it (by this thread, and by
// the lanes it synchronised with through __syncwarp / __syncthreads) are visible to whoever observes the count, and the last
// arriver's later loads see every other CTA's sums — no separate fences.
__device__ __forceinline__ unsigned int ticket_take(unsigned int* ticket) {
    unsigned int old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(ticket) : "memory");
    return old;
}

// acc: [0, D) sum x_d | [D, 2D) sum x_d^2 | [2D, 2D+3) finished-return sums.  Called by EVERY thread of the CTA.
// The whole path is latency: every step of the rollout waits for it (tools/profile/step_timeline.py).  One-warp CTAs
// transpose their 32 x K values through shared memory so that lane k adds sum k over the lanes (no shuffle butterflies) and
// stores it.  The last CTA's warp 0 loads the per-CTA rows with ALL their loads in flight at once (lane l takes rows l,
// l + 32, ...; up to 4 rows x K values per lane and pass), transposes the lanes' subtotals through shared memory the same way,
// and merges: observation dimensions on lanes 0..D-1, the return normaliser on lane 16, side by side.  Every association order
// depends on the launch geometry only: replays give the same bits.  `cta`: the partials row of this CTA (its place in the
// CTA order the last CTA adds in); on return, *flag tells whether this CTA was the last one.
template <int D>
__device__ __forceinline__ void step_stats_finish_at(const StepStats& s, double (&acc)[2 * D + 3], int64_t N, double* smem,
                                                     bool* flag, int cta) {
    constexpr int K = 2 * D + 3;
    constexpr unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    double* mine = s.partials + (int64_t)cta * kStepStatSlots;
    if (blockDim.x == 32) {
#pragma unroll
        for (int k = 0; k < K; ++k) smem[k * 32 + lane] = acc[k];
        __syncwarp();
        const double v = lane < K ? row_sum32(smem + lane * 32, lane) : 0.0;
        __syncwarp();
        if (lane < K) smem[lane] = v;
        __syncwarp();
        if (lane == 0) {                        // one thread stores the row and releases it with the ticket
#pragma unroll
            for (int k = 0; k < K; ++k) mine[k] = smem[k];
            *flag = (ticket_take(s.ticket) == gridDim.x - 1);
        }
        __syncwarp();
    } else {
        block_sum<K>(acc, smem);
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < K; ++k) mine[k] = acc[k];
            *flag = (ticket_take(s.ticket) == gridDim.x - 1);
        }
        __syncthreads();
    }
    if (!*flag) return;
    if (threadIdx.x >= 32) return;              // the rest happens in warp 0 of the last CTA
    XB_STEP_STAMP(s.ts, 102);
    // the states the merge starts from: requested now, needed after the sums are in
    const int d = lane < D ? lane : 0;
    double st_mean = 0.0, st_var = 0.0, st_count = 0.0, r_mean = 0.0, r_var = 0.0, r_count = 0.0;
    if (s.obs_state_in && !s.sums_out) {
        st_mean = s.obs_state_in[d];
        st_var = s.obs_state_in[D + d];
        st_count = s.obs_state_in[2 * D];
    }
    if (s.ret_state && !s.sums_out) {
        r_mean = s.ret_state[0];
        r_var = s.ret_state[1];
        r_count = s.ret_state[2];
    }
    XB_STEP_STAMP(s.ts, 105);
    const int grid = gridDim.x;
    double t[K];
#pragma unroll
    for (int k = 0; k < K; ++k) t[k] = 0.0;
    constexpr int U = D <= 4 ? 4 : 2;
    for (int b0 = lane; b0 < grid; b0 += 32 * U) {
        double u[U][K];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int b = b0 + 32 * j;
            const double* p = s.partials + (int64_t)(b < grid ? b : 0) * kStepStatSlots;
#pragma unroll
            for (int k = 0; k < K; ++k) u[j][k] = b < grid ? __ldcg(p + k) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < U; ++j)
#pragma unroll
            for (int k = 0; k < K; ++k) t[k] += u[j][k];
    }
    __syncwarp();                               // (shared memory is reused: every lane is past its own first pass)
#pragma unroll
    for (int k = 0; k < K; ++k) smem[k * 32 + lane] = t[k];
    __syncwarp();
    const double tot = lane < K ? row_sum32(smem + lane * 32, lane) : 0.0;
    XB_STEP_STAMP(s.ts, 106);
    if (s.sums_out) {
        if (lane < 2 * D) s.sums_out[lane] = tot;
        else if (lane < K) s.sums_out[lane + 1] = tot;
        if (lane == 0) s.sums_out[2 * D] = (double)N;
    } else {
        const double sum_d = __shfl_sync(kFull, tot, d), sumsq_d = __shfl_sync(kFull, tot, D + d);
        const double r_sum = __shfl_sync(kFull, tot, 2 * D), r_sumsq = __shfl_sync(kFull, tot, 2 * D + 1);
        const double r_n = __shfl_sync(kFull, tot, 2 * D + 2);
        if (lane < D && s.obs_state_in) {
            const double n = (double)N;
            float nm = (float)st_mean, nv = (float)st_var;
            double new_count = st_count;
            if (lane < s.dim) {
                const double bm = sum_d / n;
                double bv = sumsq_d / n - bm * bm;            // np.square(np.std(x, axis=0))
                bv = bv > 0.0 ? bv : 0.0;
                chan_merge(nm, nv, st_count, (float)bm, (float)bv, n, nm, nv, new_count);
            }
            s.obs_state_out[lane] = (double)nm;
            s.obs_state_out[D + lane] = (double)nv;
            if (lane == 0) s.obs_state_out[2 * D] = st_count + n;
        }
        if (lane == 16 && s.ret_state) {
            if (r_n > 0.0) {
                const double bm = r_sum / r_n;
                double bv = r_sumsq / r_n - bm * bm;
                bv = bv > 0.0 ? bv : 0.0;
                const double tot_n = r_count + r_n, delta = bm - r_mean;                       // Chan merge in fp64
                const double m2 = r_var * r_count + bv * r_n + delta * delta * r_count * r_n / tot_n;
                r_mean = r_mean + delta * r_n / tot_n;
                r_var = m2 / tot_n;
                s.ret_state[0] = r_mean;
                s.ret_state[1] = r_var;
                s.ret_state[2] = tot_n;
            }
            *s.rew_std = (float)fmin(fmax(sqrt(r_var), 0.1), 100.0);     // agent.py:120
        }
    }
    XB_STEP_STAMP(s.ts, 107);
    if (lane == 0) *s.ticket = 0u;
    XB_STEP_STAMP(s.ts, 103);
}
template <int D>
__device__ __forceinline__ void step_stats_finish(const StepStats& s, double (&acc)[2 * D + 3], int64_t N, double* smem,
                                                  bool* flag) {
    step_stats_finish_at<D>(s, acc, N, smem, flag, blockIdx.x);
}

}  // namespace xb
