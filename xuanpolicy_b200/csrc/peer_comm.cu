// peer_comm.cu — the two exchanges of the env-sharded PPO update over NVLink / NVSwitch PEER MEMORY, fused with
// the computation that consumes them (SURVEY.md §8(e)); no NCCL call on the update path.
//
// One process per GPU.  Every rank owns one cudaMalloc'd "comm block" that its peers map through CUDA IPC:
//
//     [ flags u32 [kPeerSlots][kPeerMaxRanks] | stats fp64 [kPeerStatsMax] | inbox fp32 [2][kPeerMaxRanks][n] ]
//
//   * xb_peer_allreduce_grad_norm — ONE kernel, ONE cross-GPU barrier per update: every CTA PUSHES its slice of the
//     local flat gradient into inbox[parity][my rank] of every peer with posted P2P stores, signals, waits for the
//     same slice from every rank, then sums the W inbox rows in rank order 0..W-1 out of LOCAL memory (bit-identical
//     sums on every rank, so the replicated Adam step stays bit-identical), writes the reduced gradient, accumulates
//     its squared norm and, in the last CTA, derives the clip coefficient / learning rate / bias corrections (what
//     grad_norm_kernel does on one GPU).  It replaces  all_reduce(flat_grad) + the norm pass of clip_grad_norm_
//     (the sharded form of ppoclip_learner.py:47-49): the collective IS the first pass of the optimiser.
//     The inbox is double-buffered by launch parity, so no second barrier is needed: a peer can only overwrite
//     inbox[p] two launches later, after a barrier that this rank enters only once it has finished reading inbox[p].
//   * xb_peer_allreduce_mean — the same push / barrier / rank-order sum, scaled by 1/W and written to local memory, without
//     the optimiser scalars: the gradient exchange of a learner that steps a torch optimiser itself (PPG_Learner).
//   * xb_peer_allreduce_f64 — the (sum adv, sum adv^2) of every minibatch of an epoch in one exchange
//     (the sharded form of memory_tools.py:241-242), fed by xb_adv_stats_minibatches.  Pull-based, two barriers.
//
// Cross-GPU barrier (per CTA, no grid-wide sync): CTA b of rank r release-stores a monotonically increasing ticket
// into flags[b][r] of every peer, then acquire-spins until its own flags[b][*] have reached the ticket.  Tickets
// come from a per-CTA device counter, so a captured CUDA graph replays correctly.
#include <cstring>

#include "normalize.cuh"
#include "optim.cuh"

namespace xb {

constexpr int kPeerMaxRanks = 8;
constexpr int kPeerSlots = 64;       // CTA slots: [0, kPeerSlots-3) gradient all-reduce, [61] the push-form statistics exchange, [62] error flag (tickets only), [63] the pull-form stats exchange
constexpr int kPeerStatsMax = 2048;  // doubles (two per minibatch of an epoch)
constexpr int64_t kPeerFlagsBytes = (int64_t)kPeerSlots * kPeerMaxRanks * sizeof(uint32_t);
constexpr int64_t kPeerStatsOff = kPeerFlagsBytes;
constexpr int64_t kPeerGradOff = kPeerStatsOff + (int64_t)kPeerStatsMax * sizeof(double);

struct PeerTable {
    char* base[kPeerMaxRanks];
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_peer_f4(const float4* p) {  // never served from a stale L1 line
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_peer_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

constexpr unsigned long long kPeerTimeoutNs = 60ULL * 1000 * 1000 * 1000;   // a peer that is 60 s late is gone
constexpr int kPeerErrSlot = kPeerSlots - 2;                                // tickets[kPeerErrSlot] != 0: a barrier timed out

// All threads of the CTA call it; `ticket` must be the same in every rank for the same barrier instance.
// A wait that exceeds kPeerTimeoutNs gives up and raises the rank-local error flag (the host turns it into an exception)
// instead of spinning forever when a peer process has died.
__device__ __forceinline__ void peer_barrier(const PeerTable& t, int rank, int W, int slot, uint32_t ticket, uint32_t* tickets) {
    __syncthreads();  // every thread's earlier accesses are ordered before the release below
    if ((int)threadIdx.x < W) {
        const int peer = threadIdx.x;
        uint32_t* theirs = reinterpret_cast<uint32_t*>(t.base[peer]) + slot * kPeerMaxRanks + rank;
        st_release_sys(theirs, ticket);
        const uint32_t* mine = reinterpret_cast<const uint32_t*>(t.base[rank]) + slot * kPeerMaxRanks + peer;
        unsigned long long t0 = 0;
        unsigned int spins = 0;
        while ((int32_t)(ld_acquire_sys(mine) - ticket) < 0) {
            if ((++spins & 0x3ffu) == 0) {           // look at the clock every 1024 polls
                const unsigned long long now = global_timer_ns();
                if (t0 == 0) t0 = now;
                else if (now - t0 > kPeerTimeoutNs) {
                    tickets[kPeerErrSlot] = 1u;
                    break;
                }
            }
        }
    }
    __syncthreads();
}

constexpr int kPeerBlock = 512;

// The gradient exchange shared by the kernels below (every CTA of the grid calls it): CTA b pushes its grid-stride slice of
// grad_in (float4 [n4]) into inbox[parity][rank] of every peer, passes ONE cross-GPU barrier on flag slot b, then calls
// visit(i, s) for each float4 i of its slice with s = the W inbox rows summed in rank order 0..W-1 out of LOCAL memory
// (bit-identical on every rank).  tickets: u32 [kPeerSlots] local per-CTA barrier counters (one tick per launch; its parity
// selects the inbox half).  Launches that share a comm block must use the same grid, i.e. the same n.
template <class Visit>
__device__ __forceinline__ void peer_grad_sum(const PeerTable& t, int rank, int W, int64_t n4, const float* __restrict__ grad_in,
                                              uint32_t* __restrict__ tickets, Visit visit) {
    const int slot = blockIdx.x;
    const uint32_t base_ticket = tickets[slot];          // read by every thread before thread 0 advances it below
    const int64_t half = (int64_t)(base_ticket & 1u) * kPeerMaxRanks * n4;   // float4 offset of this launch's inbox half
    const float4* in4 = reinterpret_cast<const float4*>(grad_in);
    // push my slice into every rank's inbox row [rank] (own row included: a plain local store)
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 g = in4[i];
        for (int r = 0; r < W; ++r) reinterpret_cast<float4*>(t.base[r] + kPeerGradOff)[half + (int64_t)rank * n4 + i] = g;
    }
    peer_barrier(t, rank, W, slot, base_ticket + 1, tickets);     // every rank's slice has landed in my inbox
    if (threadIdx.x == 0) tickets[slot] = base_ticket + 1;
    const float4* box = reinterpret_cast<const float4*>(t.base[rank] + kPeerGradOff) + half;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 s = ld_peer_f4(box + i);                  // written by remote stores: bypass any stale L1 line
        for (int r = 1; r < W; ++r) {
            const float4 g = ld_peer_f4(box + (int64_t)r * n4 + i);
            s.x += g.x; s.y += g.y; s.z += g.z; s.w += g.w;
        }
        visit(i, s);
    }
}

// ws layout = optim.cu: [0] norm [1] clip [2] lr [3] bc1 [4] sqrt(bc2) [5] ticket bits, [8..) per-CTA partials.
__global__ void __launch_bounds__(kPeerBlock)
    peer_allreduce_grad_norm_kernel(PeerTable t, int rank, int W, int64_t n4, const float* __restrict__ grad_in,
                                    float* __restrict__ grad_out, uint32_t* __restrict__ tickets,
                                    int64_t* __restrict__ step_dev, AdamHyper h, double* __restrict__ ws,
                                    float* __restrict__ lr_out, float* __restrict__ gnorm_out) {
    __shared__ double smem[32];
    __shared__ bool is_last;
    double acc[1] = {0.0};
    float4* out4 = reinterpret_cast<float4*>(grad_out);
    peer_grad_sum(t, rank, W, n4, grad_in, tickets, [&](int64_t i, const float4& s) {
        out4[i] = s;
        const double gx = (double)(s.x * h.grad_scale), gy = (double)(s.y * h.grad_scale);
        const double gz = (double)(s.z * h.grad_scale), gw = (double)(s.w * h.grad_scale);
        acc[0] += gx * gx + gy * gy + gz * gz + gw * gw;
    });
    grad_norm_finish(acc[0], step_dev, h, ws, lr_out, gnorm_out, smem, &is_last);
}

// grad_out = (sum over ranks of grad_in) * inv_w: the data-parallel mean gradient, for a caller that steps its own optimiser.
__global__ void __launch_bounds__(kPeerBlock)
    peer_allreduce_mean_kernel(PeerTable t, int rank, int W, int64_t n4, const float* __restrict__ grad_in,
                               float* __restrict__ grad_out, uint32_t* __restrict__ tickets, float inv_w) {
    float4* out4 = reinterpret_cast<float4*>(grad_out);
    peer_grad_sum(t, rank, W, n4, grad_in, tickets, [&](int64_t i, const float4& s) {
        out4[i] = make_float4(s.x * inv_w, s.y * inv_w, s.z * inv_w, s.w * inv_w);
    });
}

// out[j] = sum over ranks (rank order) of the peers' stats[j], j < n <= kPeerStatsMax.  One CTA, the last flag slot.
__global__ void __launch_bounds__(256)
    peer_allreduce_f64_kernel(PeerTable t, int rank, int W, int offset, int n, double* __restrict__ out,
                              uint32_t* __restrict__ tickets) {
    const int slot = kPeerSlots - 1;
    const uint32_t base_ticket = tickets[slot];
    peer_barrier(t, rank, W, slot, base_ticket + 1, tickets);
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        double s = 0.0;
        for (int r = 0; r < W; ++r) s += ld_peer_f64(reinterpret_cast<const double*>(t.base[r] + kPeerStatsOff) + offset + j);
        out[j] = s;
    }
    peer_barrier(t, rank, W, slot, base_ticket + 2, tickets);
    if (threadIdx.x == 0) tickets[slot] = base_ticket + 2;
}

// The per-vector-step exchange of the running-statistics sums (env-sharded use_obsnorm / use_rewnorm) as ONE kernel with ONE
// cross-GPU barrier, followed in the same kernel by the normaliser merge (normalize.cuh merge_step_sums = xb_rms_merge_sums):
// every rank PUSHES its n <= kPeerPushMax sums into row [parity][rank] of an inbox inside every peer's statistics area, signals, waits, and
// adds the W rows in rank order out of LOCAL memory (bit-identical totals on every rank).  parity = the launch counter's low bit
// (a device counter: graph replays and odd horizons are fine); a row can only be overwritten two launches later, after a
// barrier this rank enters only once it has read it — so no second barrier (the pull form above needs two), and no separate
// merge launch.  Launched with the programmatic-serialization attribute: the rollout forward that follows may become resident
// (set-up, resident weights) while this kernel waits for its peers.
constexpr int kPeerPushSlot = kPeerSlots - 3;
constexpr int kPeerPushMax = 20;       // the 2D + 4 step sums of 8-float observation rows
__global__ void __launch_bounds__(128)
    peer_allreduce_merge_kernel(PeerTable t, int rank, int W, int inbox_off, int n, const double* __restrict__ src,
                                double* __restrict__ out, uint32_t* __restrict__ tickets, const double* __restrict__ obs_state_in,
                                double* __restrict__ obs_state_out, int dim, double* __restrict__ ret_state,
                                float* __restrict__ rew_std) {
    __shared__ double sums[kPeerPushMax];
    pdl_wait();
    pdl_trigger();
    const uint32_t ticket = tickets[kPeerPushSlot] + 1;
    const int parity = (int)(ticket & 1u);
    for (int i = threadIdx.x; i < n * W; i += blockDim.x) {
        const int peer = i / n, j = i - peer * n;
        double* dst = reinterpret_cast<double*>(t.base[peer] + kPeerStatsOff) + inbox_off + (parity * kPeerMaxRanks + rank) * kPeerPushMax + j;
        *dst = src[j];
    }
    peer_barrier(t, rank, W, kPeerPushSlot, ticket, tickets);
    if ((int)threadIdx.x < kPeerPushMax) {
        double s = 0.0;
        if ((int)threadIdx.x < n) {
            const double* in = reinterpret_cast<const double*>(t.base[rank] + kPeerStatsOff) + inbox_off + parity * kPeerMaxRanks * kPeerPushMax;
            for (int r = 0; r < W; ++r) s += ld_peer_f64(in + r * kPeerPushMax + threadIdx.x);
            out[threadIdx.x] = s;
        }
        sums[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) tickets[kPeerPushSlot] = ticket;
    if (threadIdx.x < 32 && (obs_state_in || ret_state))
        merge_step_sums(sums, (n - 4) / 2, obs_state_in, obs_state_out, dim, ret_state, rew_std, threadIdx.x);
}

// (sum, sumsq) of the advantages of every minibatch of an epoch in one pass over the permutation:
// stats[m] += over i in [m*B, (m+1)*B) of adv[row(idx[i])].  `adv` has element stride `stride` floats per row.
__global__ void __launch_bounds__(256)
    adv_stats_minibatches_kernel(const int64_t* __restrict__ idx, int64_t B, int64_t T, int64_t N,
                                 const float* __restrict__ adv, int64_t stride, int chunks_per_mb, double* __restrict__ stats) {
    __shared__ double smem[2 * 32];
    const int m = blockIdx.x / chunks_per_mb, c = blockIdx.x % chunks_per_mb;
    double acc[2] = {0.0, 0.0};
    for (int64_t i = (int64_t)c * blockDim.x + threadIdx.x; i < B; i += (int64_t)chunks_per_mb * blockDim.x) {
        const int64_t k = idx[(int64_t)m * B + i];
        const int64_t env = k / T;
        const float a = adv[((k - env * T) * N + env) * stride];
        acc[0] += (double)a;
        acc[1] += (double)a * (double)a;
    }
    block_sum<2>(acc, smem);
    if (threadIdx.x == 0) {
        atomicAdd(&stats[2 * m], acc[0]);
        atomicAdd(&stats[2 * m + 1], acc[1]);
    }
}

static int make_table(const void* const* bases, int rank, int W, PeerTable* t) {
    if (!bases || W < 1 || W > kPeerMaxRanks || rank < 0 || rank >= W) return XB_E_BADARG;
    for (int r = 0; r < kPeerMaxRanks; ++r) t->base[r] = r < W ? (char*)bases[r] : nullptr;
    for (int r = 0; r < W; ++r)
        if (!t->base[r]) return XB_E_BADARG;
    return 0;
}

}  // namespace xb

using namespace xb;

extern "C" int64_t xb_peer_block_bytes(int64_t n_grad_floats) {
    return kPeerGradOff + 2 * kPeerMaxRanks * ((n_grad_floats + 3) / 4 * 4) * (int64_t)sizeof(float);
}
extern "C" int64_t xb_peer_stats_offset(void) { return kPeerStatsOff; }
extern "C" int64_t xb_peer_grad_offset(void) { return kPeerGradOff; }
extern "C" int xb_peer_stats_max(void) { return kPeerStatsMax; }

extern "C" int xb_peer_alloc(void** ptr_out /* host */, int64_t bytes) {
    if (!ptr_out || bytes <= 0) return XB_E_BADARG;
    XB_CUDA(cudaMalloc(ptr_out, (size_t)bytes));
    XB_CUDA(cudaMemset(*ptr_out, 0, (size_t)bytes));
    XB_CUDA(cudaDeviceSynchronize());
    return 0;
}
extern "C" int xb_peer_free(void* ptr) {
    XB_CUDA(cudaFree(ptr));
    return 0;
}
extern "C" int xb_peer_export(void* ptr, void* handle_out /* host, 64 bytes */) {
    if (!ptr || !handle_out) return XB_E_BADARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    XB_CUDA(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)handle_out, ptr));
    return 0;
}
extern "C" int xb_peer_import(const void* handle /* host, 64 bytes */, void** ptr_out /* host */) {
    if (!handle || !ptr_out) return XB_E_BADARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    XB_CUDA(cudaIpcOpenMemHandle(ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
extern "C" int xb_peer_close(void* ptr) {
    XB_CUDA(cudaIpcCloseMemHandle(ptr));
    return 0;
}

extern "C" int xb_peer_allreduce_grad_norm(const void* const* peer_bases /* host [W] */, int rank, int W, int64_t n,
                                           const float* grad_in, float* grad_out, uint32_t* tickets, int64_t* step_dev, float lr0,
                                           float lr_end_factor, int64_t lr_total_iters, float beta1, float beta2,
                                           float eps, float max_norm, float grad_scale, double* workspace,
                                           float* lr_out, float* gnorm_out, xb_stream_t stream) {
    PeerTable t;
    int rc = make_table(peer_bases, rank, W, &t);
    if (rc) return rc;
    if (n <= 0 || (n & 3) || !grad_in || !grad_out || !tickets || !step_dev || !workspace) return XB_E_BADARG;
    AdamHyper h{lr0, lr_end_factor, beta1, beta2, eps, max_norm, grad_scale, lr_total_iters};
    const int64_t n4 = n / 4;
    int grid = (int)((n4 + kPeerBlock - 1) / kPeerBlock);
    if (grid > kPeerSlots - 3) grid = kPeerSlots - 3;
    peer_allreduce_grad_norm_kernel<<<grid, kPeerBlock, 0, (cudaStream_t)stream>>>(t, rank, W, n4, grad_in, grad_out, tickets, step_dev,
                                                                                  h, workspace, lr_out, gnorm_out);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_peer_allreduce_mean(const void* const* peer_bases /* host [W] */, int rank, int W, int64_t n, const float* grad_in,
                                      float* grad_out, uint32_t* tickets, xb_stream_t stream) {
    PeerTable t;
    int rc = make_table(peer_bases, rank, W, &t);
    if (rc) return rc;
    if (n <= 0 || (n & 3) || !grad_in || !grad_out || !tickets) return XB_E_BADARG;
    const int64_t n4 = n / 4;
    int grid = (int)((n4 + kPeerBlock - 1) / kPeerBlock);
    if (grid > kPeerSlots - 3) grid = kPeerSlots - 3;
    peer_allreduce_mean_kernel<<<grid, kPeerBlock, 0, (cudaStream_t)stream>>>(t, rank, W, n4, grad_in, grad_out, tickets, 1.0f / (float)W);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_peer_allreduce_f64(const void* const* peer_bases /* host [W] */, int rank, int W, int offset, int n,
                                     double* out, uint32_t* tickets, xb_stream_t stream) {
    PeerTable t;
    int rc = make_table(peer_bases, rank, W, &t);
    if (rc) return rc;
    if (n <= 0 || offset < 0 || offset + n > kPeerStatsMax || !out || !tickets) return XB_E_BADARG;
    peer_allreduce_f64_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(t, rank, W, offset, n, out, tickets);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_peer_allreduce_merge(const void* const* peer_bases /* host [W] */, int rank, int W, const double* src, int n,
                                       int inbox_offset, double* out, uint32_t* tickets, const double* obs_state_in,
                                       double* obs_state_out, int dim, double* ret_state, float* rew_std, xb_stream_t stream) {
    PeerTable t;
    int rc = make_table(peer_bases, rank, W, &t);
    if (rc) return rc;
    if (!src || !out || !tickets || n <= 0 || n > kPeerPushMax || inbox_offset < 0 ||
        inbox_offset + 2 * kPeerMaxRanks * kPeerPushMax > kPeerStatsMax)
        return XB_E_BADARG;
    if ((obs_state_in || ret_state) && n != 12 && n != 20) return XB_E_BADARG;     // the merge reads the 2D + 4 step sums, D = 4 or 8
    if (obs_state_in && (!obs_state_out || obs_state_in == obs_state_out || dim < 1 || dim > (n - 4) / 2)) return XB_E_BADARG;
    if (ret_state && !rew_std) return XB_E_BADARG;
    XB_CUDA(launch_pdl(peer_allreduce_merge_kernel, dim3(1), dim3(128), 0, (cudaStream_t)stream, true, t, rank, W, inbox_offset, n, src,
                       out, tickets, obs_state_in, obs_state_out, dim, ret_state, rew_std));
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_adv_stats_minibatches(const int64_t* idx, int64_t n_minibatches, int64_t B, int64_t T, int64_t N,
                                        const float* adv, int64_t stride, double* stats, xb_stream_t stream) {
    if (!idx || !adv || !stats || n_minibatches <= 0 || B <= 0 || T <= 0 || N <= 0 || stride < 1) return XB_E_BADARG;
    cudaStream_t s = (cudaStream_t)stream;
    XB_CUDA(cudaMemsetAsync(stats, 0, (size_t)n_minibatches * 2 * sizeof(double), s));
    int chunks = (int)((B + 256 * 8 - 1) / (256 * 8));
    const int cap = (int)((int64_t)kNumSMs * 8 / n_minibatches);
    if (chunks > cap) chunks = cap;
    if (chunks < 1) chunks = 1;
    adv_stats_minibatches_kernel<<<(unsigned)(n_minibatches * chunks), 256, 0, s>>>(idx, B, T, N, adv, stride, chunks, stats);
    XB_LAUNCH_CHECK();
    return 0;
}
