// dense_tc.cu — the policy/value MLP's dense layers at large batch on the 5th-generation tensor cores (tcgen05),
// with fp32-level accuracy ("3xTF32": x = hi + lo, x*w ~= hi*whi + hi*wlo + lo*whi, fp32 accumulate in TMEM).
//
// Replaces, for the large-batch PPO update / rollout forward, the cuBLAS SIMT sgemm calls torch issues for
//   Basic_MLP.forward                      xuance/torch/representations/mlp.py:49-51
//   ActorNet/CriticNet.forward             xuance/torch/policies/categorical.py:26-32,48-54; gaussian.py:17-24,41-48
// and their autograd backward inside PPOCLIP_Learner.update (ppoclip_learner.py:47-48: loss.backward()).
// The loss tolerance (1e-4 relative in strict fp32) rules out plain TF32; the split keeps ~2^-21 relative error
// per product while running on the tensor pipe instead of the 74 TFLOP/s fp32 SIMT pipe.
//
// Kernel structure (one CTA per SM, persistent over 128-row tiles of the batch, 10 warps):
//   warp 8      TMA producer   : cp.async.bulk.tensor 2D boxes [rows][32 fp32] (128 B rows, SWIZZLE_128B) into a ring
//   warps 4-7   operand warps  : turn the raw tile into the MMA's A operand in place (hi) + a second buffer (lo);
//                                for the backward kernels the raw tile is the saved activation y and the operand is
//                                dz = (dout . w2) * leaky_relu'(y), generated on the fly (never materialised in HBM)
//   warp 9      MMA issuer     : one thread issues tcgen05.mma.kind::tf32 (M=128, N<=256, K=8) x3 per k-step,
//                                tcgen05.commit releases ring slots / publishes the accumulator
//   warps 0-3   epilogue       : tcgen05.ld the 128 x N fp32 accumulator (double-buffered in TMEM so the next
//                                tile's MMAs overlap), bias + LeakyReLU (+ fused narrow head) / activation mask, store;
//                                TS-form forward without a stored Y: the operand warps take half of each tile's columns
//                                (epilogue_share) once they have converted the next tile's k-blocks
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "normalize.cuh"
#include "optim.cuh"
#include "sm100.cuh"

#ifdef XB_STEP_TS
extern unsigned long long* g_xb_step_ts;    // env_classic.cu (debug build only)
#endif

namespace xb {
namespace dense {

using namespace sm100;

#ifdef XB_DENSE_TS   // debug build only: per-role clock64 timeline of CTA 0 ([4 roles][64 its][8 events])
static long long* g_xb_ts_host = nullptr;
#define XB_TS(role, it, ev) do { if (p.ts && blockIdx.x == 0 && (it) < 64) p.ts[((role) * 64 + (it)) * 8 + (ev)] = clock64(); } while (0)
#else
#define XB_TS(role, it, ev) do { } while (0)
#endif

constexpr int BM = 128;                 // batch rows per tile (UMMA M)
constexpr int BK = 32;                  // fp32 per k-block = one 128-byte swizzle span
constexpr int kATile = BM * BK * 4;     // 16 KB
constexpr int kOperandWarps = 8;        // K-major kernels: warps 0-3 epilogue, 4-11 operand, 12 TMA producer, 13 MMA issuer
constexpr int kProducerWarp = 4 + kOperandWarps, kMmaWarp = kProducerWarp + 1;
constexpr int kThreads = (kMmaWarp + 1) * 32;
constexpr int kMiscBytes = 9216;
constexpr int kLossRedOff = 8704;        // last 512 B of the misc area: per-warp loss sums (4 x 8 doubles) + a flag
constexpr int kWMiscBytes = 15360;      // wgrad kernel: barriers, [8 warps][3][128] head/bias-gradient scratch
constexpr int kMaxSmem = 232448;        // 227 KB opt-in limit per CTA

enum { MODE_FWD = 0, MODE_DGRAD = 1 };

// Optional fusion of the PPO-Clip loss forward + backward (ppo_loss.cu, same formulas: SURVEY.md App. C) into the FWD
// epilogue of the dual (actor | critic) launch: the epilogue thread of a row holds the head outputs in registers, so the
// actor CTA turns (mu | logits) straight into dL/dmu | dL/dlogits and the critic CTA v into dL/dv — no separate loss launch,
// no round trip of the head outputs.  Log scalars and the log-std gradient are reduced per CTA and summed in CTA order by the
// last CTA (deterministic).  scal == NULL disables it.
struct FusedLoss {
    const float4* scal;        // packed minibatch scalars [M] = {act, old_logp, adv, ret} (xb_gather_records / _trunk_fwd)
    const double* adv_stats;   // nullable (sum, sumsq) of the global minibatch's advantages -> on-the-fly normalisation
    double inv_adv_count;
    float clip_range, vf_coef, ent_coef, inv_batch;
    int gaussian;              // 1: actor head = mu (A = 1) with a shared log-std; 0: Categorical with 2 logits
    const float* logstd;       // gaussian: [1]
    float* dact;               // out [M][n_head of the actor]
    float* dv;                 // out [M]
    double* partials;          // scratch [gridDim][8]
    unsigned int* ticket;      // scratch, self-resetting
    double* scalars;           // out fp64 [8] = sums of {surrogate, (v-R)^2, entropy, v, clipped count, 0, 0, 0}
    double* dlogstd;           // out fp64 [1] (gaussian)
};

struct KParams {
    FusedLoss loss;
    int64_t M;          // rows of the batch
    int KB;             // number of 32-wide k-blocks
    int kb_split;       // DGRAD: k-blocks [0, kb_split) read source 0, the rest source 1 (actor | critic)
    int stages;         // raw ring depth
    int lo_bufs;        // lo ring depth
    int out_bufs;       // epilogue staging tiles (1 or 2)
    int h1_bufs;        // DGRAD mask tiles (1 or 2)
    float slope;
    int pdl_launch;     // launch with the programmatic-serialization attribute (the kernel waits by itself, common.cuh)
    int pdl_early;      // FWD: set-up and resident-weight loads may run before the wait (XB_FWD_WEIGHTS_STABLE)
#ifdef XB_STEP_TS
    unsigned long long* sts;
#endif
#ifdef XB_DENSE_TS
    long long* ts;
#endif
    // FWD epilogue: Y = leaky(acc + bias); optional head_out[r][j] = Y[r][:] . head_w[j][:] + head_b[j]
    const float* bias;
    float* Y;
    const float* head_w;
    const float* head_b;
    int n_head;
    float* head_out;
    // FWD from observations (TS kernels): the A operand is the trunk layer leaky(W0 obs + b0), generated by the operand
    // warps straight into tensor memory (no h1 round trip; inference / rollout only, obs_dim <= 4, K <= 256)
    const float* obs;
    int obs_ld, obs_dim;
    const float* W0;    // [K][obs_dim]
    const float* b0;    // [K]
    float* h1_out;      // nullable [M][K]: the layer-0 CTAs also store the trunk activations (training: wgrad / dgrad read them)
    // optional observation normalisation in front of the trunk (raw observations in, agent.py:112-113): states fp64 [9]
    const double* norm_new;   // rows [0, norm_rows)
    const double* norm_old;   // rows [norm_rows, M)
    int64_t norm_rows;
    float norm_clip;
    // FWD dual mode: odd CTAs evaluate a second layer on the same input (actor | critic in one launch)
    int dual;
    const float* bias1;
    const float* head_w1;
    const float* head_b1;
    int n_head1;
    float* head_out1;
    // DGRAD operand: dz_s[r][k] = (sum_j dout_s[r][j] * w2_s[j][k]) * leaky'(y_s[r][k]);  epilogue: dZ1 = acc * leaky'(H1)
    const float* dout0;
    const float* w2_0;
    int nh0;
    const float* dout1;
    const float* w2_1;
    int nh1;
    const float* H1;
    float* dZ1;
    int n_split;        // DGRAD (TS kernels): the N output columns are split over n_split CTAs per tile, each with its
                        // N/n_split weight rows resident in shared memory (instead of streaming all of them per tile)
    // DGRAD "mask form" (rank-1 head gradients: one head per source, or a 2-logit softmax head whose two gradients are
    // opposite): dz_s[r][k] = e_s[r] * w2'_s[k] * leaky'(y_s[r][k]) with w2' = w2[0] (- w2[1]).  The column scale w2' moves
    // into the weight operand (Wt'[n][k] = w2'[k] * W[k][n], prepared by the forward launch, see prep_*), so the A operand
    // is e_s[r] or slope * e_s[r]: two hi/lo pairs per row and source, selected per element by the sign of y — no per-element
    // multiply / split in the operand warps.
    int mask_form;
    // TS kernels: the 8 operand warps work as TWO groups of 4 that convert alternate k-blocks (each warp all 32 k-columns of
    // its 32 rows) instead of one group of 8 on every k-block (each warp 16 columns): the per-k-block latency chain
    // (barrier check -> shared-memory read -> split -> tcgen05.st -> wait -> arrive) of one group overlaps the other's.
    int alt_groups;
    // FWD: optional preparation of that weight operand for the dgrad launch that follows (done by the epilogue warps of
    // every CTA before their first tile; 2 H^2 elements in total)
    const float* prep_W[2];     // fp32 master weights [H][H] of the two hidden layers
    const float* prep_w2[2];    // their head weights [nh][H]
    int prep_nh[2];
    float* prep_thi;            // [H][2H]: Wt'[n][s * H + k]
    float* prep_tlo;
    int prep_H;
    // Activation SIGN WORDS.  The backward kernels need the hidden activations only through leaky'(y) = (y > 0 ? 1 : slope), so
    // the FWD epilogue can leave one bit per element: sign_out[row * sign_ld + layer * (N / 32) + c] bit j = (y[row][32 c + j] > 0)
    // (layer = 0 actor, 1 critic in dual mode), and the TS-form DGRAD reads `signs` [M][KB] (one word per row and k-block, the
    // same layout) instead of TMA-loading the two activation tiles: no raw A ring, no A loads, a deeper weight ring.
    uint32_t* sign_out;
    int sign_ld;
    const uint32_t* signs;
    // DGRAD epilogue mask dZ1 = acc * leaky'(H1) from the trunk's sign words h1_signs [M][4] (bit l of word e = H1[4 l + e] > 0; xb_gather_trunk_fwd /
    // xb_mlp_trunk_fwd) instead of TMA-loaded H1 tiles: no mask ring, no 4 N B/row read (N = 128, with `signs` only)
    const uint32_t* h1_signs;
};

// Wt'[n][s * H + k] = split_tf32(w2'_s[k] * W_s[k][n]) — `tid` in [0, 128), all CTAs share the work.
__device__ __forceinline__ void prep_dgrad_operand(const KParams& p, int tid) {
    if (!p.prep_thi) return;
    const int H = p.prep_H, ldt = 2 * H;
    const int total = 2 * H * H;
    for (int i = blockIdx.x * 128 + tid; i < total; i += gridDim.x * 128) {
        const int s = i / (H * H), j = i - s * H * H;
        const int n = j / H, k = j - n * H;                 // consecutive threads: consecutive k -> coalesced stores
        const float* w2 = p.prep_w2[s];
        float c = w2[k];
        if (p.prep_nh[s] == 2) c -= w2[H + k];
        float hi, lo;
        split_tf32(c * p.prep_W[s][k * H + n], hi, lo);
        p.prep_thi[n * ldt + s * H + k] = hi;
        p.prep_tlo[n * ldt + s * H + k] = lo;
    }
}

struct TMaps {          // TMA descriptors: A sources, weight hi/lo, output, DGRAD mask tile; *1 = second layer of FWD dual mode
    CUtensorMap a0, a1, bhi, blo, out, h1, bhi1, blo1, out1;
};

// byte offset of logical 16-byte chunk c (0..7) of row r inside a [rows][128 B] SWIZZLE_128B tile
__device__ __forceinline__ uint32_t sw128_off(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }
// same for the 32-byte-atom flavour (SWIZZLE_128B_ATOM_32B): 32-byte chunk index XOR (row & 3)
__device__ __forceinline__ uint32_t sw32_off(int r, int c) {
    return (uint32_t)(r * 128 + ((((c >> 1) ^ (r & 3)) << 5) | ((c & 1) << 4)));
}

// ------------------------------------------------------------------------------------------------ epilogue (warps 0-3)
// Each warp owns TMEM lanes 32w..32w+31 = 32 rows of the tile and is fully autonomous: accumulator chunk -> registers
// (tcgen05.ld) -> bias/activation/head or activation mask -> its own swizzled 4 KB staging sub-tile -> its own TMA
// store of a [32 rows][32 cols] box (coalesced, off the LSU store path; rows beyond M are clipped by the tensor map).
// DGRAD: the trunk-activation sub-tile for the mask is TMA-loaded per warp, one chunk ahead (double-buffered).
struct EpiCtx {
    uint32_t tmem_base, bar_tfull, bar_tempty, bar_h1w, out_ring, h1_ring;
    int O, HB;
    int64_t tile0, tile_step, n_tiles, M;
    const CUtensorMap* map_out;
    const CUtensorMap* map_h1;
    const float* sf;
    float slope;
    int n_head;
    const float* head_b;
    float* head_out;
    int n_off;         // first output column of this CTA (DGRAD n_split)
    bool store_y;      // FWD: false = only the fused head outputs are wanted (rollout / inference)
    FusedLoss loss;    // FWD: fused PPO loss (loss.scal != NULL)
    int sel;           // FWD dual: 0 = actor CTA, 1 = critic CTA
    uint32_t* sign_out;   // FWD: nullable activation sign words (KParams::sign_out), already offset to this CTA's layer
    int sign_ld;
    const uint32_t* h1_signs;   // DGRAD: nullable trunk sign words [M][4] (N = 128): the mask without the H1 tiles
    double* red;       // shared memory [4 warps][8] for the per-CTA loss sums
    int epi_sets = 1;           // warp sets sharing each tile's columns (TS FWD without a stored Y: 1 + operand-warp sets)
    uint32_t head_terms = 0;    // epi_sets > 1: shared memory [N/32 - kEpiOwnChunks][8][BM] float2 head terms of the other sets
#ifdef XB_DENSE_TS
    long long* ts;
#endif
};

// FWD, 4-column group q of an accumulator chunk: bias + LeakyReLU in place, its 4 activation sign bits into `sign_word`
__device__ __forceinline__ void bias_leaky_group(float4& f, const float* b, float slope, int q, uint32_t& sign_word) {
    f.x += b[0]; f.y += b[1]; f.z += b[2]; f.w += b[3];
    sign_word |= (f.x > 0.f ? 1u : 0u) << (4 * q) | (f.y > 0.f ? 2u : 0u) << (4 * q) |
                 (f.z > 0.f ? 4u : 0u) << (4 * q) | (f.w > 0.f ? 8u : 0u) << (4 * q);
    f.x = f.x > 0.f ? f.x : f.x * slope;
    f.y = f.y > 0.f ? f.y : f.y * slope;
    f.z = f.z > 0.f ? f.z : f.z * slope;
    f.w = f.w > 0.f ? f.w : f.w * slope;
}
// FWD head term of one 4-column group: both the owner warp and the operand-warp sets evaluate it through this one expression,
// so its rounding (and the FMA contraction) is the same wherever a group is computed
__device__ __forceinline__ float head_term(const float4& f, const float* w) {
    return f.x * w[0] + f.y * w[1] + f.z * w[2] + f.w * w[3];
}

// Split FWD epilogue (TS kernel, no stored Y): the epilogue warp of lane quarter lq owns the first N/64 chunks of each tile,
// the operand warps 4 + lq (set 1) and 8 + lq (set 2) take the remaining chunks alternately.  Named barriers per lane quarter:
// kEpiBarFull + lq (the other sets' head terms of a tile are in shared memory), kEpiBarEmpty + lq (the owner has read them).
constexpr int kEpiBarFull = 1, kEpiBarEmpty = 5;
template <int N>
__host__ __device__ constexpr int epi_own_chunks() { return N / 64 > 0 ? N / 64 : 1; }
template <int N>
__host__ __device__ constexpr int epi_sets_of() { return 1 + (N / 32 - epi_own_chunks<N>() < 2 ? N / 32 - epi_own_chunks<N>() : 2); }

template <int N, int MODE>
__device__ __forceinline__ void epilogue_warp(const EpiCtx& c, int warp, int lane) {
    constexpr int kChunks = N / 32;
    const int own_chunks = c.epi_sets > 1 ? epi_own_chunks<N>() : kChunks;
    constexpr uint32_t kSub = 32 * 128;                               // one warp's sub-tile: 32 rows x 128 B
    const uint32_t bar_h1 = c.bar_h1w + warp * 16;                    // 2 barriers per warp
    uint32_t lt = 0, g = 0;
    const uint32_t elected = elect_one_pred();     // the lane that issues this warp's TMA loads / stores (and owns its bulk group)
    // fused loss state (FWD only): advantage normalisation, Gaussian constants, this thread's partial sums
    const bool with_loss = MODE == MODE_FWD && c.loss.scal != nullptr;
    float l_mean = 0.f, l_denom = 1.f, l_ls = 0.f, l_inv_var = 1.f;
    bool l_norm = false;
    double lacc[6] = {0, 0, 0, 0, 0, 0};   // surrogate, value loss, entropy, v, clipped count, dlogstd
    if (with_loss) {
        if (c.loss.adv_stats) {
            const double mean = c.loss.adv_stats[0] * c.loss.inv_adv_count;
            const double var = c.loss.adv_stats[1] * c.loss.inv_adv_count - mean * mean;
            l_mean = (float)mean;
            l_denom = (float)sqrt(var > 0.0 ? var : 0.0) + 1e-8f;
            l_norm = true;
        }
        if (c.loss.gaussian) {
            l_ls = c.loss.logstd[0];
            const float sd = expf(l_ls);
            l_inv_var = 1.0f / (sd * sd);
        }
    }
    const bool mask_bits = MODE == MODE_DGRAD && c.h1_signs != nullptr;
    if (MODE == MODE_DGRAD && !mask_bits && c.tile0 < c.n_tiles) {
        mbar_arrive_expect_tx_if(elected, bar_h1, kSub);
        tma_load_2d_if(elected, c.h1_ring + warp * kSub, c.map_h1, c.n_off, (int)(c.tile0 * BM + warp * 32), bar_h1);
    }
    for (int64_t tile = c.tile0; tile < c.n_tiles; tile += c.tile_step, ++lt) {
        const uint32_t acc = lt & 1, tph = (lt >> 1) & 1;
        const int64_t row = tile * BM + warp * 32 + lane;
        uint4 hw4 = make_uint4(0u, 0u, 0u, 0u);                        // mask_bits: this row's 128 trunk sign bits
        if (mask_bits && row < c.M) hw4 = __ldg(reinterpret_cast<const uint4*>(c.h1_signs) + row);
        mbar_wait(c.bar_tfull + 8 * acc, tph);
#ifdef XB_DENSE_TS
        if (threadIdx.x == 0 && c.ts && blockIdx.x == 0 && lt < 64) c.ts[(3 * 64 + lt) * 8 + 0] = clock64();
#endif
        tc_fence_after();
        const uint32_t taddr = c.tmem_base + ((uint32_t)(warp * 32) << 16) + acc * N;
        float h0 = 0.f, h1 = 0.f;
#pragma unroll 1
        for (int cc = 0; cc < own_chunks; ++cc, ++g) {
#ifdef XB_DENSE_TS
            if (threadIdx.x == 0 && c.ts && blockIdx.x == 0 && lt < 64) c.ts[(3 * 64 + lt) * 8 + 1 + cc] = clock64();
#endif
            uint32_t v[32];
            tmem_ld_32x32(taddr + cc * 32, v);
            const bool store = MODE != MODE_FWD || c.store_y;
            // the staging sub-tile about to be overwritten must have been read out by its previous TMA store
            if (elected && store) {         // at most O - 1 of this warp's stores may still be reading their sub-tiles
                if (c.O > 3) asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory");
                else if (c.O == 3) asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");
                else if (c.O == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
            __syncwarp();
            const uint32_t obuf = c.out_ring + (g % (uint32_t)c.O) * kATile + warp * kSub;
            uint32_t hbuf = 0;
            // (word e of the row holds bit l = feature 4 l + e: this chunk's columns 32 cc + 4 q + e are bits 8 cc + q)
            const uint32_t hx = hw4.x >> (8 * cc), hy = hw4.y >> (8 * cc), hz = hw4.z >> (8 * cc), hw_ = hw4.w >> (8 * cc);
            if (MODE == MODE_DGRAD && !mask_bits) {
                const uint32_t hb = c.HB > 1 ? (g & 1) : 0, hph = c.HB > 1 ? ((g >> 1) & 1) : (g & 1);
                {                      // prefetch the next chunk's mask sub-tile (or, single-buffered, load this chunk's now)
                    int ncc = cc + (c.HB > 1 ? 1 : 0);
                    int64_t ntile = tile;
                    if (ncc == kChunks) { ncc = 0; ntile = tile + c.tile_step; }
                    if (c.HB > 1 ? ntile < c.n_tiles : g > 0) {
                        const uint32_t nb = c.HB > 1 ? ((g + 1) & 1) : 0;
                        mbar_arrive_expect_tx_if(elected, bar_h1 + 8 * nb, kSub);
                        tma_load_2d_if(elected, c.h1_ring + nb * kATile + warp * kSub, c.map_h1, c.n_off + ncc * 32,
                                       (int)(ntile * BM + warp * 32), bar_h1 + 8 * nb);
                    }
                }
                hbuf = c.h1_ring + hb * kATile + warp * kSub;
                mbar_wait(bar_h1 + 8 * hb, hph);
            }
            tmem_ld_wait();
            uint32_t sign_word = 0u;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float4 f = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                                       __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
                if (MODE == MODE_FWD) {
                    const float* b = c.sf + cc * 32 + 4 * q;
                    bias_leaky_group(f, b, c.slope, q, sign_word);
                    const float* w = b + N;
                    h0 += head_term(f, w);
                    h1 += head_term(f, w + N);
                } else if (mask_bits) {
                    f.x *= ((hx >> q) & 1u) ? 1.f : c.slope;
                    f.y *= ((hy >> q) & 1u) ? 1.f : c.slope;
                    f.z *= ((hz >> q) & 1u) ? 1.f : c.slope;
                    f.w *= ((hw_ >> q) & 1u) ? 1.f : c.slope;
                } else {
                    const float4 m = lds128(hbuf + sw128_off(lane, q));
                    f.x *= m.x > 0.f ? 1.f : c.slope;
                    f.y *= m.y > 0.f ? 1.f : c.slope;
                    f.z *= m.z > 0.f ? 1.f : c.slope;
                    f.w *= m.w > 0.f ? 1.f : c.slope;
                }
                if (store) sts128(obuf + sw128_off(lane, q), f);
            }
            if (MODE == MODE_FWD && c.sign_out && row < c.M) c.sign_out[row * c.sign_ld + cc] = sign_word;
            if (store) {
                fence_proxy_async_smem();
                __syncwarp();
                tma_store_2d_commit_if(elected, c.map_out, obuf, c.n_off + cc * 32, (int)(tile * BM + warp * 32));
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(c.bar_tempty + 8 * acc);
        if (MODE == MODE_FWD && c.epi_sets > 1) {     // the other sets' head terms, added in column order after this warp's own
            constexpr int kTerms = (kChunks - epi_own_chunks<N>()) * 8;
            bar_sync_named(kEpiBarFull + warp, 32 * c.epi_sets);
            const uint32_t tb = c.head_terms + (uint32_t)(warp * 32 + lane) * 8;
#pragma unroll
            for (int j = 0; j < kTerms; ++j) {
                const float2 t = lds64(tb + j * (BM * 8));
                h0 += t.x;
                h1 += t.y;
            }
            if (tile + c.tile_step < c.n_tiles) bar_arrive_named(kEpiBarEmpty + warp, 32 * c.epi_sets);
        }
#ifdef XB_DENSE_TS
        if (threadIdx.x == 0 && c.ts && blockIdx.x == 0 && lt < 64) c.ts[(3 * 64 + lt) * 8 + 7] = clock64();
#endif
        if (MODE == MODE_FWD && row < c.M) {
            if (c.n_head > 0) c.head_out[row * c.n_head] = h0 + c.head_b[0];
            if (c.n_head > 1) c.head_out[row * c.n_head + 1] = h1 + c.head_b[1];
            if (with_loss) {
                const float4 sc = c.loss.scal[row];                 // {act, old_logp, adv, ret}
                const float ib = c.loss.inv_batch;
                if (c.sel == 1) {                                   // critic CTA: value loss (ppoclip_learner.py:41)
                    const float v = h0 + c.head_b[0];
                    const float verr = v - sc.w;
                    c.loss.dv[row] = c.loss.vf_coef * ib * (2.0f * verr);
                    lacc[1] += (double)(verr * verr);
                    lacc[3] += (double)v;
                } else {                                            // actor CTA: clipped surrogate + entropy (:33-39,:43)
                    float A = sc.z;
                    if (l_norm) A = (A - l_mean) / l_denom;
                    const float lo = 1.0f - c.loss.clip_range, hi = 1.0f + c.loss.clip_range;
                    const float ge = c.loss.ent_coef * ib;
                    float logp, H, z0 = h0 + c.head_b[0], z1 = 0.f, lse = 0.f, diff = 0.f;
                    int a = 0;
                    if (c.loss.gaussian) {
                        diff = sc.x - z0;
                        logp = -(diff * diff) * (0.5f * l_inv_var) - l_ls - 0.9189385332046727f;
                        H = 0.5f + 0.9189385332046727f + l_ls;
                    } else {
                        z1 = h1 + c.head_b[1];
                        a = (int)sc.x;
                        const float zmax = fmaxf(z0, z1);
                        lse = zmax + logf(expf(z0 - zmax) + expf(z1 - zmax));
                        const float lp0 = z0 - lse, lp1 = z1 - lse;
                        H = -(expf(lp0) * lp0) - expf(lp1) * lp1;
                        logp = a ? lp1 : lp0;
                    }
                    float m, dlogp, ratio = 1.0f;
                    if (c.loss.clip_range > 0.0f) {
                        ratio = expf(logp - sc.y);
                        const float s1 = fminf(fmaxf(ratio, lo), hi) * A;
                        const float s2 = A * ratio;
                        m = fminf(s1, s2);
                        const bool inactive = (A > 0.0f && ratio > hi) || (A < 0.0f && ratio < lo);
                        dlogp = inactive ? 0.0f : -ib * A * ratio;
                    } else {
                        m = A * logp;
                        dlogp = -ib * A;
                    }
                    if (c.loss.gaussian) {
                        c.loss.dact[row] = dlogp * diff * l_inv_var;
                        lacc[5] += (double)(dlogp * (diff * diff * l_inv_var - 1.0f)) - (double)ge;
                    } else {
                        const float lp0 = z0 - lse, lp1 = z1 - lse;
                        const float p0 = expf(lp0), p1 = expf(lp1);
                        c.loss.dact[row * 2] = dlogp * ((a == 0 ? 1.0f : 0.0f) - p0) + ge * p0 * (lp0 + H);
                        c.loss.dact[row * 2 + 1] = dlogp * ((a == 1 ? 1.0f : 0.0f) - p1) + ge * p1 * (lp1 + H);
                    }
                    lacc[0] += (double)m;
                    lacc[2] += (double)H;
                    lacc[4] += (c.loss.clip_range > 0.0f && (ratio < lo || ratio > hi)) ? 1.0 : 0.0;
                }
            }
        }
    }
    if (elected) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (with_loss) {                                                // this warp's sums -> shared memory (finished by the CTA)
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const double v = warp_sum(lacc[k]);
            if (lane == 0) c.red[warp * 8 + k] = v;
        }
    }
}

// Split FWD epilogue, operand-warp side: set `set` (1 or 2) of lane quarter lq takes chunks epi_own_chunks + set - 1, + 2, ...
// of tile `tile` (its lt-th): bias + LeakyReLU, sign words, and the head terms of every 4-column group into `head_terms`, where
// the owner warp adds them to its row sums in column order.  Called after the operand warps have converted the next tile's
// k-blocks, so the MMA stream does not wait on it.
template <int N>
__device__ __forceinline__ void epilogue_share(const EpiCtx& c, int set, int lq, int lane, int64_t tile, uint32_t lt) {
    constexpr int kChunks = N / 32, kOwn = epi_own_chunks<N>();
    const uint32_t acc = lt & 1, tph = (lt >> 1) & 1;
    const int64_t row = tile * BM + lq * 32 + lane;
    if (lt > 0) bar_sync_named(kEpiBarEmpty + lq, 32 * c.epi_sets);     // the owner has read the previous tile's terms
    mbar_wait(c.bar_tfull + 8 * acc, tph);
    tc_fence_after();
    const uint32_t taddr = c.tmem_base + ((uint32_t)(lq * 32) << 16) + acc * N;
#pragma unroll 1
    for (int cc = kOwn + set - 1; cc < kChunks; cc += 2) {
        uint32_t v[32];
        tmem_ld_32x32(taddr + cc * 32, v);
        const uint32_t tb = c.head_terms + ((uint32_t)((cc - kOwn) * 8 * BM) + lq * 32 + lane) * 8;
        tmem_ld_wait();
        uint32_t sign_word = 0u;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float4 f = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                                   __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
            const float* b = c.sf + cc * 32 + 4 * q;
            bias_leaky_group(f, b, c.slope, q, sign_word);
            const float* w = b + N;
            sts64(tb + q * (BM * 8), head_term(f, w), head_term(f, w + N));
        }
        if (c.sign_out && row < c.M) c.sign_out[row * c.sign_ld + cc] = sign_word;
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(c.bar_tempty + 8 * acc);
    bar_arrive_named(kEpiBarFull + lq, 32 * c.epi_sets);
}

// After the CTA-wide barrier that follows the epilogue: CTA sums -> global partials -> the last CTA adds all CTAs' partials
// in CTA order and writes the loss scalars / log-std gradient.  Called by every thread of the CTA.
__device__ __forceinline__ void fused_loss_finish(const FusedLoss& L, const double* red, bool* flag_smem) {
    if (!L.scal) return;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 6; ++k) L.partials[blockIdx.x * 8 + k] = (red[k] + red[8 + k]) + (red[16 + k] + red[24 + k]);
        __threadfence();
        *flag_smem = (atomicAdd(L.ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!*flag_smem) return;
    __threadfence();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < 6) {
        double s = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) s += L.partials[b * 8 + warp];
        s = warp_sum(s);
        if (lane == 0) {
            if (warp < 5) L.scalars[warp] = s;
            else if (L.gaussian && L.dlogstd) L.dlogstd[0] = s;
        }
    }
    if (threadIdx.x < 3) L.scalars[5 + threadIdx.x] = 0.0;
    if (threadIdx.x == 0) *L.ticket = 0u;
}

template <int N, bool B_RES, int MODE>
__global__ void __launch_bounds__(kThreads, 1)
    dense_kmajor_kernel(const __grid_constant__ TMaps maps, const KParams p) {
    constexpr int kBTile = N * BK * 4;                  // one k-block of the weight operand, hi or lo
    constexpr int kTmemCols = 2 * N;                    // double-buffered accumulator (power of two for N in {64,128,256})
    constexpr uint32_t kIdesc = umma_idesc_tf32(BM, N, 0, 0);
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int S = p.stages, L = p.lo_bufs, O = p.out_bufs, HB = p.h1_bufs, KB = p.KB;
    const uint32_t bres = base;                                              // [2][KB][kBTile] when B_RES
    const uint32_t ring = base + (B_RES ? 2u * KB * kBTile : 0u);
    const uint32_t stage_bytes = kATile + (B_RES ? 0 : 2 * kBTile);
    const uint32_t lo_ring = ring + (uint32_t)S * stage_bytes;
    const uint32_t out_ring = lo_ring + (uint32_t)L * kATile;                // epilogue staging tiles [128][128 B]
    const uint32_t h1_ring = out_ring + (uint32_t)O * kATile;                // DGRAD: trunk activation tiles for the mask
    const uint32_t misc = h1_ring + (MODE == MODE_DGRAD ? (uint32_t)HB * kATile : 0u);
    const uint32_t bar_full = misc, bar_conv = misc + 64, bar_empty = misc + 128, bar_loempty = misc + 192;
    const uint32_t bar_tfull = misc + 224, bar_tempty = misc + 240, bar_bfull = misc + 256;
    const uint32_t tmem_slot = misc + 264, bar_h1w = misc + 352;
    unsigned char* misc_ptr = smem_raw + (misc - smem_u32(smem_raw));
    float* sf = reinterpret_cast<float*>(misc_ptr + 512);                    // per-mode float scratch (<= 8 KB)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_tiles = (p.M + BM - 1) / BM;
    // FWD dual mode: CTA parity selects the layer; both walk the same tiles
    const int n_src = (MODE == MODE_FWD && p.dual) ? 2 : 1;
    const int sel = (MODE == MODE_FWD && p.dual) ? (int)(blockIdx.x & 1) : 0;
    const int64_t tile0 = blockIdx.x / n_src, tile_step = gridDim.x / n_src;
    const CUtensorMap* map_a0 = &maps.a0;
    const CUtensorMap* map_a1 = &maps.a1;
    const CUtensorMap* map_bhi = sel ? &maps.bhi1 : &maps.bhi;
    const CUtensorMap* map_blo = sel ? &maps.blo1 : &maps.blo;
    const CUtensorMap* map_out = sel ? &maps.out1 : &maps.out;
    const CUtensorMap* map_h1 = &maps.h1;
    const float* e_bias = sel ? p.bias1 : p.bias;
    const float* e_head_w = sel ? p.head_w1 : p.head_w;
    const float* e_head_b = sel ? p.head_b1 : p.head_b;
    const int e_n_head = sel ? p.n_head1 : p.n_head;
    float* e_head_out = sel ? p.head_out1 : p.head_out;

    // ---------------------------------------------------------------- one-time setup
    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_conv + 8 * s, kOperandWarps);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int j = 0; j < L; ++j) mbar_init(bar_loempty + 8 * j, 1);
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull + 8 * a, 1);
            mbar_init(bar_tempty + 8 * a, 4);
        }
        for (int a = 0; a < 8; ++a) mbar_init(bar_h1w + 8 * a, 1);
        mbar_init(bar_bfull, 1);
        mbar_fence_init();
    }
    if (warp == kMmaWarp) tmem_alloc<kTmemCols>(tmem_slot);
    if (MODE == MODE_FWD) {
        // sf: bias[N] | head_w[2][N]
        for (int i = threadIdx.x; i < N; i += kThreads) {
            sf[i] = e_bias ? e_bias[i] : 0.f;
            sf[N + i] = e_n_head > 0 ? e_head_w[i] : 0.f;
            sf[2 * N + i] = e_n_head > 1 ? e_head_w[N + i] : 0.f;
        }
    } else {
        // sf: w2[src][head][256] (4 x 256 floats) | dout[2 tile parities][128 rows][2 src][2 heads]
        const int K0 = p.kb_split * BK, K1 = (KB - p.kb_split) * BK;
        for (int i = threadIdx.x; i < 256; i += kThreads) {
            sf[i] = (i < K0 && p.nh0 > 0) ? p.w2_0[i] : 0.f;
            sf[256 + i] = (i < K0 && p.nh0 > 1) ? p.w2_0[K0 + i] : 0.f;
            sf[512 + i] = (i < K1 && p.nh1 > 0) ? p.w2_1[i] : 0.f;
            sf[768 + i] = (i < K1 && p.nh1 > 1) ? p.w2_1[K1 + i] : 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == kProducerWarp) {
        // ============================================================ TMA producer (one thread)
        {   // the whole warp walks the loop, one elected lane issues (uniform operands, see tma_load_2d_if)
            const uint32_t elected = elect_one_pred();
            if (lane == 0) {
                tma_prefetch_desc(map_a0);
                tma_prefetch_desc(map_bhi);
                tma_prefetch_desc(map_blo);
                if (MODE == MODE_DGRAD) tma_prefetch_desc(map_a1);
            }
            __syncwarp();
            if (B_RES) {
                mbar_arrive_expect_tx_if(elected, bar_bfull, 2u * KB * kBTile);
                for (int kb = 0; kb < KB; ++kb) {
                    tma_load_2d_if(elected, bres + kb * kBTile, map_bhi, kb * BK, 0, bar_bfull);
                    tma_load_2d_if(elected, bres + (KB + kb) * kBTile, map_blo, kb * BK, 0, bar_bfull);
                }
            }
            uint32_t s = 0, ph = 0, it = 0;
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_step) {
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    mbar_wait(bar_empty + 8 * s, ph ^ 1);
                    XB_TS(0, it, 0);
                    const uint32_t st = ring + s * stage_bytes;
                    mbar_arrive_expect_tx_if(elected, bar_full + 8 * s, stage_bytes);
                    const bool src1 = (MODE == MODE_DGRAD) && kb >= p.kb_split;
                    const int kcol = (src1 ? kb - p.kb_split : kb) * BK;
                    tma_load_2d_if(elected, st, src1 ? map_a1 : map_a0, kcol, (int)(tile * BM), bar_full + 8 * s);
                    if (!B_RES) {
                        tma_load_2d_if(elected, st + kATile, map_bhi, kb * BK, 0, bar_full + 8 * s);
                        tma_load_2d_if(elected, st + kATile + kBTile, map_blo, kb * BK, 0, bar_full + 8 * s);
                    }
                    if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ============================================================ MMA issuer (whole warp walks, one elected lane issues)
        {
            const uint32_t elected = elect_one_pred();
            const uint32_t tmem_base_u = __reduce_max_sync(0xffffffffu, tmem_base);
            if (B_RES) mbar_wait(bar_bfull, 0);
            uint32_t s = 0, ph = 0, j = 0, lt = 0, it = 0;
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++lt) {
                const uint32_t acc = lt & 1, aph = (lt >> 1) & 1;
                mbar_wait(bar_tempty + 8 * acc, aph ^ 1);
                const uint32_t d_tmem = tmem_base_u + acc * N;
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    XB_TS(1, it, 0);
                    mbar_wait(bar_conv + 8 * s, ph);          // operand warps arrive after they saw the TMA bytes land
                    XB_TS(1, it, 1);
                    tc_fence_after();
                    const uint32_t st = ring + s * stage_bytes;
                    const uint32_t a_hi = st, a_lo = lo_ring + j * kATile;
                    const uint32_t b_hi = B_RES ? bres + kb * kBTile : st + kATile;
                    const uint32_t b_lo = B_RES ? bres + (KB + kb) * kBTile : st + kATile + kBTile;
#pragma unroll
                    for (int k = 0; k < BK / 8; ++k) {
                        const uint64_t da_hi = umma_desc_sw128(a_hi + k * 32, 16, 1024);
                        const uint64_t da_lo = umma_desc_sw128(a_lo + k * 32, 16, 1024);
                        const uint64_t db_hi = umma_desc_sw128(b_hi + k * 32, 16, 1024);
                        const uint64_t db_lo = umma_desc_sw128(b_lo + k * 32, 16, 1024);
                        mma_tf32_ss_if(elected, d_tmem, da_lo, db_hi, kIdesc, (kb | k) != 0);
                        mma_tf32_ss_if(elected, d_tmem, da_hi, db_lo, kIdesc, 1);
                        mma_tf32_ss_if(elected, d_tmem, da_hi, db_hi, kIdesc, 1);
                    }
                    XB_TS(1, it, 2);
                    mma_commit_if(elected, bar_empty + 8 * s);
                    mma_commit_if(elected, bar_loempty + 8 * j);
                    if (kb == KB - 1) mma_commit_if(elected, bar_tfull + 8 * acc);
                    XB_TS(1, it, 3);
                    if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
                    if (++j == (uint32_t)L) j = 0;
                }
            }
        }
    } else if (warp >= 4) {
        // ============================================================ operand warps (256 threads)
        const int t = threadIdx.x - 128;
        const int c = t & 7, r0 = t >> 3;                 // logical 16-byte chunk, first row; rows r0 + 32 i
        float* sdout = sf + 1024;                          // DGRAD: [2 tile parities][128 rows][2 src][2 heads]
        uint32_t s = 0, ph = 0, j = 0, jph = 0, lt = 0, it = 0;
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++lt) {
            if (MODE == MODE_DGRAD) {
                if (t < BM) {
                    const int64_t row = tile * BM + t;
                    float* d = sdout + (lt & 1) * 512 + t * 4;
                    const bool ok = row < p.M;
                    d[0] = (ok && p.nh0 > 0) ? p.dout0[row * p.nh0] : 0.f;
                    d[1] = (ok && p.nh0 > 1) ? p.dout0[row * p.nh0 + 1] : 0.f;
                    d[2] = (ok && p.nh1 > 0) ? p.dout1[row * p.nh1] : 0.f;
                    d[3] = (ok && p.nh1 > 1) ? p.dout1[row * p.nh1 + 1] : 0.f;
                }
                bar_sync_named(1, kOperandWarps * 32);
            }
            for (int kb = 0; kb < KB; ++kb, ++it) {
                mbar_wait(bar_full + 8 * s, ph);
                if (t == 0) XB_TS(2, it, 0);
                mbar_wait(bar_loempty + 8 * j, jph ^ 1);
                if (t == 0) XB_TS(2, it, 1);
                const uint32_t a_raw = ring + s * stage_bytes, a_lo = lo_ring + j * kATile;
                float w0[4] = {0, 0, 0, 0}, w1[4] = {0, 0, 0, 0};
                int src = 0;
                if (MODE == MODE_DGRAD) {
                    src = kb >= p.kb_split;
                    const int kcol = (src ? kb - p.kb_split : kb) * BK + 4 * c;
                    const float* w = sf + src * 512 + kcol;
#pragma unroll
                    for (int q = 0; q < 4; ++q) { w0[q] = w[q]; w1[q] = w[256 + q]; }
                }
                float4 xs[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) xs[i] = lds128(a_raw + sw128_off(r0 + 32 * i, c));
                if (MODE == MODE_DGRAD && p.mask_form) {
                    // rank-1 head gradients: the operand is e[r] (y > 0) or slope * e[r], split once per row
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int r = r0 + 32 * i;
                        const uint32_t off = sw128_off(r, c);
                        const float e = sdout[(lt & 1) * 512 + r * 4 + src * 2];
                        float ph, pl, qh, ql;
                        split_tf32(e, ph, pl);
                        split_tf32(e * p.slope, qh, ql);
                        const float4 x = xs[i];
                        sts128(a_raw + off, make_float4(x.x > 0.f ? ph : qh, x.y > 0.f ? ph : qh, x.z > 0.f ? ph : qh, x.w > 0.f ? ph : qh));
                        sts128(a_lo + off, make_float4(x.x > 0.f ? pl : ql, x.y > 0.f ? pl : ql, x.z > 0.f ? pl : ql, x.w > 0.f ? pl : ql));
                    }
                } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = r0 + 32 * i;
                    const uint32_t off = sw128_off(r, c);
                    float4 x = xs[i];
                    if (MODE == MODE_DGRAD) {
                        const float* d = sdout + (lt & 1) * 512 + r * 4 + src * 2;
                        const float d0 = d[0], d1 = d[1];
                        x.x = (d0 * w0[0] + d1 * w1[0]) * (x.x > 0.f ? 1.f : p.slope);
                        x.y = (d0 * w0[1] + d1 * w1[1]) * (x.y > 0.f ? 1.f : p.slope);
                        x.z = (d0 * w0[2] + d1 * w1[2]) * (x.z > 0.f ? 1.f : p.slope);
                        x.w = (d0 * w0[3] + d1 * w1[3]) * (x.w > 0.f ? 1.f : p.slope);
                    }
                    float4 hi, lo;
                    split_tf32(x.x, hi.x, lo.x);
                    split_tf32(x.y, hi.y, lo.y);
                    split_tf32(x.z, hi.z, lo.z);
                    split_tf32(x.w, hi.w, lo.w);
                    sts128(a_raw + off, hi);
                    sts128(a_lo + off, lo);
                }
                }
                if (t == 0) XB_TS(2, it, 2);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_conv + 8 * s);
                if (t == 0) XB_TS(2, it, 3);
                if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
                if (++j == (uint32_t)L) { j = 0; jph ^= 1; }
            }
        }
    } else {
        // ============================================================ epilogue warps 0-3
        EpiCtx c;
        c.tmem_base = tmem_base; c.bar_tfull = bar_tfull; c.bar_tempty = bar_tempty; c.bar_h1w = bar_h1w;
        c.out_ring = out_ring; c.h1_ring = h1_ring; c.O = O; c.HB = HB;
        c.tile0 = tile0; c.tile_step = tile_step; c.n_tiles = n_tiles; c.M = p.M;
        c.map_out = map_out; c.map_h1 = map_h1; c.sf = sf; c.slope = p.slope;
        c.n_head = e_n_head; c.head_b = e_head_b; c.head_out = e_head_out;
        c.store_y = MODE != MODE_FWD || p.Y != nullptr;
        c.n_off = 0;
        c.loss = p.loss; c.sel = sel; c.red = reinterpret_cast<double*>(misc_ptr + kLossRedOff);
        c.sign_out = (MODE == MODE_FWD && p.sign_out) ? p.sign_out + sel * (N / 32) : nullptr;
        c.sign_ld = p.sign_ld;
        c.h1_signs = nullptr;
#ifdef XB_DENSE_TS
        c.ts = p.ts;
#endif
        if (MODE == MODE_FWD) prep_dgrad_operand(p, threadIdx.x);      // idle until the first accumulator is ready
        epilogue_warp<N, MODE>(c, warp, lane);
    }

    // ---------------------------------------------------------------- teardown
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc<kTmemCols>(tmem_base);
    }
    if (MODE == MODE_FWD)
        fused_loss_finish(p.loss, reinterpret_cast<const double*>(misc_ptr + kLossRedOff),
                          reinterpret_cast<bool*>(misc_ptr + kLossRedOff + 256));
}

// ---------------------------------------------------------------------------------------------- weight preparation
// W [N][K] row-major -> hi/lo [N][K] (forward operand) and, transposed, hi/lo rows of Wt [K][ldt] at column offset
// `toff` (dgrad operand: dX = dZ . W needs W^T K-major; actor and critic are concatenated along the reduction dim).
struct SplitJob {
    const float* W;
    float* hi;
    float* lo;
    int toff;
};
__global__ void split_weights_kernel(SplitJob j0, SplitJob j1, int N, int K, float* __restrict__ thi,
                                     float* __restrict__ tlo, int ldt) {
    const SplitJob j = blockIdx.y ? j1 : j0;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * K || !j.W) return;
    const int n = i / K, k = i - n * K;
    float h, l;
    split_tf32(j.W[i], h, l);
    j.hi[i] = h;
    j.lo[i] = l;
    if (thi) {
        thi[(int64_t)k * ldt + j.toff + n] = h;
        tlo[(int64_t)k * ldt + j.toff + n] = l;
    }
}

template <int N, bool B_RES, int MODE>
static int launch_kmajor(const TMaps& maps, KParams p, cudaStream_t s) {
    const int kBTile = N * BK * 4;
    const int bres = B_RES ? 2 * p.KB * kBTile : 0;
    const int stage = kATile + (B_RES ? 0 : 2 * kBTile);
    const int avail = kMaxSmem - 1024 - kMiscBytes - bres;
    // minimum: 2 raw stages, 1 lo buffer, 1 staging tile (+ 1 mask tile); then deepen in order of measured benefit
    int S = 2, L = 1, O = 1, HB = MODE == MODE_DGRAD ? 1 : 0;
    auto bytes = [&]() { return S * stage + (L + O + HB) * kATile; };
    if (bytes() > avail) return XB_E_UNSUPPORTED;
    ++L; if (bytes() > avail) --L;
    if (MODE == MODE_DGRAD) { ++HB; if (bytes() > avail) --HB; }
    ++O; if (bytes() > avail) --O;
    while (S < 4) { ++S; if (bytes() > avail) { --S; break; } }
    p.stages = S;
    p.lo_bufs = L;
    p.out_bufs = O;
    p.h1_bufs = HB;
#ifdef XB_DENSE_TS
    p.ts = g_xb_ts_host;
#endif
    const int smem = 1024 + bres + bytes() + kMiscBytes;
    auto kern = dense_kmajor_kernel<N, B_RES, MODE>;
    XB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));   // per device, cheap: set on every launch
    const int64_t tiles = (p.M + BM - 1) / BM;
    const int n_src = MODE == MODE_FWD ? (p.dual ? 2 : 1) : (p.n_split > 1 ? p.n_split : 1);
    const int64_t want = tiles * n_src;
    const int grid = (int)(want < kNumSMs ? want : (kNumSMs / n_src) * n_src);
    kern<<<grid, kThreads, smem, s>>>(maps, p);
    XB_LAUNCH_CHECK();
    return 0;
}

// ================================================================================================ TS variant
// Same kernels with the A operand in TENSOR MEMORY (tcgen05.mma "TS" form) for N <= 128.  The SS form above is bound
// by shared-memory bandwidth: every M=128 x N=128 x K=8 MMA streams 4 KB of A and 4 KB of B out of shared memory in
// its 64 cycles (the full 128 B/clk), on top of the operand warps' own hi/lo traffic.  Here the operand warps read the
// raw tile once (row per thread, un-swizzling as they go), split it in registers and tcgen05.st the hi/lo halves into
// a 4-deep ring of TMEM columns; the MMAs then read only B from shared memory, the raw stage is released as soon as it
// has been read (not when the MMAs retire), and the lo ring disappears from shared memory.
// TMEM budget (512 columns): accumulator 2 x N | A ring 4 x (32 hi + 32 lo).
constexpr int kTA = 4;                    // TMEM A-operand stages

// Split-phase mbarrier checks for the operand warps: `XB_TRYWAIT_ISSUE(P, bar, parity)` issues a NON-BLOCKING phase check
// (test_wait: try_wait would suspend the warp right there when the phase is not complete yet) into the
// function-scope predicate register P (declared once with XB_DECLARE_PREDS at the top of the kernel) and returns at once;
// `xb_trywait_result_P()` consumes it later.  Independent work placed in between hides the ~250-cycle latency of the
// check; a false result (phase not complete yet) falls back to the blocking wait.
// timing experiment only (-DXB_HACK_MMA2: WRONG results): drop the hi x hi MMA of every k-step to measure what a 2-MMA form would cost
#ifdef XB_HACK_MMA2
#define XB_MMA3(s) ""
#else
#define XB_MMA3(s) s
#endif
#define XB_DECLARE_PREDS() asm volatile(".reg .pred xb_pf, xb_pa;")
#define XB_TRYWAIT_ISSUE(P, bar, parity) \
    asm volatile("mbarrier.test_wait.parity.shared::cta.b64 " #P ", [%0], %1;" ::"r"(bar), "r"(parity) : "memory")
#define XB_TRYWAIT_RESULT(P, out) asm volatile("selp.u32 %0, 1, 0, " #P ";" : "=r"(out)::"memory")
constexpr int kTsTmemCols = 512;

__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const float (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
        "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// One k-block of the TS main loop issued by the MMA thread as a single instruction stream: non-blocking phase checks
// (test_wait) of the NEXT k-block's barriers are issued first and only consumed after the 12 MMAs and the commits, so their ~300-cycle
// latency (measured: passing an already-complete mbarrier) overlaps MMA issue instead of idling the tensor pipe.
// Returns a bit mask: 1 = next A stage ready, 2 = next B stage ready.
__device__ __forceinline__ uint32_t ts_kblock(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint64_t db_hi,
                                              uint64_t db_lo, uint32_t idesc, uint32_t accumulate_first,
                                              uint32_t next_bar_a, uint32_t next_par_a, uint32_t next_bar_b,
                                              uint32_t next_par_b, uint32_t commit0, uint32_t commit1, uint32_t commit2,
                                              uint32_t elected) {
    uint32_t ready;
    asm volatile(
        "{\n"
        ".reg .pred pa, pb, p0, p1, c1, c2, pe;\n"
        "setp.ne.b32 pe, %15, 0;\n"
        ".reg .b32 ah, al, r;\n"
        ".reg .b64 bh, bl;\n"
        "setp.ne.b32 p0, %7, 0;\n"
        "setp.ne.b32 p1, 1, 0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [%3], %4, %6, p0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [%2], %5, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [%2], %4, %6, p1;\n")
        "add.u32 ah, %2, 8;  add.u32 al, %3, 8;  add.u64 bh, %4, 2;  add.u64 bl, %5, 2;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [al], bh, %6, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bl, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bh, %6, p1;\n")
        // the NEXT k-block's phase checks go out in the middle of the MMA stream (timelines: issued in front of it they
        // mostly come back "not yet" — the operand warps run less than one k-block ahead — and the blocking re-check then
        // costs ~300 cycles in which the tensor pipe drains; issued here the remaining six MMAs still cover their latency)
        "mbarrier.test_wait.parity.shared::cta.b64 pa, [%8], %9;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 pb, [%10], %11;\n"
        "add.u32 ah, %2, 16; add.u32 al, %3, 16; add.u64 bh, %4, 4;  add.u64 bl, %5, 4;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [al], bh, %6, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bl, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bh, %6, p1;\n")
        "add.u32 ah, %2, 24; add.u32 al, %3, 24; add.u64 bh, %4, 6;  add.u64 bl, %5, 6;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [al], bh, %6, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bl, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bh, %6, p1;\n")
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%12];\n"
        "setp.ne.b32 c1, %13, 0;\n"
        "setp.ne.b32 c2, %14, 0;\n"
        "and.pred c1, c1, pe;\n"
        "and.pred c2, c2, pe;\n"
        "@c1 tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%13];\n"
        "@c2 tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%14];\n"
        "selp.u32 %0, 1, 0, pa;\n"
        "selp.u32 r, 2, 0, pb;\n"
        "or.b32 %0, %0, r;\n"
        "}\n"
        : "=r"(ready)
        : "r"(d_tmem), "r"(a_hi), "r"(a_lo), "l"(db_hi), "l"(db_lo), "r"(idesc), "r"(accumulate_first), "r"(next_bar_a),
          "r"(next_par_a), "r"(next_bar_b), "r"(next_par_b), "r"(commit0), "r"(commit1), "r"(commit2), "r"(elected)
        : "memory");
    return ready;
}

#ifdef XB_DENSE_TS
__device__ __forceinline__ uint32_t ts_kblock_timed(long long* tq, uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint64_t db_hi,
                                              uint64_t db_lo, uint32_t idesc, uint32_t accumulate_first,
                                              uint32_t next_bar_a, uint32_t next_par_a, uint32_t next_bar_b,
                                              uint32_t next_par_b, uint32_t commit0, uint32_t commit1, uint32_t commit2,
                                              uint32_t elected) {
    uint32_t ready;
    long long t1, t2, t3;
    asm volatile(
        "{\n"
        ".reg .pred pa, pb, p0, p1, c1, c2, pe;\n"
        "setp.ne.b32 pe, %18, 0;\n"
        ".reg .b32 ah, al, r;\n"
        ".reg .b64 bh, bl;\n"
        "setp.ne.b32 p0, %10, 0;\n"
        "setp.ne.b32 p1, 1, 0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [%6], %7, %9, p0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [%5], %8, %9, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [%5], %7, %9, p1;\n")
        "add.u32 ah, %5, 8;  add.u32 al, %6, 8;  add.u64 bh, %7, 2;  add.u64 bl, %8, 2;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [al], bh, %9, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [ah], bl, %9, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [ah], bh, %9, p1;\n")
        // the NEXT k-block's phase checks go out in the middle of the MMA stream (timelines: issued in front of it they
        // mostly come back "not yet" — the operand warps run less than one k-block ahead — and the blocking re-check then
        // costs ~300 cycles in which the tensor pipe drains; issued here the remaining six MMAs still cover their latency)
        "mov.u64 %1, %%clock64;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 pa, [%11], %12;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 pb, [%13], %14;\n"
        "add.u32 ah, %5, 16; add.u32 al, %6, 16; add.u64 bh, %7, 4;  add.u64 bl, %8, 4;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [al], bh, %9, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [ah], bl, %9, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [ah], bh, %9, p1;\n")
        "add.u32 ah, %5, 24; add.u32 al, %6, 24; add.u64 bh, %7, 6;  add.u64 bl, %8, 6;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [al], bh, %9, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [ah], bl, %9, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%4], [ah], bh, %9, p1;\n")
        "mov.u64 %2, %%clock64;\n"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%15];\n"
        "setp.ne.b32 c1, %16, 0;\n"
        "setp.ne.b32 c2, %17, 0;\n"
        "and.pred c1, c1, pe;\n"
        "and.pred c2, c2, pe;\n"
        "@c1 tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%16];\n"
        "@c2 tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%17];\n"
        "mov.u64 %3, %%clock64;\n"
        "selp.u32 %0, 1, 0, pa;\n"
        "selp.u32 r, 2, 0, pb;\n"
        "or.b32 %0, %0, r;\n"
        "}\n"
        : "=r"(ready), "=l"(t1), "=l"(t2), "=l"(t3)
        : "r"(d_tmem), "r"(a_hi), "r"(a_lo), "l"(db_hi), "l"(db_lo), "r"(idesc), "r"(accumulate_first), "r"(next_bar_a),
          "r"(next_par_a), "r"(next_bar_b), "r"(next_par_b), "r"(commit0), "r"(commit1), "r"(commit2), "r"(elected)
        : "memory");
    if (tq) { tq[4] = t1; tq[5] = t2; tq[6] = t3; }
    return ready;
}

#endif

template <int N, bool B_RES, int MODE>
__global__ void __launch_bounds__(kThreads, 1)
    dense_kmajor_ts_kernel(const __grid_constant__ TMaps maps, const KParams p) {
    static_assert(N <= 128, "TS variant: accumulators (2N) + A ring (256) must fit the 512 TMEM columns");
    constexpr int kBTile = N * BK * 4;
    constexpr uint32_t kIdesc = umma_idesc_tf32(BM, N, 0, 0);
    constexpr uint32_t kACol = 2 * N;                   // first TMEM column of the A ring
    extern __shared__ unsigned char smem_raw[];
    XB_DECLARE_PREDS();
    // programmatic dependent launch: with `pdl_early` (the caller vouches that the launch before this one writes no weights)
    // the set-up below and the resident-weight loads overlap that launch; everything else starts after pdl_wait()
    const bool pdl_early = MODE == MODE_FWD && p.pdl_early != 0;
#ifdef XB_STEP_TS
    unsigned long long* const sts = (blockIdx.x == 0 && threadIdx.x == 0 && MODE == MODE_FWD && p.obs) ? p.sts : nullptr;
#endif
    XB_STEP_STAMP(sts, 200);
    if (threadIdx.x == 0) XB_TS(0, 62, 0);
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int S = p.stages, SB = p.lo_bufs, O = p.out_bufs, HB = p.h1_bufs, KB = p.KB;   // lo_bufs doubles as B-ring depth
    const uint32_t bres = base;                                              // [2][KB][kBTile] when B_RES
    const uint32_t ring = base + (B_RES ? 2u * KB * kBTile : 0u);            // raw A tiles
    const uint32_t b_ring = ring + (uint32_t)S * kATile;                     // streamed weight k-blocks (hi | lo)
    const uint32_t out_ring = b_ring + (B_RES ? 0u : (uint32_t)SB * 2 * kBTile);
    const uint32_t h1_ring = out_ring + (uint32_t)O * kATile;
    const uint32_t misc = h1_ring + (MODE == MODE_DGRAD ? (uint32_t)HB * kATile : 0u);
    const uint32_t bar_full = misc, bar_conv = misc + 64, bar_empty = misc + 128, bar_aempty = misc + 192;
    const uint32_t bar_tfull = misc + 224, bar_tempty = misc + 240, bar_bfull = misc + 256;
    // (sign-word DGRAD: no raw ring, so the weight ring takes the raw ring's 8 + 8 barrier slots and may be up to 8 deep)
    const bool no_raw_k = MODE == MODE_DGRAD && p.signs != nullptr;
    const uint32_t tmem_slot = misc + 264, bar_h1w = misc + 352;
    const uint32_t bar_bfull_r = no_raw_k ? misc : misc + 288, bar_bempty = no_raw_k ? misc + 128 : misc + 320;
    unsigned char* misc_ptr = smem_raw + (misc - smem_u32(smem_raw));
    float* sf = reinterpret_cast<float*>(misc_ptr + 512);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_tiles = (p.M + BM - 1) / BM;
    // FWD dual: CTA parity selects the layer.  DGRAD n_split: CTA parity selects which N-column slice of the output
    // (and which weight rows) this CTA owns.  Either way the CTAs of a group walk the same tiles.
    const int n_src = MODE == MODE_FWD ? (p.dual ? 2 : 1) : (p.n_split > 1 ? p.n_split : 1);
    const int part = (int)(blockIdx.x % n_src);
    const int sel = MODE == MODE_FWD ? part : 0;
    const int n_off = MODE == MODE_DGRAD ? part * N : 0;
    const int64_t tile0 = blockIdx.x / n_src, tile_step = gridDim.x / n_src;
    const CUtensorMap* map_a0 = &maps.a0;
    const CUtensorMap* map_a1 = &maps.a1;
    const CUtensorMap* map_bhi = sel ? &maps.bhi1 : &maps.bhi;
    const CUtensorMap* map_blo = sel ? &maps.blo1 : &maps.blo;
    const CUtensorMap* map_out = sel ? &maps.out1 : &maps.out;
    const CUtensorMap* map_h1 = &maps.h1;
    const float* e_bias = sel ? p.bias1 : p.bias;
    const float* e_head_w = sel ? p.head_w1 : p.head_w;
    const float* e_head_b = sel ? p.head_b1 : p.head_b;
    const int e_n_head = sel ? p.n_head1 : p.n_head;
    float* e_head_out = sel ? p.head_out1 : p.head_out;
    // FWD without a stored Y (rollout, rank-1 training): the operand warps take part of every tile's epilogue, with the
    // idle staging ring holding their head terms
    const int epi_sets = (MODE == MODE_FWD && p.Y == nullptr) ? epi_sets_of<N>() : 1;

    if (threadIdx.x == 0) {
        const int n_conv = p.alt_groups ? kOperandWarps / 2 : kOperandWarps;    // operand warps per k-block
        for (int s = 0; s < S; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, n_conv);                 // released by the operand warps once they have read it
        }
        for (int a = 0; a < kTA; ++a) {
            mbar_init(bar_conv + 8 * a, n_conv);
            mbar_init(bar_aempty + 8 * a, 1);
        }
        for (int b = 0; b < (no_raw_k ? 8 : 4); ++b) {
            mbar_init(bar_bfull_r + 8 * b, 1);
            mbar_init(bar_bempty + 8 * b, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull + 8 * a, 1);
            mbar_init(bar_tempty + 8 * a, 4 * epi_sets);
        }
        for (int a = 0; a < 8; ++a) mbar_init(bar_h1w + 8 * a, 1);
        mbar_init(bar_bfull, 1);
        mbar_fence_init();
    }
    if (warp == kMmaWarp) tmem_alloc<kTsTmemCols>(tmem_slot);
    if (!pdl_early) pdl_wait();           // (barriers and tensor memory above: no global data touched)
    if (MODE == MODE_FWD) {
        for (int i = threadIdx.x; i < N; i += kThreads) {
            sf[i] = e_bias ? e_bias[i] : 0.f;
            sf[N + i] = e_n_head > 0 ? e_head_w[i] : 0.f;
            sf[2 * N + i] = e_n_head > 1 ? e_head_w[N + i] : 0.f;
        }
        if (p.obs) {    // trunk parameters: sf[3N + i*K + k] = W0[k][i] (i < obs_dim), sf[3N + 4K + k] = b0[k]
            const int K = KB * BK;
            for (int i = threadIdx.x; i < 5 * K; i += kThreads) {
                const int d = i / K, kk = i - d * K;
                sf[3 * N + i] = d == 4 ? p.b0[kk] : (d < p.obs_dim ? p.W0[kk * p.obs_dim + d] : 0.f);
            }
        }
    } else {
        const int K0 = p.kb_split * BK, K1 = (KB - p.kb_split) * BK;
        for (int i = threadIdx.x; i < 256; i += kThreads) {
            sf[i] = (i < K0 && p.nh0 > 0) ? p.w2_0[i] : 0.f;
            sf[256 + i] = (i < K0 && p.nh0 > 1) ? p.w2_0[K0 + i] : 0.f;
            sf[512 + i] = (i < K1 && p.nh1 > 0) ? p.w2_1[i] : 0.f;
            sf[768 + i] = (i < K1 && p.nh1 > 1) ? p.w2_1[K1 + i] : 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    if (threadIdx.x == 0) XB_TS(0, 62, 1);
    const bool is_producer = warp == kProducerWarp;     // (the whole warp: it walks the producer loop converged)
    if (!is_producer) {
        XB_STEP_STAMP(sts, 201);
        if (pdl_early) pdl_wait();
        XB_STEP_STAMP(sts, 202);
        pdl_trigger();
    }
    // epilogue context: warps 0-3, and with epi_sets > 1 the operand warps' share of it (built inside each role's branch)
    auto epi_ctx = [&]() {
        EpiCtx c;
        c.tmem_base = tmem_base; c.bar_tfull = bar_tfull; c.bar_tempty = bar_tempty; c.bar_h1w = bar_h1w;
        c.out_ring = out_ring; c.h1_ring = h1_ring; c.O = O; c.HB = HB;
        c.tile0 = tile0; c.tile_step = tile_step; c.n_tiles = n_tiles; c.M = p.M;
        c.map_out = map_out; c.map_h1 = map_h1; c.sf = sf; c.slope = p.slope;
        c.n_head = e_n_head; c.head_b = e_head_b; c.head_out = e_head_out;
        c.store_y = MODE != MODE_FWD || p.Y != nullptr;
        c.n_off = n_off;
        c.loss = p.loss; c.sel = sel; c.red = reinterpret_cast<double*>(misc_ptr + kLossRedOff);
        c.sign_out = (MODE == MODE_FWD && p.sign_out) ? p.sign_out + sel * (N / 32) : nullptr;
        c.sign_ld = p.sign_ld;
        c.h1_signs = (MODE == MODE_DGRAD && N == 128 && p.n_split <= 1) ? p.h1_signs : nullptr;
        c.epi_sets = epi_sets;
        c.head_terms = out_ring;      // (unused staging when Y is not stored: [N/32 - own chunks][8][128] float2 <= kATile)
#ifdef XB_DENSE_TS
        c.ts = p.ts;
#endif
        return c;
    };

    if (warp == kProducerWarp) {
        // ============================================================ TMA producer: the whole warp walks the loop, one elected
        // lane issues (uniform operands: no R2UR waterfall around every UTMALDG, see tma_load_2d_if)
        {
            const uint32_t elected = elect_one_pred();
            if (lane == 0) {
                tma_prefetch_desc(map_a0);
                tma_prefetch_desc(map_bhi);
                tma_prefetch_desc(map_blo);
                if (MODE == MODE_DGRAD) tma_prefetch_desc(map_a1);
            }
            __syncwarp();
            if (B_RES) {
                mbar_arrive_expect_tx_if(elected, bar_bfull, 2u * KB * kBTile);
                for (int kb = 0; kb < KB; ++kb) {
                    tma_load_2d_if(elected, bres + kb * kBTile, map_bhi, kb * BK, n_off, bar_bfull);
                    tma_load_2d_if(elected, bres + (KB + kb) * kBTile, map_blo, kb * BK, n_off, bar_bfull);
                }
            }
            if (pdl_early) pdl_wait();          // (the resident weights are on their way; activations only from here)
            pdl_trigger();
            uint32_t s = 0, ph = 0, sb = 0, bph = 0, it = 0;
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_step) {
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    if (!(MODE == MODE_FWD && p.obs) && !(MODE == MODE_DGRAD && p.signs)) {
                        mbar_wait(bar_empty + 8 * s, ph ^ 1);
                        XB_TS(0, it, 0);
                        mbar_arrive_expect_tx_if(elected, bar_full + 8 * s, kATile);
                        const bool src1 = (MODE == MODE_DGRAD) && kb >= p.kb_split;
                        const int kcol = (src1 ? kb - p.kb_split : kb) * BK;
                        tma_load_2d_if(elected, ring + s * kATile, src1 ? map_a1 : map_a0, kcol, (int)(tile * BM), bar_full + 8 * s);
                        if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
                    }
                    if (!B_RES) {
                        mbar_wait(bar_bempty + 8 * sb, bph ^ 1);
                        const uint32_t bs = b_ring + sb * 2 * kBTile;
                        mbar_arrive_expect_tx_if(elected, bar_bfull_r + 8 * sb, 2 * kBTile);
                        tma_load_2d_if(elected, bs, map_bhi, kb * BK, n_off, bar_bfull_r + 8 * sb);
                        tma_load_2d_if(elected, bs + kBTile, map_blo, kb * BK, n_off, bar_bfull_r + 8 * sb);
                        if (++sb == (uint32_t)SB) { sb = 0; bph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ============================================================ MMA issuer
        // The WHOLE warp walks the loop and one elected lane issues: with the loop inside `if (lane == 0)` every descriptor /
        // address operand of tcgen05.mma lives in a per-thread register and ptxas wraps each instruction in an ELECT + 4 x
        // R2UR.BROADCAST "waterfall" (~80 cycles per MMA in the issuing thread — more than the 64 cycles the MMA itself takes:
        // the timelines' real limiter).  Warp-uniform operands go through the uniform datapath instead.
        {
            const uint32_t elected = elect_one_pred();
            const uint32_t tmem_base_u = __reduce_max_sync(0xffffffffu, tmem_base);     // same value, provably warp-uniform
            if (B_RES) mbar_wait(bar_bfull, 0);
            // a barrier/parity pair that always tests complete, for the unused prefetch slot
            const uint32_t dummy_bar = bar_bfull, dummy_par = B_RES ? 0u : 1u;
            uint32_t ta = 0, aph = 0, sb = 0, bph = 0, lt = 0, it = 0;
            uint32_t ready = 0;                             // bit 0: A stage `ta` known ready, bit 1: B stage `sb`
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++lt) {
                const uint32_t acc = lt & 1, tph = (lt >> 1) & 1;
                mbar_wait(bar_tempty + 8 * acc, tph ^ 1);
                const uint32_t d_tmem = tmem_base_u + acc * N;
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    XB_TS(1, it, 0);
                    if (!(ready & 1)) mbar_wait(bar_conv + 8 * ta, aph);
                    if (!B_RES && !(ready & 2)) mbar_wait(bar_bfull_r + 8 * sb, bph);
                    XB_TS(1, it, 1);
                    tc_fence_after();
                    const uint32_t a_hi = tmem_base_u + kACol + ta * 64, a_lo = a_hi + 32;
                    const uint32_t b_hi = B_RES ? bres + kb * kBTile : b_ring + sb * 2 * kBTile;
                    const uint32_t b_lo = B_RES ? bres + (KB + kb) * kBTile : b_hi + kBTile;
                    // next k-block's stages (the tile boundary does not matter: the rings run continuously)
                    const uint32_t nta = ta + 1 == kTA ? 0 : ta + 1, naph = ta + 1 == kTA ? aph ^ 1 : aph;
                    const uint32_t nsb = sb + 1 == (uint32_t)SB ? 0 : sb + 1, nbph = sb + 1 == (uint32_t)SB ? bph ^ 1 : bph;
#ifdef XB_DENSE_TS
                    ready = ts_kblock_timed((p.ts && blockIdx.x == 0 && it < 64) ? p.ts + (1 * 64 + it) * 8 : nullptr,
                                      d_tmem, a_hi, a_lo, umma_desc_sw128(b_hi, 16, 1024), umma_desc_sw128(b_lo, 16, 1024),
#else
                    ready = ts_kblock(d_tmem, a_hi, a_lo, umma_desc_sw128(b_hi, 16, 1024), umma_desc_sw128(b_lo, 16, 1024),
#endif
                                      kIdesc, kb != 0, bar_conv + 8 * nta, naph, B_RES ? dummy_bar : bar_bfull_r + 8 * nsb,
                                      B_RES ? dummy_par : nbph, bar_aempty + 8 * ta, B_RES ? 0u : bar_bempty + 8 * sb,
                                      kb == KB - 1 ? bar_tfull + 8 * acc : 0u, elected);
                    XB_TS(1, it, 3);
                    ta = nta; aph = naph;
                    if (!B_RES) { sb = nsb; bph = nbph; }
                }
            }
        }
    } else if (warp >= 4) {
        // ============================================================ operand warps (256 threads): raw tile -> TMEM
        const int lq = warp & 3, ch = (warp - 4) >> 2;    // TMEM lane quarter (warp % 4), half of the 32 k-columns
        const int r = 32 * lq + lane;                     // row of the tile = TMEM lane
        const uint32_t lane_base = (uint32_t)(32 * lq) << 16;
        uint32_t s = 0, ph = 0, ta = 0, aph = 0, it = 0;
        const bool from_bits = MODE == MODE_DGRAD && p.signs != nullptr;    // activation sign words instead of activation tiles
        const bool from_obs = (MODE == MODE_FWD && p.obs != nullptr) || from_bits;   // = no raw A ring: the operand is generated
        const bool alt = p.alt_groups != 0;     // ch is then the GROUP (k-block parity) instead of the column half
        // epilogue set 1 + ch: its share of tile t runs once tile t + 1's k-blocks are converted (the last tile's at the end)
        const bool epi_share = MODE == MODE_FWD && 1 + ch < epi_sets;
        uint32_t elt = 0;
        if (!from_obs && !alt && tile0 < n_tiles) XB_TRYWAIT_ISSUE(xb_pf, bar_full + 8 * s, ph);    // first stage's phase check
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_step) {
            float d00 = 0.f, d01 = 0.f, d10 = 0.f, d11 = 0.f;   // DGRAD: dL/d(head outputs) of this row
            if (MODE == MODE_DGRAD) {
                const int64_t row = tile * BM + r;
                if (row < p.M) {
                    d00 = p.nh0 > 0 ? __ldg(p.dout0 + row * p.nh0) : 0.f;
                    d01 = p.nh0 > 1 ? __ldg(p.dout0 + row * p.nh0 + 1) : 0.f;
                    d10 = p.nh1 > 0 ? __ldg(p.dout1 + row * p.nh1) : 0.f;
                    d11 = p.nh1 > 1 ? __ldg(p.dout1 + row * p.nh1 + 1) : 0.f;
                }
            }
            // mask form: hi/lo of e_s and slope * e_s for this row (e_s = the source's first head gradient)
            float m0ph = 0.f, m0pl = 0.f, m0qh = 0.f, m0ql = 0.f, m1ph = 0.f, m1pl = 0.f, m1qh = 0.f, m1ql = 0.f;
            if (MODE == MODE_DGRAD && p.mask_form) {
                split_tf32(d00, m0ph, m0pl);
                split_tf32(d00 * p.slope, m0qh, m0ql);
                split_tf32(d10, m1ph, m1pl);
                split_tf32(d10 * p.slope, m1qh, m1ql);
            }
            uint32_t sw[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};       // from_bits: this row's sign words (KB <= 8)
            if (from_bits) {
                const int64_t row = tile * BM + r;
                if (row < p.M) {
                    const uint32_t* sp = p.signs + row * KB;
#pragma unroll
                    for (int j = 0; j < 8; ++j) sw[j] = j < KB ? __ldg(sp + j) : 0u;
                }
            }
            float o4[4] = {0.f, 0.f, 0.f, 0.f};
            if (MODE == MODE_FWD && from_obs) {
                const int64_t row = tile * BM + r;
                if (row < p.M) {
                    for (int i = 0; i < p.obs_dim; ++i) o4[i] = __ldg(p.obs + row * p.obs_ld + i);
                    if (p.norm_new) {      // raw observations in: normalise in front of the trunk (agent.py:112-113)
                        const double* st = row < p.norm_rows ? p.norm_new : p.norm_old;
                        for (int i = 0; i < p.obs_dim; ++i) {
                            float mean, den;
                            norm_coeffs(st, 4, i, mean, den);
                            o4[i] = norm_apply(o4[i], mean, den, p.norm_clip);
                        }
                    }
                }
            }
            for (int kb = 0; kb < KB; ++kb, ++it) {
                const uint32_t ns = s + 1 == (uint32_t)S ? 0 : s + 1, nph = s + 1 == (uint32_t)S ? ph ^ 1 : ph;
                if (alt && (it & 1u) != (uint32_t)ch) {      // the other group's k-block
                    if (!from_obs) { s = ns; ph = nph; }
                    if (++ta == kTA) { ta = 0; aph ^= 1; }
                    continue;
                }
                if (alt) {
                    if (!from_obs) mbar_wait(bar_full + 8 * s, ph);
                } else if (!from_obs) {
                    uint32_t ok;
                    XB_TRYWAIT_RESULT(xb_pf, ok);                      // issued one k-block ago
                    if (!ok) mbar_wait(bar_full + 8 * s, ph);
                }
                if (threadIdx.x == 128) XB_TS(2, it, 0);
                const uint32_t a_raw = ring + s * kATile;
                const uint32_t acol0 = tmem_base + lane_base + kACol + ta * 64;
                const int n_half = alt ? 2 : 1;
                for (int hh = 0; hh < n_half; ++hh) {
                    const int chh = alt ? hh : ch;             // which 16 of the 32 k-columns
                    float x[16];
                    uint32_t w16 = 0u;                    // from_bits: the 16 sign bits of this thread's columns
                    if (from_bits) {
                        if (!alt) XB_TRYWAIT_ISSUE(xb_pa, bar_aempty + 8 * ta, aph ^ 1);
                        uint32_t word = sw[0];
#pragma unroll
                        for (int j = 1; j < 8; ++j) word = kb == j ? sw[j] : word;
                        w16 = word >> (16 * chh);
                    } else if (from_obs) {                // trunk layer on the fly: x = leaky(b0 + W0 obs)
                        if (!alt) XB_TRYWAIT_ISSUE(xb_pa, bar_aempty + 8 * ta, aph ^ 1);
                        const int K = KB * BK;
                        const float* w = sf + 3 * N + kb * BK + 16 * chh;
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            float a = w[4 * K + q];
                            a += o4[0] * w[q];
                            a += o4[1] * w[K + q];
                            a += o4[2] * w[2 * K + q];
                            a += o4[3] * w[3 * K + q];
                            x[q] = a > 0.f ? a : a * p.slope;
                        }
                        if (MODE == MODE_FWD && p.h1_out && sel == 0) {     // 64 contiguous bytes of this row's trunk activations
                            const int64_t row = tile * BM + r;
                            if (row < p.M) {
                                float4* dst = reinterpret_cast<float4*>(p.h1_out + row * (int64_t)K + kb * BK + 16 * chh);
#pragma unroll
                                for (int i = 0; i < 4; ++i) dst[i] = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
                            }
                        }
                    } else {
                        float4 xs[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) xs[i] = lds128(a_raw + sw128_off(r, 4 * chh + i));
                        if (!alt) XB_TRYWAIT_ISSUE(xb_pa, bar_aempty + 8 * ta, aph ^ 1);   // overlaps the transform + split below
                        x[0] = xs[0].x; x[1] = xs[0].y; x[2] = xs[0].z; x[3] = xs[0].w;
                        x[4] = xs[1].x; x[5] = xs[1].y; x[6] = xs[1].z; x[7] = xs[1].w;
                        x[8] = xs[2].x; x[9] = xs[2].y; x[10] = xs[2].z; x[11] = xs[2].w;
                        x[12] = xs[3].x; x[13] = xs[3].y; x[14] = xs[3].z; x[15] = xs[3].w;
                    }
                    float hi[16], lo[16];
                    if (MODE == MODE_DGRAD && p.mask_form) {
                        const int src = kb >= p.kb_split;
                        const float ph_ = src ? m1ph : m0ph, pl_ = src ? m1pl : m0pl, qh_ = src ? m1qh : m0qh, ql_ = src ? m1ql : m0ql;
                        if (from_bits) {
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                const bool pos = (w16 >> q) & 1u;
                                hi[q] = pos ? ph_ : qh_;
                                lo[q] = pos ? pl_ : ql_;
                            }
                        } else {
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                const bool pos = x[q] > 0.f;
                                hi[q] = pos ? ph_ : qh_;
                                lo[q] = pos ? pl_ : ql_;
                            }
                        }
                    } else {
                        if (MODE == MODE_DGRAD) {
                            const int src = kb >= p.kb_split;
                            const float* w = sf + src * 512 + (src ? kb - p.kb_split : kb) * BK + 16 * chh;
                            const float e0 = src ? d10 : d00, e1 = src ? d11 : d01;
                            if (from_bits) {
#pragma unroll
                                for (int q = 0; q < 16; ++q) x[q] = (e0 * w[q] + e1 * w[256 + q]) * (((w16 >> q) & 1u) ? 1.f : p.slope);
                            } else {
#pragma unroll
                                for (int q = 0; q < 16; ++q) x[q] = (e0 * w[q] + e1 * w[256 + q]) * (x[q] > 0.f ? 1.f : p.slope);
                            }
                        }
#pragma unroll
                        for (int q = 0; q < 16; ++q) split_tf32(x[q], hi[q], lo[q]);
                    }
                    if (threadIdx.x == 128) XB_TS(2, it, 1);
                    if (hh == 0) {
                        if (alt) {
                            mbar_wait(bar_aempty + 8 * ta, aph ^ 1);
                        } else {
                            uint32_t ok;
                            XB_TRYWAIT_RESULT(xb_pa, ok);
                            if (!ok) mbar_wait(bar_aempty + 8 * ta, aph ^ 1);
                        }
                        if (threadIdx.x == 128) XB_TS(2, it, 2);
                        // the next raw stage's phase check overlaps the TMEM stores below
                        if (!from_obs && !alt) XB_TRYWAIT_ISSUE(xb_pf, bar_full + 8 * ns, nph);
                        tc_fence_after();
                    }
                    tmem_st_32x16(acol0 + 16 * chh, hi);
                    tmem_st_32x16(acol0 + 16 * chh + 32, lo);
                }
                __syncwarp();
                if (lane == 0 && !from_obs) mbar_arrive(bar_empty + 8 * s);   // the raw tile has been consumed: hand the slot back
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_conv + 8 * ta);
                if (threadIdx.x == 128) XB_TS(2, it, 3);
                if (!from_obs) { s = ns; ph = nph; }
                if (++ta == kTA) { ta = 0; aph ^= 1; }
            }
            if (epi_share && tile != tile0) epilogue_share<N>(epi_ctx(), 1 + ch, lq, lane, tile - tile_step, elt++);
        }
        if (epi_share && tile0 < n_tiles) epilogue_share<N>(epi_ctx(), 1 + ch, lq, lane, tile0 + (int64_t)elt * tile_step, elt);
    } else {
        // ============================================================ epilogue warps 0-3
        if (MODE == MODE_FWD) prep_dgrad_operand(p, threadIdx.x);      // idle until the first accumulator is ready
        epilogue_warp<N, MODE>(epi_ctx(), warp, lane);
    }

    if (threadIdx.x == 0) XB_TS(0, 63, 0);
    tc_fence_before();
    __syncthreads();
    XB_STEP_STAMP(sts, 203);
    if (threadIdx.x == 0) XB_TS(0, 63, 1);
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc<kTsTmemCols>(tmem_base);
    }
    if (MODE == MODE_FWD)
        fused_loss_finish(p.loss, reinterpret_cast<const double*>(misc_ptr + kLossRedOff),
                          reinterpret_cast<bool*>(misc_ptr + kLossRedOff + 256));
}

template <int N, bool B_RES, int MODE>
static int launch_kmajor_ts(const TMaps& maps, KParams p, cudaStream_t s) {
    const int kBTile = N * BK * 4;
    const int bres = B_RES ? 2 * p.KB * kBTile : 0;
    const int avail = kMaxSmem - 1024 - kMiscBytes - bres;
    // minimum: 2 raw stages, (2 weight stages), 1 staging tile (+ 1 mask tile); then deepen
    const bool no_raw = MODE == MODE_DGRAD && p.signs != nullptr;    // sign words: no raw A ring, a deeper weight ring instead
    const bool mask_bits = no_raw && p.h1_signs != nullptr && N == 128 && p.n_split <= 1;      // no H1 mask tiles either
    int S = no_raw ? 0 : 2, SB = B_RES ? 0 : 2, O = 1, HB = (MODE == MODE_DGRAD && !mask_bits) ? 1 : 0;
    auto bytes = [&]() { return (S + O + HB) * kATile + SB * 2 * kBTile; };
    if (bytes() > avail) return XB_E_UNSUPPORTED;
    ++O; if (bytes() > avail) --O;
    if (MODE == MODE_DGRAD && !mask_bits) { ++HB; if (bytes() > avail) --HB; }
    while (!no_raw && S < 4) { ++S; if (bytes() > avail) { --S; break; } }
    if (!B_RES) { ++SB; if (bytes() > avail) --SB; }
    // sign-word DGRAD: whatever is left goes to the streamed weight ring (8 barrier slots; L2 -> smem latency ~1.5 k cycles)
    while (!B_RES && no_raw && SB < 8) { ++SB; if (bytes() > avail) { --SB; break; } }
    {   // experiment knobs: XB_DENSE_S / XB_DENSE_O override the ring depths when they fit
        static const int s_env = []() { const char* e = getenv("XB_DENSE_S"); return e ? atoi(e) : 0; }();
        static const int o_env = []() { const char* e = getenv("XB_DENSE_O"); return e ? atoi(e) : 0; }();
        static const int sb_env = []() { const char* e = getenv("XB_DENSE_SB"); return e ? atoi(e) : 0; }();
        static const int hb_env = []() { const char* e = getenv("XB_DENSE_HB"); return e ? atoi(e) : 0; }();
        const int S0 = S, O0 = O, SB0 = SB, HB0 = HB;
        if (!no_raw && s_env >= 2 && s_env <= 4) S = s_env;
        if (o_env >= 1 && o_env <= 4) O = o_env;
        if (!B_RES && sb_env >= 2 && sb_env <= (no_raw ? 8 : 4)) SB = sb_env;
        if (MODE == MODE_DGRAD && !mask_bits && hb_env >= 1 && hb_env <= 2) HB = hb_env;
        if (bytes() > avail) { S = S0; O = O0; SB = SB0; HB = HB0; }
    }
    p.stages = S;
    p.lo_bufs = SB;
    p.out_bufs = O;
    p.h1_bufs = HB;
    static const int alt_env = []() { const char* e = getenv("XB_DENSE_ALT"); return e ? atoi(e) : -1; }();
    p.alt_groups = alt_env >= 0 ? alt_env : (no_raw ? 1 : 0);    // sign-word DGRAD: two groups of 4 operand warps on alternate k-blocks (measured -5 %)
#ifdef XB_DENSE_TS
    p.ts = g_xb_ts_host;
#endif
#ifdef XB_STEP_TS
    p.sts = g_xb_step_ts;
#endif
    const int smem = 1024 + bres + bytes() + kMiscBytes;
    auto kern = dense_kmajor_ts_kernel<N, B_RES, MODE>;
    XB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));   // per device, cheap: set on every launch
    const int64_t tiles = (p.M + BM - 1) / BM;
    const int n_src = MODE == MODE_FWD ? (p.dual ? 2 : 1) : (p.n_split > 1 ? p.n_split : 1);
    const int64_t want = tiles * n_src;
    const int grid = (int)(want < kNumSMs ? want : (kNumSMs / n_src) * n_src);
    XB_CUDA(launch_pdl(kern, dim3(grid), dim3(kThreads), (size_t)smem, s, true, maps, p));
    XB_LAUNCH_CHECK();
    return 0;
}

template <int MODE>
static int dispatch_kmajor(int N, bool bres, const TMaps& maps, const KParams& p_in, cudaStream_t s) {
    const KParams& p = p_in;
    const int kBTile = N * BK * 4;
    static const bool use_ts = []() { const char* e = getenv("XB_DENSE_SS"); return !(e && e[0] == '1'); }();
    if (use_ts && MODE == MODE_DGRAD && p.n_split == 2 && N == 128)      // two CTAs per tile, 64 columns each, weights resident
        return launch_kmajor_ts<64, true, MODE>(maps, p, s);
    if (use_ts && N <= 128) {            // A operand in tensor memory
        if (bres && (kMaxSmem - 1024 - kMiscBytes - 2 * p.KB * kBTile) < (2 + 1 + (MODE == MODE_DGRAD)) * kATile) bres = false;
        if (N == 64)
            return bres ? launch_kmajor_ts<64, true, MODE>(maps, p, s) : launch_kmajor_ts<64, false, MODE>(maps, p, s);
        if (N == 128)
            return bres ? launch_kmajor_ts<128, true, MODE>(maps, p, s) : launch_kmajor_ts<128, false, MODE>(maps, p, s);
        return XB_E_UNSUPPORTED;
    }
    if (bres && (kMaxSmem - 1024 - kMiscBytes - 2 * p.KB * kBTile) < (2 + 1 + 1 + (MODE == MODE_DGRAD)) * kATile) bres = false;
    KParams q = p_in;
    q.signs = nullptr;          // the SS-form DGRAD reads the activation tiles
    q.h1_signs = nullptr;
    switch (N) {
        case 64:
            return bres ? launch_kmajor<64, true, MODE>(maps, q, s) : launch_kmajor<64, false, MODE>(maps, q, s);
        case 128:
            return bres ? launch_kmajor<128, true, MODE>(maps, q, s) : launch_kmajor<128, false, MODE>(maps, q, s);
        case 256:
            return launch_kmajor<256, false, MODE>(maps, q, s);
        default:
            return XB_E_UNSUPPORTED;
    }
}

// ================================================================================================ weight gradients
// dW[m][n] = sum_b dz[b][m] * x[b][n],  db[m] = sum_b dz[b][m]   for the hidden layer of the actor and of the critic,
// plus the narrow head's gradients dw2[j][m] = sum_b dout[b][j] * y[b][m], db2[j] = sum_b dout[b][j].
// The reduction runs over the BATCH, so both MMA operands are "MN-major": a k-block is 32 batch rows, each a 128-byte
// row of 32 features, exactly what TMA delivers from the row-major activations (no transpose anywhere).
// dz is generated on the fly from the saved activation y like in the dgrad kernel; db (and the head gradients) are
// column sums the operand warps keep in registers while they generate dz.
// Grid: CTA i works on job (i % n_jobs) = (source, 128-row half of H_out) and on a contiguous slice of the batch;
// each CTA writes its partial [128][H_in + 4] (column H_in = db) and a deterministic reduce kernel sums the slices.
// One k-block (32 batch rows = 4 k-steps of 8) of the wgrad main loop as a single instruction stream, like ts_kblock:
// the NEXT k-block's conv barrier is tested (non-blocking) before the 12 SS-form MMAs and consumed after the commits.
// All four operand descriptors advance by 1024 B (+64 in descriptor units) per k-step.  Returns 1 if the next k-block's
// operands are already in place.
__device__ __forceinline__ uint32_t ss_kblock_mn(uint32_t d_tmem, uint64_t da_hi, uint64_t da_lo, uint64_t db_hi,
                                                 uint64_t db_lo, uint32_t idesc, uint32_t accumulate_first,
                                                 uint32_t next_bar, uint32_t next_par, uint32_t commit0,
                                                 uint32_t commit1, uint32_t commit2, uint32_t elected) {
    uint32_t ready;
    asm volatile(
        "{\n"
        ".reg .pred pn, p0, p1, c2, pe;\n"
        "setp.ne.b32 pe, %13, 0;\n"
        ".reg .b64 ah, al, bh, bl;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 pn, [%8], %9;\n"
        "setp.ne.b32 p0, %7, 0;\n"
        "setp.ne.b32 p1, 1, 0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], %3, %4, %6, p0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], %2, %5, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], %2, %4, %6, p1;\n")
        "add.u64 ah, %2, 64;  add.u64 al, %3, 64;  add.u64 bh, %4, 64;  add.u64 bl, %5, 64;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], al, bh, %6, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bl, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bh, %6, p1;\n")
        "add.u64 ah, %2, 128; add.u64 al, %3, 128; add.u64 bh, %4, 128; add.u64 bl, %5, 128;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], al, bh, %6, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bl, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bh, %6, p1;\n")
        "add.u64 ah, %2, 192; add.u64 al, %3, 192; add.u64 bh, %4, 192; add.u64 bl, %5, 192;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], al, bh, %6, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bl, %6, p1;\n"
        XB_MMA3("@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bh, %6, p1;\n")
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%10];\n"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%11];\n"
        "setp.ne.b32 c2, %12, 0;\n"
        "and.pred c2, c2, pe;\n"
        "@c2 tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%12];\n"
        "selp.u32 %0, 1, 0, pn;\n"
        "}\n"
        : "=r"(ready)
        : "r"(d_tmem), "l"(da_hi), "l"(da_lo), "l"(db_hi), "l"(db_lo), "r"(idesc), "r"(accumulate_first), "r"(next_bar),
          "r"(next_par), "r"(commit0), "r"(commit1), "r"(commit2), "r"(elected)
        : "memory");
    return ready;
}

struct WParams {
    int64_t B;
    int n_jobs;       // sources x (H_out / 128)
    int halves;       // H_out / 128
    int H_out;
    float slope;
    int stages, lo_bufs;
#ifdef XB_DENSE_TS
    long long* ts;
#endif
    const float* dout[2];
    const float* w2[2];
    int nh[2];
    float* part;       // [grid][128][HIN + 4]
    float* head_part;  // [grid][2][128]   dw2 partial of this CTA's 128 features
    float* db2_part;   // [grid][2]
};

template <int HIN>
__global__ void __launch_bounds__(kThreads, 1)
    dense_wgrad_kernel(const __grid_constant__ CUtensorMap map_y0, const __grid_constant__ CUtensorMap map_y1,
                       const __grid_constant__ CUtensorMap map_x, const WParams p) {
    constexpr int NBX = HIN / 32;                  // 32-feature boxes of x
    constexpr int kBox = 32 * 128;                 // one box: 32 batch rows x 128 B
    constexpr int kStage = 4 * kBox + NBX * kBox;  // dz operand (128 features) | x operand
    constexpr int kTmemCols = HIN;                 // power of two (128 / 256)
    constexpr uint32_t kIdescMain = umma_idesc_tf32(128, HIN, 1, 1);
    extern __shared__ unsigned char smem_raw[];
    if (threadIdx.x == 0) XB_TS(0, 62, 0);
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int S = p.stages, L = p.lo_bufs;
    const uint32_t ring = base, lo_ring = ring + (uint32_t)S * kStage, misc = lo_ring + (uint32_t)L * kStage;
    const uint32_t bar_full = misc, bar_conv = misc + 64, bar_empty = misc + 128, bar_loempty = misc + 192;
    const uint32_t bar_tfull = misc + 224, tmem_slot = misc + 264;
    unsigned char* misc_ptr = smem_raw + (misc - smem_u32(smem_raw));
    float* sf = reinterpret_cast<float*>(misc_ptr + 2048);   // head/bias-gradient reduction scratch: [8 warps][3][128] + [8][2]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int job = blockIdx.x % p.n_jobs, q = blockIdx.x / p.n_jobs;
    const int cj = (gridDim.x - job + p.n_jobs - 1) / p.n_jobs;          // CTAs working on this job
    const int src = job / p.halves, m0 = (job % p.halves) * 128;
    const int64_t nblk = (p.B + 31) / 32;
    const int64_t blk0 = nblk * q / cj, blk1 = nblk * (q + 1) / cj;
    const int nkb = (int)(blk1 - blk0);

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_conv + 8 * s, kOperandWarps / 2);   // one group of 4 operand warps per k-block
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int j = 0; j < L; ++j) mbar_init(bar_loempty + 8 * j, 1);
        mbar_init(bar_tfull, 1);
        mbar_fence_init();
    }
    if (warp == kMmaWarp) tmem_alloc<kTmemCols>(tmem_slot);
    pdl_wait();                           // (set-up above overlaps the launch before this one, common.cuh)
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == kProducerWarp) {
        // ============================================================ TMA producer (whole warp walks, one elected lane issues)
        {
            const uint32_t elected = elect_one_pred();
            const CUtensorMap* my = src ? &map_y1 : &map_y0;
            if (lane == 0) {
                tma_prefetch_desc(my);
                tma_prefetch_desc(&map_x);
            }
            __syncwarp();
            uint32_t s = 0, ph = 0;
            for (int it = 0; it < nkb; ++it) {
                mbar_wait(bar_empty + 8 * s, ph ^ 1);
                XB_TS(0, it, 0);
                const uint32_t st = ring + s * kStage;
                mbar_arrive_expect_tx_if(elected, bar_full + 8 * s, kStage);
                const int row = (int)((blk0 + it) * 32);
#pragma unroll
                for (int g = 0; g < 4; ++g) tma_load_2d_if(elected, st + g * kBox, my, m0 + g * 32, row, bar_full + 8 * s);
#pragma unroll
                for (int g = 0; g < NBX; ++g) tma_load_2d_if(elected, st + (4 + g) * kBox, &map_x, g * 32, row, bar_full + 8 * s);
                if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp == kMmaWarp) {
        // ============================================================ MMA issuer: the whole warp walks the loop, one elected lane
        // issues (warp-uniform descriptors go through the uniform datapath — see the K-major TS kernel)
        {
            const uint32_t elected = elect_one_pred();
            const uint32_t tmem_base_u = __reduce_max_sync(0xffffffffu, tmem_base);
            uint32_t s = 0, ph = 0, j = 0, ready = 0;
            for (int it = 0; it < nkb; ++it) {
                XB_TS(1, it, 0);
                if (!ready) mbar_wait(bar_conv + 8 * s, ph);   // operand warps arrive after they saw the TMA bytes land
                XB_TS(1, it, 1);
                tc_fence_after();
                const uint32_t a_hi = ring + s * kStage, b_hi = a_hi + 4 * kBox;
                const uint32_t a_lo = lo_ring + j * kStage, b_lo = a_lo + 4 * kBox;
                const uint32_t ns = s + 1 == (uint32_t)S ? 0 : s + 1, nph = s + 1 == (uint32_t)S ? ph ^ 1 : ph;
                ready = ss_kblock_mn(tmem_base_u, umma_desc_sw128_base32(a_hi, kBox, 512), umma_desc_sw128_base32(a_lo, kBox, 512),
                                     umma_desc_sw128_base32(b_hi, kBox, 512), umma_desc_sw128_base32(b_lo, kBox, 512),
                                     kIdescMain, it != 0, bar_conv + 8 * ns, nph, bar_empty + 8 * s, bar_loempty + 8 * j,
                                     it == nkb - 1 ? bar_tfull : 0u, elected);
                XB_TS(1, it, 3);
                s = ns;
                ph = nph;
                if (++j == (uint32_t)L) j = 0;
            }
        }
    } else if (warp >= 4) {
        // ============================================================ operand warps
        // The 8 operand warps work as two groups of 4 that take alternate k-blocks, so that one group's barrier latency
        // (~450 cycles per k-block) overlaps the other's work.  (Three groups with the idle epilogue warps measured no
        // better: at ~1.7 k cycles per k-block the kernel sits at its shared-memory bandwidth floor — 224 KB of TMA
        // writes, operand-warp reads/writes and MMA operand reads per k-block at 128 B/clk.)
        const int t = threadIdx.x - 128;
        const int w = t >> 5;                       // 0..7: slot of this warp's partial sums in the final reduction
        const int grp = w >> 2, wr = w & 3;         // group (k-block parity), row group: rows 8 wr .. 8 wr + 7
        const int g = (t & 31) >> 3, c = t & 7;     // feature box, 16-byte chunk: features m0 + 32g + 4c .. +3
        const int nh = src ? p.nh[1] : p.nh[0];
        const float* dout = src ? p.dout[1] : p.dout[0];
        const float* w2p = src ? p.w2[1] : p.w2[0];
        float w2a[4], w2b[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int m = m0 + 32 * g + 4 * c + e;
            w2a[e] = w2p[m];
            w2b[e] = nh > 1 ? w2p[p.H_out + m] : 0.f;
        }
        float ga[4] = {0, 0, 0, 0}, gb[4] = {0, 0, 0, 0}, sa = 0.f, sb = 0.f;   // head-gradient accumulators
        float gz[4] = {0, 0, 0, 0};                                             // bias gradient: column sums of dz
        float d0[8], d1[8];
        auto load_dout = [&](int it) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int64_t b = (blk0 + it) * 32 + 8 * wr + i;
                const bool ok = it < nkb && b < p.B;
                d0[i] = ok ? __ldg(dout + b * nh) : 0.f;
                d1[i] = (ok && nh > 1) ? __ldg(dout + b * nh + 1) : 0.f;
            }
        };
        load_dout(grp);
        for (int it = grp; it < nkb; it += 2) {
            const uint32_t s = it % S, ph = (it / S) & 1, j = it % L;
            float c0[8], c1[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { c0[i] = d0[i]; c1[i] = d1[i]; }
            load_dout(it + 2);                       // prefetch this group's next k-block's head gradients
            mbar_wait(bar_full + 8 * s, ph);
            if ((t & 127) == 0) XB_TS(2, it, 0);
            mbar_wait(bar_loempty + 8 * j, ((it / L) & 1) ^ 1);
            if ((t & 127) == 0) XB_TS(2, it, 1);
            const uint32_t raw = ring + s * kStage, lo_b = lo_ring + j * kStage;
            float4 ys[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) ys[i] = lds128(raw + g * kBox + sw32_off(8 * wr + i, c));
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int r = 8 * wr + i;
                const uint32_t off = g * kBox + sw32_off(r, c);
                const float4 y = ys[i];
                const float e0 = c0[i], e1 = c1[i];
                ga[0] += e0 * y.x; ga[1] += e0 * y.y; ga[2] += e0 * y.z; ga[3] += e0 * y.w;
                gb[0] += e1 * y.x; gb[1] += e1 * y.y; gb[2] += e1 * y.z; gb[3] += e1 * y.w;
                sa += e0; sb += e1;
                float4 dz;
                dz.x = (e0 * w2a[0] + e1 * w2b[0]) * (y.x > 0.f ? 1.f : p.slope);
                dz.y = (e0 * w2a[1] + e1 * w2b[1]) * (y.y > 0.f ? 1.f : p.slope);
                dz.z = (e0 * w2a[2] + e1 * w2b[2]) * (y.z > 0.f ? 1.f : p.slope);
                dz.w = (e0 * w2a[3] + e1 * w2b[3]) * (y.w > 0.f ? 1.f : p.slope);
                gz[0] += dz.x; gz[1] += dz.y; gz[2] += dz.z; gz[3] += dz.w;
                float4 hi, lo;
                split_tf32(dz.x, hi.x, lo.x);
                split_tf32(dz.y, hi.y, lo.y);
                split_tf32(dz.z, hi.z, lo.z);
                split_tf32(dz.w, hi.w, lo.w);
                sts128(raw + off, hi);
                sts128(lo_b + off, lo);
            }
#pragma unroll
            for (int gg = 0; gg < NBX / 4; ++gg) {   // x operand: plain split, same thread mapping per group of 4 boxes
                float4 xs[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) xs[i] = lds128(raw + (4 + 4 * gg + g) * kBox + sw32_off(8 * wr + i, c));
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t off = (4 + 4 * gg + g) * kBox + sw32_off(8 * wr + i, c);
                    const float4 x = xs[i];
                    float4 hi, lo;
                    split_tf32(x.x, hi.x, lo.x);
                    split_tf32(x.y, hi.y, lo.y);
                    split_tf32(x.z, hi.z, lo.z);
                    split_tf32(x.w, hi.w, lo.w);
                    sts128(raw + off, hi);
                    sts128(lo_b + off, lo);
                }
            }
            if ((t & 127) == 0) XB_TS(2, it, 2);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_conv + 8 * s);
            if ((t & 127) == 0) XB_TS(2, it, 3);
        }
        if (t == 0) XB_TS(2, 63, 0);
        // head and bias gradients: sum the 8 warps' partial sums in a fixed order
        float* hs = sf + w * 384;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            hs[32 * g + 4 * c + e] = ga[e];
            hs[128 + 32 * g + 4 * c + e] = gb[e];
            hs[256 + 32 * g + 4 * c + e] = gz[e];
        }
        if ((t & 31) == 0) { sf[3072 + 2 * w] = sa; sf[3072 + 2 * w + 1] = sb; }
        bar_sync_named(1, kOperandWarps * 32);
        for (int i = t; i < 384; i += kOperandWarps * 32) {
            const float v = ((sf[i] + sf[384 + i]) + (sf[768 + i] + sf[1152 + i])) +
                            ((sf[1536 + i] + sf[1920 + i]) + (sf[2304 + i] + sf[2688 + i]));
            if (i < 256) p.head_part[(int64_t)blockIdx.x * 256 + i] = v;
            else p.part[((int64_t)blockIdx.x * 128 + (i - 256)) * (HIN + 4) + HIN] = v;      // bias column of the partial
        }
        if (t < 2)
            p.db2_part[(int64_t)blockIdx.x * 2 + t] = ((sf[3072 + t] + sf[3074 + t]) + (sf[3076 + t] + sf[3078 + t])) +
                                                      ((sf[3080 + t] + sf[3082 + t]) + (sf[3084 + t] + sf[3086 + t]));
    } else {
        // ============================================================ epilogue: partial [128][HIN + 4]
        float* out = p.part + ((int64_t)blockIdx.x * 128 + warp * 32 + lane) * (HIN + 4);
        if (nkb > 0) {
            mbar_wait(bar_tfull, 0);
            tc_fence_after();
        }
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
        for (int cc = 0; cc < HIN / 32; ++cc) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + cc * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 8; ++e)
                reinterpret_cast<float4*>(out + cc * 32)[e] =
                    nkb > 0 ? make_float4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]),
                                          __uint_as_float(v[4 * e + 2]), __uint_as_float(v[4 * e + 3]))
                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }

    if (threadIdx.x == 0) XB_TS(0, 63, 0);
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) XB_TS(0, 63, 1);
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc<kTmemCols>(tmem_base);
    }
}


// ================================================================================================ weight gradients, BINARY form
// Rank-1 head gradients (one head per source, or the two opposite logit gradients of a softmax pair):
//     dz_s[b][m] = e_s[b] * w2'_s[m] * leaky'(y_s[b][m]),   leaky' = slope + (1 - slope) * bin,   bin = (y > 0) in {0, 1}
// so with   A[m][n] = sum_b bin[b][m] * (e[b] x[b][n]),   G[n] = sum_b e[b] x[b][n],   S[m] = sum_b e[b] bin[b][m],   E = sum_b e[b]:
//     Gm[m][n] = (1 - slope) A[m][n] + slope G[n]         gm[m] = (1 - slope) S[m] + slope E
//     dW[m][n] = w2'[m] Gm[m][n]      db[m] = w2'[m] gm[m]      dw2[m] = sum_n W[m][n] Gm[m][n] + b[m] gm[m]  (= sum_b e y)      db2 = E
// The MMA's A operand is the 0/1 matrix `bin`, which TF32 holds EXACTLY: only the B operand (e x) needs the hi/lo split, i.e.
// 2 MMAs per k-step instead of 3, no lo copy of A, and — with the forward's activation sign words — no load of the activations
// at all (the head-weight gradient comes out of Gm in the reduce kernel).  Shared-memory traffic per 32-row k-block drops from
// 224 KB to 144 KB and the operand warps' work from ~1 k to ~0.4 k instructions.  Partials: part[cta][m][0..HIN) = A, [HIN] = S;
// head_part[cta][0..HIN) = G; db2_part[cta][0] = E.  The scaling above happens in wgrad_reduce_kernel (BinArgs).
__device__ __forceinline__ uint32_t ss_kblock_mn_bin(uint32_t d_tmem, uint64_t da, uint64_t db_hi, uint64_t db_lo, uint32_t idesc,
                                                     uint32_t accumulate_first, uint32_t next_bar, uint32_t next_par,
                                                     uint32_t commit0, uint32_t commit1, uint32_t commit2, uint32_t elected) {
    uint32_t ready;
    asm volatile(
        "{\n"
        ".reg .pred pn, p0, p1, c2, pe;\n"
        ".reg .b64 a, bh, bl;\n"
        "setp.ne.b32 pe, %12, 0;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 pn, [%7], %8;\n"
        "setp.ne.b32 p0, %6, 0;\n"
        "setp.ne.b32 p1, 1, 0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], %2, %3, %5, p0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], %2, %4, %5, p1;\n"
        "add.u64 a, %2, 64;  add.u64 bh, %3, 64;  add.u64 bl, %4, 64;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], a, bh, %5, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], a, bl, %5, p1;\n"
        "add.u64 a, %2, 128; add.u64 bh, %3, 128; add.u64 bl, %4, 128;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], a, bh, %5, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], a, bl, %5, p1;\n"
        "add.u64 a, %2, 192; add.u64 bh, %3, 192; add.u64 bl, %4, 192;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], a, bh, %5, p1;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%1], a, bl, %5, p1;\n"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%9];\n"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%10];\n"
        "setp.ne.b32 c2, %11, 0;\n"
        "and.pred c2, c2, pe;\n"
        "@c2 tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%11];\n"
        "selp.u32 %0, 1, 0, pn;\n"
        "}\n"
        : "=r"(ready)
        : "r"(d_tmem), "l"(da), "l"(db_hi), "l"(db_lo), "r"(idesc), "r"(accumulate_first), "r"(next_bar), "r"(next_par),
          "r"(commit0), "r"(commit1), "r"(commit2), "r"(elected)
        : "memory");
    return ready;
}

struct WBinParams {
    int64_t B;
    int n_jobs, halves, H_out;
    int stages, lo_bufs;
    const float* dout[2];      // e_s[b] = dout_s[b * nh_s]  (nh = 2: softmax pair, the second gradient is -e and is not read)
    int nh[2];
    const uint32_t* signs;     // [B][sign_ld] activation sign words: source s, features 32 c .. 32 c + 31 -> word s * (H_out / 32) + c
    int sign_ld;
    float* part;
    float* head_part;
    float* db2_part;
};

template <int HIN>
__global__ void __launch_bounds__(kThreads, 1)
    dense_wgrad_bin_kernel(const __grid_constant__ CUtensorMap map_x, const WBinParams p) {
    constexpr int NBX = HIN / 32;                  // 32-feature boxes of x
    constexpr int kBox = 32 * 128;                 // one box: 32 batch rows x 128 B
    constexpr int kStage = 4 * kBox + NBX * kBox;  // bin operand (128 features, written by the operand warps) | x operand -> hi
    constexpr int kLo = NBX * kBox;                // lo half of the x operand
    constexpr int kTmemCols = HIN;
    constexpr int kGroups = HIN == 128 ? 3 : 2;   // operand-warp groups (HIN = 256: the reduction scratch of 12 warps would not fit)
    constexpr int kOw = 4 * kGroups;               // operand warps
    constexpr uint32_t kIdescMain = umma_idesc_tf32(128, HIN, 1, 1);
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int S = p.stages, L = p.lo_bufs;
    const uint32_t ring = base, lo_ring = ring + (uint32_t)S * kStage, misc = lo_ring + (uint32_t)L * kLo;
    const uint32_t bar_full = misc, bar_conv = misc + 64, bar_empty = misc + 128, bar_loempty = misc + 192;
    const uint32_t bar_tfull = misc + 256, tmem_slot = misc + 264;
    unsigned char* misc_ptr = smem_raw + (misc - smem_u32(smem_raw));
    float* sf = reinterpret_cast<float*>(misc_ptr + 2048);   // reduction scratch: [8 warps][128 S | HIN G] + [8] E

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int job = blockIdx.x % p.n_jobs, q = blockIdx.x / p.n_jobs;
    const int cj = (gridDim.x - job + p.n_jobs - 1) / p.n_jobs;          // CTAs working on this job
    const int src = job / p.halves, m0 = (job % p.halves) * 128;
    const int64_t nblk = (p.B + 31) / 32;
    const int64_t blk0 = nblk * q / cj, blk1 = nblk * (q + 1) / cj;
    const int nkb = (int)(blk1 - blk0);

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_conv + 8 * s, kOperandWarps / 2);   // one group of 4 operand warps per k-block
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int j = 0; j < L; ++j) mbar_init(bar_loempty + 8 * j, 1);
        mbar_init(bar_tfull, 1);
        mbar_fence_init();
    }
    if (warp == kMmaWarp) tmem_alloc<kTmemCols>(tmem_slot);
    pdl_wait();
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == kProducerWarp) {
        // ============================================================ TMA producer: x boxes only (whole warp, one elected lane)
        const uint32_t elected = elect_one_pred();
        if (lane == 0) tma_prefetch_desc(&map_x);
        __syncwarp();
        uint32_t s = 0, ph = 0;
        for (int it = 0; it < nkb; ++it) {
            mbar_wait(bar_empty + 8 * s, ph ^ 1);
            const uint32_t st = ring + s * kStage;
            mbar_arrive_expect_tx_if(elected, bar_full + 8 * s, NBX * kBox);
            const int row = (int)((blk0 + it) * 32);
#pragma unroll
            for (int g = 0; g < NBX; ++g) tma_load_2d_if(elected, st + (4 + g) * kBox, &map_x, g * 32, row, bar_full + 8 * s);
            if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
        }
    } else if (warp == kMmaWarp) {
        // ============================================================ MMA issuer (whole warp, one elected lane): 8 MMAs per k-block
        const uint32_t elected = elect_one_pred();
        const uint32_t tmem_base_u = __reduce_max_sync(0xffffffffu, tmem_base);
        uint32_t s = 0, ph = 0, j = 0, ready = 0;
        for (int it = 0; it < nkb; ++it) {
            if (!ready) mbar_wait(bar_conv + 8 * s, ph);
            tc_fence_after();
            const uint32_t a = ring + s * kStage, b_hi = a + 4 * kBox, b_lo = lo_ring + j * kLo;
            const uint32_t ns = s + 1 == (uint32_t)S ? 0 : s + 1, nph = s + 1 == (uint32_t)S ? ph ^ 1 : ph;
            ready = ss_kblock_mn_bin(tmem_base_u, umma_desc_sw128_base32(a, kBox, 512), umma_desc_sw128_base32(b_hi, kBox, 512),
                                     umma_desc_sw128_base32(b_lo, kBox, 512), kIdescMain, it != 0, bar_conv + 8 * ns, nph,
                                     bar_empty + 8 * s, bar_loempty + 8 * j, it == nkb - 1 ? bar_tfull : 0u, elected);
            s = ns;
            ph = nph;
            if (++j == (uint32_t)L) j = 0;
        }
    } else {
      // ============================================================ operand warps: groups of 4 on k-blocks it = grp (mod kGroups).
      // HIN = 128: THREE groups — the epilogue warps 0-3 are idle until the accumulator is complete and the loop is bound by the
      // operand warps' latency chains (measured 1 550 cycles per k-block with two groups against a 1 125-cycle shared-memory floor)
      if (warp >= 4 || kGroups == 3) {
        const int w = warp >= 4 ? warp - 4 : warp + 8;   // 0..11: slot of this warp's partial sums in the final reduction
        const int t = w * 32 + lane;
        const int grp = w >> 2, wr = w & 3;         // group, row group: rows 8 wr .. 8 wr + 7
        const int g = (t & 31) >> 3, c = t & 7;     // feature box, 16-byte chunk: features m0 + 32 g + 4 c .. + 3
        const int nh = p.nh[src];
        const float* dout = p.dout[src];
        const int word = src * (p.H_out >> 5) + (m0 >> 5) + g;      // this thread's sign word of a row
        float sacc[4] = {0, 0, 0, 0};               // S[m]: sum_b e[b] bin[b][m] for this thread's 4 features
        float gacc[NBX / 4][4];                     // G[n]: sum_b e[b] x[b][n] for this thread's x columns
#pragma unroll
        for (int gg = 0; gg < NBX / 4; ++gg)
#pragma unroll
            for (int e = 0; e < 4; ++e) gacc[gg][e] = 0.f;
        float esum = 0.f;
        float d0[8];
        uint32_t sw[8];
        auto prefetch = [&](int it) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int64_t b = (blk0 + it) * 32 + 8 * wr + i;
                const bool ok = it < nkb && b < p.B;
                d0[i] = ok ? __ldg(dout + b * nh) : 0.f;
                sw[i] = ok ? __ldg(p.signs + b * p.sign_ld + word) : 0u;
            }
        };
        prefetch(grp);
        for (int it = grp; it < nkb; it += kGroups) {
            const uint32_t s = it % S, ph = (it / S) & 1, j = it % L;
            float ev[8];
            uint32_t bits[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { ev[i] = d0[i]; bits[i] = sw[i] >> (4 * c); }
            prefetch(it + kGroups);                  // this group's next k-block
            mbar_wait(bar_full + 8 * s, ph);         // (x landed; the stage was released by the MMAs of its previous use)
            mbar_wait(bar_loempty + 8 * j, ((it / L) & 1) ^ 1);
            const uint32_t raw = ring + s * kStage, lo_b = lo_ring + j * kLo;
#pragma unroll
            for (int i = 0; i < 8; ++i) {            // A operand: the 0/1 matrix itself
                const uint32_t off = g * kBox + sw32_off(8 * wr + i, c);
                const float e = ev[i];
                float4 a;
                a.x = (bits[i] & 1u) ? 1.f : 0.f;
                a.y = (bits[i] & 2u) ? 1.f : 0.f;
                a.z = (bits[i] & 4u) ? 1.f : 0.f;
                a.w = (bits[i] & 8u) ? 1.f : 0.f;
                sacc[0] += e * a.x; sacc[1] += e * a.y; sacc[2] += e * a.z; sacc[3] += e * a.w;
                esum += e;
                sts128(raw + off, a);
            }
#pragma unroll
            for (int gg = 0; gg < NBX / 4; ++gg) {   // B operand: e[b] x[b][n], split hi (in place) / lo
                float4 xs[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) xs[i] = lds128(raw + (4 + 4 * gg + g) * kBox + sw32_off(8 * wr + i, c));
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t off = (4 * gg + g) * kBox + sw32_off(8 * wr + i, c);
                    const float e = ev[i];
                    float4 v = make_float4(e * xs[i].x, e * xs[i].y, e * xs[i].z, e * xs[i].w);
                    gacc[gg][0] += v.x; gacc[gg][1] += v.y; gacc[gg][2] += v.z; gacc[gg][3] += v.w;
                    float4 hi, lo;
                    split_tf32(v.x, hi.x, lo.x);
                    split_tf32(v.y, hi.y, lo.y);
                    split_tf32(v.z, hi.z, lo.z);
                    split_tf32(v.w, hi.w, lo.w);
                    sts128(raw + 4 * kBox + off, hi);
                    sts128(lo_b + off, lo);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_conv + 8 * s);
        }
        // column sums: the operand warps' partials in a fixed order
        constexpr int kCols = 128 + HIN;
        float* hs = sf + w * kCols;
#pragma unroll
        for (int e = 0; e < 4; ++e) hs[32 * g + 4 * c + e] = sacc[e];
#pragma unroll
        for (int gg = 0; gg < NBX / 4; ++gg)
#pragma unroll
            for (int e = 0; e < 4; ++e) hs[128 + 32 * (4 * gg + g) + 4 * c + e] = gacc[gg][e];
        // (esum: every thread of a warp saw the same 8 rows per k-block; one lane per warp reports it)
        if ((t & 31) == 0) sf[kOw * kCols + w] = esum;
        bar_sync_named(1, kOw * 32);
        for (int i = t; i < kCols; i += kOw * 32) {
            float v = ((sf[i] + sf[kCols + i]) + (sf[2 * kCols + i] + sf[3 * kCols + i])) +
                      ((sf[4 * kCols + i] + sf[5 * kCols + i]) + (sf[6 * kCols + i] + sf[7 * kCols + i]));
            if (kGroups == 3) v += (sf[8 * kCols + i] + sf[9 * kCols + i]) + (sf[10 * kCols + i] + sf[11 * kCols + i]);
            if (i < 128) p.part[((int64_t)blockIdx.x * 128 + i) * (HIN + 4) + HIN] = v;       // S[m]: the bias column
            else p.head_part[(int64_t)blockIdx.x * 256 + (i - 128)] = v;                     // G[n]
        }
        if (t == 0) {
            const float* es = sf + kOw * kCols;
            float e = ((es[0] + es[1]) + (es[2] + es[3])) + ((es[4] + es[5]) + (es[6] + es[7]));
            if (kGroups == 3) e += (es[8] + es[9]) + (es[10] + es[11]);
            p.db2_part[(int64_t)blockIdx.x * 2] = e;
            p.db2_part[(int64_t)blockIdx.x * 2 + 1] = 0.f;
        }
      }
      if (warp < 4) {
        // ============================================================ epilogue: partial [128][HIN + 4]
        float* out = p.part + ((int64_t)blockIdx.x * 128 + warp * 32 + lane) * (HIN + 4);
        if (nkb > 0) {
            mbar_wait(bar_tfull, 0);
            tc_fence_after();
        }
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
        for (int cc = 0; cc < HIN / 32; ++cc) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + cc * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 8; ++e)
                reinterpret_cast<float4*>(out + cc * 32)[e] =
                    nkb > 0 ? make_float4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]),
                                          __uint_as_float(v[4 * e + 2]), __uint_as_float(v[4 * e + 3]))
                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc<kTmemCols>(tmem_base);
    }
}

// Finishing the BINARY-form partials in wgrad_reduce_kernel (see dense_wgrad_bin_kernel): per source the master weights
// W [H_out][HIN] and bias [H_out] of the hidden layer, the head weights w2 [nh][H_out] (nh = 2: softmax pair, w2' = w2[0] - w2[1]).
struct BinArgs {
    int on;
    float slope;
    const float* W[2];
    const float* b[2];
    const float* w2[2];
};

// Sums the per-CTA partials of the wgrad kernel in a fixed order (deterministic) and scatters them to the parameter
// gradients.  One block per (job, output row m): 4 thread groups each add a quarter of the CTAs' partials for their
// column (loads unrolled so many are in flight), then the groups are combined through shared memory.
// Optional tail work of the same launch (blocks beyond the n_jobs * 128 reduce blocks): the trunk layer's partial sums
// (mlp_trunk.cu: [n_part][H][OBS + 1]) -> dW0, db0, one warp per output; and the fp64 log-std gradient of the loss kernel
// -> the fp32 parameter gradient.  Saves two launches per update.
struct TailArgs {
    const float* trunk_part;
    int n_part, H, OBS;
    float* dW0t;
    float* db0t;
    const double* dls64;
    float* dls32;
    int A;
    // optional: this launch finishes EVERY gradient of the policy, so it can also take their global norm and derive the
    // clipped-Adam step scalars (what grad_norm_kernel does in a launch of its own); norm_ws = optim workspace or NULL
    double* norm_ws;
    int64_t* step_dev;
    xb::AdamHyper hyper;
    float* lr_out;
    float* gnorm_out;
};

__global__ void __launch_bounds__(512, 2) wgrad_reduce_kernel(const float* __restrict__ part, const float* __restrict__ head_part,
                                    const float* __restrict__ db2_part, int grid, int n_jobs, int halves, int HIN,
                                    int H_out, float* dW0, float* db0, float* dw2_0, float* db2_0, int nh0, float* dW1,
                                    float* db1, float* dw2_1, float* db2_1, int nh1, TailArgs tail, BinArgs bin) {
    __shared__ float red[4][260];
    __shared__ float bin_g[256], bin_g4[4][256], bin_red[4], bin_e;
    __shared__ double norm_smem[32];
    __shared__ bool norm_last;
    pdl_wait();
    pdl_trigger();
    const float gs = tail.hyper.grad_scale;
    double sq = 0.0;                                   // this thread's share of sum((grad * grad_scale)^2)
#define XB_SQ(x) do { const double g__ = (double)((x) * gs); sq += g__ * g__; } while (0)
    if ((int)blockIdx.x >= n_jobs * 128) {
        const int tb = blockIdx.x - n_jobs * 128, lane = threadIdx.x & 31;
        const int n_out = tail.H * (tail.OBS + 1);
        const int k = tb * 16 + (threadIdx.x >> 5);
        if (tail.trunk_part && k < n_out) {
            float sum = 0.f;
            for (int q = lane; q < tail.n_part; q += 32) sum += tail.trunk_part[(int64_t)q * n_out + k];
            sum = warp_sum(sum);
            if (lane == 0) {
                const int n = k / (tail.OBS + 1), i = k % (tail.OBS + 1);
                if (i < tail.OBS) tail.dW0t[n * tail.OBS + i] = sum;
                else tail.db0t[n] = sum;
                XB_SQ(sum);
            }
        }
        if (tb == 0 && tail.dls64 && (int)threadIdx.x < tail.A) {
            const float g = (float)tail.dls64[threadIdx.x];
            tail.dls32[threadIdx.x] = g;
            XB_SQ(g);
        }
    } else {
        const int job = blockIdx.x / 128, r = blockIdx.x % 128;
        const int src = job / halves, m = (job % halves) * 128 + r;
        float* dW = src ? dW1 : dW0;
        float* db = src ? db1 : db0;
        float* dw2 = src ? dw2_1 : dw2_0;
        float* db2 = src ? db2_1 : db2_0;
        const int nh = src ? nh1 : nh0;
        const int grp = threadIdx.x >> 7, t = threadIdx.x & 127;
        const int n_cta = (grid - job + n_jobs - 1) / n_jobs;          // CTAs that worked on this job: job, job + n_jobs, ...
        const int ncol = bin.on ? HIN + 1 : HIN + 3;                    // HIN weights | bias | head 0 | head 1
        // BINARY form: the scaling operands, loaded up front so that they travel with the partials' round trip
        float bw[2] = {0.f, 0.f}, w2m = 0.f, bias_m = 0.f;
        if (bin.on) {
            const float* w2p = bin.w2[src];
            w2m = nh > 1 ? w2p[m] - w2p[H_out + m] : w2p[m];
            bias_m = bin.b[src][m];
            if (grp == 0) {
                bw[0] = bin.W[src][(int64_t)m * HIN + t];
                if (HIN > 128) bw[1] = bin.W[src][(int64_t)m * HIN + 128 + t];
            }
        }
        for (int n = t; n < ncol; n += 128) {
            float acc = 0.f;
            const float* src_ptr;
            int64_t stride;
            if (n <= HIN) {
                src_ptr = part + ((int64_t)job * 128 + r) * (HIN + 4) + n;
                stride = (int64_t)n_jobs * 128 * (HIN + 4);
            } else {
                src_ptr = head_part + (int64_t)job * 256 + (n - HIN - 1) * 128 + r;
                stride = (int64_t)n_jobs * 256;
            }
            float v[20];                                                // all of this group's partials in flight (<= 148/4/... )
#pragma unroll
            for (int u = 0; u < 20; ++u) {
                const int c = grp + 4 * u;
                v[u] = c < n_cta ? src_ptr[c * stride] : 0.f;
            }
            // BINARY form: the column sums G[n] (head_part rows of this job's CTAs) ride in the same round trip
            const bool with_g = bin.on && n < HIN;
            const float* g_ptr = head_part + (int64_t)job * 256 + n;
            const int64_t g_stride = (int64_t)n_jobs * 256;
            float v2[20], acc2 = 0.f;
#pragma unroll
            for (int u = 0; u < 20; ++u) {
                const int c = grp + 4 * u;
                v2[u] = (with_g && c < n_cta) ? g_ptr[c * g_stride] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 20; ++u) acc += v[u];
            for (int c = grp + 80; c < n_cta; c += 4) acc += src_ptr[c * stride];
            red[grp][n] = acc;
            if (with_g) {
#pragma unroll
                for (int u = 0; u < 20; ++u) acc2 += v2[u];
                for (int c = grp + 80; c < n_cta; c += 4) acc2 += g_ptr[c * g_stride];
                bin_g4[grp][n] = acc2;
            }
        }
        if (bin.on) {
            // BINARY form (dense_wgrad_bin_kernel): column sums G[n] (head_part rows of this job's CTAs) and E (db2_part), every
            // block for itself; then Gm = (1 - slope) A + slope G, gm = (1 - slope) S + slope E and the scalings by w2' / W / b
            if (threadIdx.x >= 480) {                                   // last warp: E
                float e = 0.f;
                for (int c = t - 96; c < n_cta; c += 32) e += db2_part[(int64_t)(job + c * n_jobs) * 2];
                e = warp_sum(e);
                if (t == 96) bin_e = e;
            }
        }
        __syncthreads();
        if (bin.on) {
            for (int n = threadIdx.x; n < HIN; n += 512) bin_g[n] = (bin_g4[0][n] + bin_g4[1][n]) + (bin_g4[2][n] + bin_g4[3][n]);
            __syncthreads();
            const float sl = bin.slope, om = 1.0f - bin.slope;
            float dot = 0.f;                                            // this thread's share of sum_n W[m][n] Gm[n]
            if (grp == 0) {
                for (int n = t; n < HIN; n += 128) {
                    const float A = (red[0][n] + red[1][n]) + (red[2][n] + red[3][n]);
                    const float gm_n = om * A + sl * bin_g[n];
                    const float gw = w2m * gm_n;
                    dW[(int64_t)m * HIN + n] = gw;
                    XB_SQ(gw);
                    dot += bw[n >> 7] * gm_n;
                }
                dot = warp_sum(dot);
                if ((t & 31) == 0) bin_red[t >> 5] = dot;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                const float S = (red[0][HIN] + red[1][HIN]) + (red[2][HIN] + red[3][HIN]);
                const float gm = om * S + sl * bin_e;
                const float gb = w2m * gm;
                db[m] = gb;
                XB_SQ(gb);
                const float g2 = ((bin_red[0] + bin_red[1]) + (bin_red[2] + bin_red[3])) + bias_m * gm;
                dw2[m] = g2;
                XB_SQ(g2);
                if (nh > 1) { dw2[H_out + m] = -g2; XB_SQ(g2); }
                if (m == 0) {
                    db2[0] = bin_e;
                    XB_SQ(bin_e);
                    if (nh > 1) { db2[1] = -bin_e; XB_SQ(bin_e); }
                }
            }
        } else if (grp == 0) {
            for (int n = t; n < ncol; n += 128) {
                const float acc = (red[0][n] + red[1][n]) + (red[2][n] + red[3][n]);
                if (n < HIN) { dW[(int64_t)m * HIN + n] = acc; XB_SQ(acc); }
                else if (n == HIN) { db[m] = acc; XB_SQ(acc); }
                else if (n - HIN - 1 < nh) { dw2[(int64_t)(n - HIN - 1) * H_out + m] = acc; XB_SQ(acc); }
            }
        }
        if (!bin.on && m == 0 && grp >= 1 && grp - 1 < nh && t < 32) {  // db2: this job's CTAs cover the whole batch; one warp per head
            const int h = grp - 1;
            float s = 0.f;
            for (int c = t; c < n_cta; c += 32) s += db2_part[(int64_t)(job + c * n_jobs) * 2 + h];
            s = warp_sum(s);
            if (t == 0) { db2[h] = s; XB_SQ(s); }
        }
    }
#undef XB_SQ
    if (tail.norm_ws)   // uniform across the grid
        grad_norm_finish(sq, tail.step_dev, tail.hyper, tail.norm_ws, tail.lr_out, tail.gnorm_out, norm_smem, &norm_last);
}

template <int HIN>
static int launch_wgrad(const CUtensorMap& my0, const CUtensorMap& my1, const CUtensorMap& mx, WParams p, int grid,
                        cudaStream_t s) {
    const int stage = (4 + HIN / 32) * 4096;
    const int avail = kMaxSmem - 1024 - kWMiscBytes;
    int L = 2, S = (avail - L * stage) / stage;
    if (S < 2) { L = 1; S = (avail - L * stage) / stage; }
    if (S < 2) return XB_E_UNSUPPORTED;
    if (S > 6) S = 6;
    p.stages = S;
    p.lo_bufs = L;
#ifdef XB_DENSE_TS
    p.ts = g_xb_ts_host;
#endif
    const int smem = 1024 + (S + L) * stage + kWMiscBytes;
    auto kern = dense_wgrad_kernel<HIN>;
    XB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));   // per device, cheap: set on every launch
    XB_CUDA(launch_pdl(kern, dim3(grid), dim3(kThreads), (size_t)smem, s, true, my0, my1, mx, p));
    XB_LAUNCH_CHECK();
    return 0;
}

}  // namespace dense
}  // namespace xb

using namespace xb;
using namespace xb::dense;

static inline bool al16(const void* q) { return ((uintptr_t)q & 15u) == 0; }

#ifdef XB_DENSE_TS
extern "C" int xb_dense_debug_set_ts(long long* buf) {
    xb::dense::g_xb_ts_host = buf;
    return 0;
}
#endif

extern "C" int xb_dense_split_weights(const float* W, int N, int K, float* hi, float* lo, float* thi, float* tlo,
                                      int ldt, int toff, xb_stream_t stream) {
    if (!W || !hi || !lo || N <= 0 || K <= 0 || (thi && !tlo)) return XB_E_BADARG;
    const int n = N * K;
    SplitJob j0{W, hi, lo, toff}, j1{nullptr, nullptr, nullptr, 0};
    split_weights_kernel<<<dim3((n + 255) / 256, 1), 256, 0, (cudaStream_t)stream>>>(j0, j1, N, K, thi, tlo, ldt);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_dense_split_weights2(const float* W0, float* hi0, float* lo0, const float* W1, float* hi1, float* lo1,
                                       int N, int K, float* thi, float* tlo, xb_stream_t stream) {
    if (!W0 || !hi0 || !lo0 || !W1 || !hi1 || !lo1 || N <= 0 || K <= 0 || (thi && !tlo)) return XB_E_BADARG;
    const int n = N * K;
    SplitJob j0{W0, hi0, lo0, 0}, j1{W1, hi1, lo1, N};
    split_weights_kernel<<<dim3((n + 255) / 256, 2), 256, 0, (cudaStream_t)stream>>>(j0, j1, N, K, thi, tlo, 2 * N);
    XB_LAUNCH_CHECK();
    return 0;
}

struct TrunkArgs {
    const float* obs;
    int ld, obs_dim;
    const float* W0;
    const float* b0;
    const double* norm_new;
    const double* norm_old;
    int64_t norm_rows;
    float norm_clip;
    int flags;
    float* h1_out;
};

static int dense_fwd_impl(const float* X, const TrunkArgs* trunk, int64_t M, int K, int N, float slope, int n_layers, const float* const* Whi,
                          const float* const* Wlo, const float* const* bias, float* const* Y, const float* const* head_w,
                          const float* const* head_b, const int* n_head, float* const* head_out, int b_resident,
                          xb_stream_t stream, const FusedLoss* loss = nullptr, const float* const* prep_W = nullptr,
                          float* prep_thi = nullptr, float* prep_tlo = nullptr, uint32_t* sign_out = nullptr) {
    if ((!X && !trunk) || M <= 0) return XB_E_BADARG;
    if (K % BK != 0 || K < BK || K > 256 || (X && !al16(X))) return XB_E_UNSUPPORTED;
    if (trunk && (!trunk->obs || !trunk->W0 || !trunk->b0 || trunk->obs_dim < 1 || trunk->obs_dim > 4 ||
                  trunk->ld < trunk->obs_dim || N > 128))
        return XB_E_UNSUPPORTED;
    TMaps maps;
    memset(&maps, 0, sizeof(maps));
    for (int l = 0; l < n_layers; ++l) {
        if (!Whi[l] || !Wlo[l] || (!Y[l] && !n_head[l]) || (!Y[0] != !Y[l])) return XB_E_BADARG;
        if (n_head[l] < 0 || n_head[l] > 2 || (n_head[l] && (!head_w[l] || !head_b[l] || !head_out[l]))) return XB_E_UNSUPPORTED;
        if (!al16(Whi[l]) || !al16(Wlo[l]) || (Y[l] && !al16(Y[l]))) return XB_E_UNSUPPORTED;
        CUtensorMap* mh = l ? &maps.bhi1 : &maps.bhi;
        CUtensorMap* ml = l ? &maps.blo1 : &maps.blo;
        CUtensorMap* mo = l ? &maps.out1 : &maps.out;
        if (!xb_make_map_f32_2d(mh, Whi[l], N, K, K, N, BK, 1) || !xb_make_map_f32_2d(ml, Wlo[l], N, K, K, N, BK, 1) ||
            !(Y[l] ? xb_make_map_f32_2d(mo, Y[l], M, N, N, 32, 32, 1)       // Y == NULL: heads only, map never used
                   : xb_make_map_f32_2d(mo, Whi[l], N, K, K, 32, 32, 1)))
            return XB_E_DRIVER;
    }
    if (n_layers == 1) { maps.bhi1 = maps.bhi; maps.blo1 = maps.blo; maps.out1 = maps.out; }
    maps.h1 = maps.out;
    if (X) {
        if (!xb_make_map_f32_2d(&maps.a0, X, M, K, K, BM, BK, 1)) return XB_E_DRIVER;
    } else {
        maps.a0 = maps.out;      // never dereferenced: the operand warps generate A from the observations
    }
    maps.a1 = maps.a0;
    KParams p{};
    if (!X) {
        p.obs = trunk->obs;
        p.obs_ld = trunk->ld;
        p.obs_dim = trunk->obs_dim;
        p.W0 = trunk->W0;
        p.b0 = trunk->b0;
        p.norm_new = trunk->norm_new;
        p.norm_old = trunk->norm_old;
        p.norm_rows = trunk->norm_rows;
        p.norm_clip = trunk->norm_clip;
        p.pdl_launch = 1;
        p.pdl_early = (trunk->flags & XB_FWD_WEIGHTS_STABLE) ? 1 : 0;
        if (trunk->h1_out && !al16(trunk->h1_out)) return XB_E_UNSUPPORTED;
        p.h1_out = trunk->h1_out;
    }
    p.M = M;
    p.KB = K / BK;
    p.kb_split = p.KB;
    p.slope = slope;
    p.bias = bias[0];
    p.Y = Y[0];
    p.head_w = head_w[0];
    p.head_b = head_b[0];
    p.n_head = n_head[0];
    p.head_out = head_out[0];
    p.dual = n_layers == 2;
    if (p.dual) {
        p.bias1 = bias[1];
        p.head_w1 = head_w[1];
        p.head_b1 = head_b[1];
        p.n_head1 = n_head[1];
        p.head_out1 = head_out[1];
    }
    if (loss) {
        if (n_layers != 2 || n_head[1] != 1 || n_head[0] != (loss->gaussian ? 1 : 2)) return XB_E_UNSUPPORTED;
        p.loss = *loss;
    }
    if (prep_thi) {     // weight operand of the mask-form dgrad launch that follows (see KParams::mask_form)
        if (n_layers != 2 || K != N || !prep_tlo || !prep_W || !prep_W[0] || !prep_W[1] || n_head[0] < 1 || n_head[1] < 1) return XB_E_BADARG;
        for (int l = 0; l < 2; ++l) {
            p.prep_W[l] = prep_W[l];
            p.prep_w2[l] = head_w[l];
            p.prep_nh[l] = n_head[l];
        }
        p.prep_thi = prep_thi;
        p.prep_tlo = prep_tlo;
        p.prep_H = N;
    }
    p.sign_out = sign_out;
    p.sign_ld = n_layers * (N / 32);
    return dispatch_kmajor<MODE_FWD>(N, b_resident != 0, maps, p, (cudaStream_t)stream);
}

extern "C" int xb_dense_fwd(const float* X, int64_t M, int K, const float* Whi, const float* Wlo, int N,
                            const float* bias, float slope, float* Y, const float* head_w, const float* head_b,
                            int n_head, float* head_out, int b_resident, xb_stream_t stream) {
    return dense_fwd_impl(X, nullptr, M, K, N, slope, 1, &Whi, &Wlo, &bias, &Y, &head_w, &head_b, &n_head, &head_out, b_resident,
                          stream);
}

extern "C" int xb_dense_fwd2(const float* X, int64_t M, int K, int N, float slope, const float* Whi0, const float* Wlo0,
                             const float* bias0, float* Y0, const float* head_w0, const float* head_b0, int n_head0,
                             float* head_out0, const float* Whi1, const float* Wlo1, const float* bias1, float* Y1,
                             const float* head_w1, const float* head_b1, int n_head1, float* head_out1, int b_resident,
                             const float* prep_W0, const float* prep_W1, float* prep_thi, float* prep_tlo, uint32_t* sign_out,
                             xb_stream_t stream) {
    const float* Whi[2] = {Whi0, Whi1};
    const float* Wlo[2] = {Wlo0, Wlo1};
    const float* bias[2] = {bias0, bias1};
    float* Y[2] = {Y0, Y1};
    const float* hw[2] = {head_w0, head_w1};
    const float* hb[2] = {head_b0, head_b1};
    const int nh[2] = {n_head0, n_head1};
    float* ho[2] = {head_out0, head_out1};
    const float* pw[2] = {prep_W0, prep_W1};
    return dense_fwd_impl(X, nullptr, M, K, N, slope, 2, Whi, Wlo, bias, Y, hw, hb, nh, ho, b_resident, stream, nullptr, pw,
                          prep_thi, prep_tlo, sign_out);
}

extern "C" int xb_dense_fwd2_loss(const float* X, int64_t M, int K, int N, float slope, const float* Whi0, const float* Wlo0,
                                  const float* bias0, float* Y0, const float* head_w0, const float* head_b0, int n_head0,
                                  float* head_out0, const float* Whi1, const float* Wlo1, const float* bias1, float* Y1,
                                  const float* head_w1, const float* head_b1, int n_head1, float* head_out1, int b_resident,
                                  const float* scal, const double* adv_stats, int64_t adv_count, float clip_range,
                                  float vf_coef, float ent_coef, float inv_batch, const float* logstd, float* dact, float* dv,
                                  double* loss_partials, uint32_t* loss_ticket, double* scalars, double* dlogstd,
                                  const float* prep_W0, const float* prep_W1, float* prep_thi, float* prep_tlo,
                                  uint32_t* sign_out, xb_stream_t stream) {
    if (!scal || !dact || !dv || !loss_partials || !loss_ticket || !scalars) return XB_E_BADARG;
    if (adv_stats && adv_count <= 0) return XB_E_BADARG;
    if (logstd && !dlogstd) return XB_E_BADARG;
    if (((uintptr_t)scal & 15u)) return XB_E_BADARG;
    const float* Whi[2] = {Whi0, Whi1};
    const float* Wlo[2] = {Wlo0, Wlo1};
    const float* bias[2] = {bias0, bias1};
    float* Y[2] = {Y0, Y1};
    const float* hw[2] = {head_w0, head_w1};
    const float* hb[2] = {head_b0, head_b1};
    const int nh[2] = {n_head0, n_head1};
    float* ho[2] = {head_out0, head_out1};
    FusedLoss L{(const float4*)scal, adv_stats, adv_stats ? 1.0 / (double)adv_count : 0.0, clip_range, vf_coef, ent_coef,
                inv_batch, logstd ? 1 : 0, logstd, dact, dv, loss_partials, loss_ticket, scalars, dlogstd};
    const float* pw[2] = {prep_W0, prep_W1};
    return dense_fwd_impl(X, nullptr, M, K, N, slope, 2, Whi, Wlo, bias, Y, hw, hb, nh, ho, b_resident, stream, &L, pw, prep_thi,
                          prep_tlo, sign_out);
}

extern "C" int xb_mlp_fwd_from_obs(const float* obs, int ld, int obs_dim, const float* W0, const float* b0, int64_t M, int H,
                                   float slope, const float* Whi0, const float* Wlo0, const float* bias0, float* Y0,
                                   const float* head_w0, const float* head_b0, int n_head0, float* head_out0,
                                   const float* Whi1, const float* Wlo1, const float* bias1, float* Y1,
                                   const float* head_w1, const float* head_b1, int n_head1, float* head_out1,
                                   const double* norm_new, const double* norm_old, int64_t norm_rows, float norm_clip,
                                   int flags, xb_stream_t stream) {
    if ((norm_new != nullptr) != (norm_old != nullptr)) return XB_E_BADARG;
    const float* Whi[2] = {Whi0, Whi1};
    const float* Wlo[2] = {Wlo0, Wlo1};
    const float* bias[2] = {bias0, bias1};
    float* Y[2] = {Y0, Y1};
    const float* hw[2] = {head_w0, head_w1};
    const float* hb[2] = {head_b0, head_b1};
    const int nh[2] = {n_head0, n_head1};
    float* ho[2] = {head_out0, head_out1};
    TrunkArgs t{obs, ld, obs_dim, W0, b0, norm_new, norm_old, norm_rows, norm_clip, flags, nullptr};
    return dense_fwd_impl(nullptr, &t, M, H, H, slope, 2, Whi, Wlo, bias, Y, hw, hb, nh, ho, 1, stream);
}

extern "C" int xb_dense_dgrad(const float* Y0, const float* dout0, const float* w2_0, int nh0, int K0, const float* Y1,
                              const float* dout1, const float* w2_1, int nh1, int K1, int64_t M, const float* Wthi,
                              const float* Wtlo, int N, const float* H1, float slope, float* dZ1, int wt_form,
                              const uint32_t* signs, const uint32_t* h1_signs, xb_stream_t stream) {
    if (wt_form != 0 && wt_form != 1) return XB_E_BADARG;
    if (h1_signs && ((uintptr_t)h1_signs & 15u)) return XB_E_BADARG;
    if (!Y0 || !dout0 || !w2_0 || !Wthi || !Wtlo || !H1 || !dZ1 || M <= 0) return XB_E_BADARG;
    if (K0 % BK != 0 || K0 < BK || K0 > 256 || nh0 < 1 || nh0 > 2) return XB_E_UNSUPPORTED;
    if (Y1 && (K1 % BK != 0 || K1 < BK || K1 > 256 || nh1 < 1 || nh1 > 2 || !dout1 || !w2_1)) return XB_E_UNSUPPORTED;
    if (!Y1) K1 = 0;
    if (!al16(Y0) || !al16(Wthi) || !al16(Wtlo) || !al16(H1) || !al16(dZ1) || (Y1 && !al16(Y1))) return XB_E_UNSUPPORTED;
    const int K = K0 + K1;
    // N = 128, K <= 256: split the output columns over two CTAs per tile so that each keeps its 64 weight rows (hi + lo,
    // <= 128 KB) resident in shared memory; otherwise every tile would re-stream all of W^T from L2 (134 MB per launch)
    // (opt-in: measured slower at 65 536 x 128 — the duplicated on-the-fly operand generation outweighs the L2 saving)
    static const bool want_split = []() { const char* e = getenv("XB_DGRAD_SPLIT"); return e && e[0] == '1'; }();
    const bool split = N == 128 && K <= 256 && want_split;
    const int brows = split ? 64 : N;
    TMaps maps;
    if (!xb_make_map_f32_2d(&maps.out, dZ1, M, N, N, 32, 32, 1) || !xb_make_map_f32_2d(&maps.h1, H1, M, N, N, 32, 32, 1) ||
        !xb_make_map_f32_2d(&maps.a0, Y0, M, K0, K0, BM, BK, 1) ||
        !xb_make_map_f32_2d(&maps.a1, Y1 ? Y1 : Y0, M, Y1 ? K1 : K0, Y1 ? K1 : K0, BM, BK, 1) ||
        !xb_make_map_f32_2d(&maps.bhi, Wthi, N, K, K, brows, BK, 1) || !xb_make_map_f32_2d(&maps.blo, Wtlo, N, K, K, brows, BK, 1))
        return XB_E_DRIVER;
    maps.bhi1 = maps.bhi; maps.blo1 = maps.blo; maps.out1 = maps.out;
    KParams p{};
    p.M = M;
    p.KB = K / BK;
    p.kb_split = K0 / BK;
    p.slope = slope;
    p.dout0 = dout0;
    p.w2_0 = w2_0;
    p.nh0 = nh0;
    p.dout1 = dout1;
    p.w2_1 = w2_1;
    p.nh1 = Y1 ? nh1 : 0;
    p.H1 = H1;
    p.dZ1 = dZ1;
    p.n_split = split ? 2 : 1;
    p.mask_form = wt_form;
    p.signs = (K / BK <= 8) ? signs : nullptr;       // (the operand warps keep a row's <= 8 words in registers)
    p.h1_signs = (p.signs && N == 128) ? h1_signs : nullptr;
    return dispatch_kmajor<MODE_DGRAD>(N, false, maps, p, (cudaStream_t)stream);
}

extern "C" int xb_dense_wgrad_workspace_floats(int H_in) { return kNumSMs * (128 * (H_in + 4) + 256 + 2); }

extern "C" int xb_dense_wgrad(const float* Y0, const float* dout0, const float* w2_0, int nh0, const float* Y1,
                              const float* dout1, const float* w2_1, int nh1, const float* X, int64_t B, int H_out,
                              int H_in, float slope, float* workspace, float* dW0, float* db0, float* dw2_0,
                              float* db2_0, float* dW1, float* db1, float* dw2_1, float* db2_1, xb_stream_t stream) {
    if (!Y0 || !dout0 || !w2_0 || !X || !workspace || B <= 0) return XB_E_BADARG;
    if (dW0 && (!db0 || !dw2_0 || !db2_0)) return XB_E_BADARG;
    if ((H_out != 128 && H_out != 256) || (H_in != 128 && H_in != 256) || nh0 < 1 || nh0 > 2) return XB_E_UNSUPPORTED;
    if (Y1 && (!dout1 || !w2_1 || nh1 < 1 || nh1 > 2 || (dW0 && (!dW1 || !db1 || !dw2_1 || !db2_1)))) return XB_E_BADARG;
    if (!al16(Y0) || !al16(X) || !al16(workspace) || (Y1 && !al16(Y1))) return XB_E_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    CUtensorMap my0, my1, mx;
    if (!xb_make_map_f32_2d(&my0, Y0, B, H_out, H_out, 32, 32, 2) ||
        !xb_make_map_f32_2d(&my1, Y1 ? Y1 : Y0, B, H_out, H_out, 32, 32, 2) ||
        !xb_make_map_f32_2d(&mx, X, B, H_in, H_in, 32, 32, 2))
        return XB_E_DRIVER;
    WParams p{};
    p.B = B;
    p.halves = H_out / 128;
    p.n_jobs = (Y1 ? 2 : 1) * p.halves;
    p.H_out = H_out;
    p.slope = slope;
    p.dout[0] = dout0; p.w2[0] = w2_0; p.nh[0] = nh0;
    p.dout[1] = dout1; p.w2[1] = w2_1; p.nh[1] = Y1 ? nh1 : 0;
    const int grid = kNumSMs;
    p.part = workspace;
    p.head_part = workspace + (int64_t)grid * 128 * (H_in + 4);
    p.db2_part = p.head_part + (int64_t)grid * 256;
    // (a TS-form variant — dz^T generated per feature lane into tensor memory — measured slower, 70 vs 57 us at 65 536 x 128:
    // 16 scalar shared-memory reads + 32 broadcast head-gradient reads per thread per k-block make operand generation the
    // bottleneck; the SS form with 8 operand warps stays)
    int rc = H_in == 128 ? launch_wgrad<128>(my0, my1, mx, p, grid, s) : launch_wgrad<256>(my0, my1, mx, p, grid, s);
    if (rc) return rc;
    if (!dW0) return 0;                      // partials only: the caller finishes with xb_mlp_backward_tail
    TailArgs tail{};
    wgrad_reduce_kernel<<<p.n_jobs * 128, 512, 0, s>>>(p.part, p.head_part, p.db2_part, grid, p.n_jobs, p.halves, H_in,
                                                      H_out, dW0, db0, dw2_0, db2_0, nh0, dW1, db1, dw2_1, db2_1,
                                                      Y1 ? nh1 : 0, tail, BinArgs{});
    XB_LAUNCH_CHECK();
    return 0;
}

static int backward_tail_impl(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1, float* dW0,
                              float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1, float* dw2_1, float* db2_1,
                              const float* trunk_ws, int trunk_parts, int obs_dim, float* dWt, float* dbt,
                              const double* dls64, float* dls32, int A, double* norm_ws, int64_t* step_dev,
                              const xb::AdamHyper& hyper, float* lr_out, float* gnorm_out, cudaStream_t stream,
                              const BinArgs& bin = BinArgs{}) {
    if (!wgrad_ws || !dW0 || !db0 || !dw2_0 || !db2_0 || (n_sources == 2 && (!dW1 || !db1 || !dw2_1 || !db2_1)))
        return XB_E_BADARG;
    if ((H_out != 128 && H_out != 256) || (H_in != 128 && H_in != 256) || n_sources < 1 || n_sources > 2) return XB_E_UNSUPPORTED;
    if (trunk_ws && (!dWt || !dbt || trunk_parts < 1 || obs_dim < 1)) return XB_E_BADARG;
    if (dls64 && (!dls32 || A < 1 || A > 512)) return XB_E_BADARG;
    if (norm_ws && !step_dev) return XB_E_BADARG;
    const int grid = kNumSMs, halves = H_out / 128, n_jobs = n_sources * halves;
    const float* part = wgrad_ws;
    const float* head_part = wgrad_ws + (int64_t)grid * 128 * (H_in + 4);
    const float* db2_part = head_part + (int64_t)grid * 256;
    TailArgs tail{trunk_ws, trunk_parts, H_in, obs_dim, dWt, dbt, dls64, dls32, A, norm_ws, step_dev, hyper, lr_out, gnorm_out};
    const int tail_blocks = trunk_ws ? (H_in * (obs_dim + 1) + 15) / 16 : (dls64 ? 1 : 0);
    if (n_jobs * 128 + tail_blocks > xb::kOptMaxGrid) return XB_E_UNSUPPORTED;
    XB_CUDA(launch_pdl(wgrad_reduce_kernel, dim3(n_jobs * 128 + tail_blocks), dim3(512), 0, stream, true, part, head_part, db2_part,
                       grid, n_jobs, halves, H_in, H_out, dW0, db0, dw2_0, db2_0, nh0, dW1, db1, dw2_1, db2_1,
                       n_sources == 2 ? nh1 : 0, tail, bin));
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_mlp_backward_tail(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1,
                                    float* dW0, float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1,
                                    float* dw2_1, float* db2_1, const float* trunk_ws, int trunk_parts, int obs_dim,
                                    float* dWt, float* dbt, const double* dls64, float* dls32, int A,
                                    xb_stream_t stream) {
    xb::AdamHyper none{};
    none.grad_scale = 1.0f;
    return backward_tail_impl(wgrad_ws, H_out, H_in, n_sources, nh0, nh1, dW0, db0, dw2_0, db2_0, dW1, db1, dw2_1, db2_1,
                              trunk_ws, trunk_parts, obs_dim, dWt, dbt, dls64, dls32, A, nullptr, nullptr, none, nullptr,
                              nullptr, (cudaStream_t)stream);
}

extern "C" int xb_mlp_backward_tail_norm(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1,
                                         float* dW0, float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1,
                                         float* dw2_1, float* db2_1, const float* trunk_ws, int trunk_parts, int obs_dim,
                                         float* dWt, float* dbt, const double* dls64, float* dls32, int A,
                                         double* norm_workspace, int64_t* step_dev, float lr0, float lr_end_factor,
                                         int64_t lr_total_iters, float beta1, float beta2, float max_norm, float grad_scale,
                                         float* lr_out, float* gnorm_out, xb_stream_t stream) {
    if (!norm_workspace || !step_dev || !trunk_ws) return XB_E_BADARG;   // needs every gradient of the policy in this launch
    xb::AdamHyper h{lr0, lr_end_factor, beta1, beta2, 0.0f, max_norm, grad_scale, lr_total_iters};
    return backward_tail_impl(wgrad_ws, H_out, H_in, n_sources, nh0, nh1, dW0, db0, dw2_0, db2_0, dW1, db1, dw2_1, db2_1,
                              trunk_ws, trunk_parts, obs_dim, dWt, dbt, dls64, dls32, A, norm_workspace, step_dev, h, lr_out,
                              gnorm_out, (cudaStream_t)stream);
}


// ------------------------------------------------------------------------------------------------ binary-form weight gradients
template <int HIN>
static int launch_wgrad_bin(const CUtensorMap& mx, WBinParams p, int grid, cudaStream_t s) {
    const int stage = (4 + HIN / 32) * 4096, lo = (HIN / 32) * 4096;
    const int avail = kMaxSmem - 1024 - kWMiscBytes;
    int L = 2, S = (avail - L * lo) / stage;
    if (S < 2) return XB_E_UNSUPPORTED;
    if (S > 6) S = 6;
    if ((avail - S * stage) / lo >= 3) L = 3;
    p.stages = S;
    p.lo_bufs = L;
    const int smem = 1024 + S * stage + L * lo + kWMiscBytes;
    auto kern = dense_wgrad_bin_kernel<HIN>;
    XB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    XB_CUDA(launch_pdl(kern, dim3(grid), dim3(kThreads), (size_t)smem, s, true, mx, p));
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_dense_wgrad_bin(const uint32_t* signs, int sign_ld, const float* dout0, int nh0, const float* dout1, int nh1,
                                  const float* X, int64_t B, int H_out, int H_in, float* workspace, xb_stream_t stream) {
    if (!signs || !dout0 || !X || !workspace || B <= 0) return XB_E_BADARG;
    if ((H_out != 128 && H_out != 256) || (H_in != 128 && H_in != 256) || nh0 < 1 || nh0 > 2) return XB_E_UNSUPPORTED;
    if (dout1 && (nh1 < 1 || nh1 > 2)) return XB_E_BADARG;
    const int n_src = dout1 ? 2 : 1;
    if (sign_ld < n_src * (H_out / 32)) return XB_E_BADARG;
    if (!al16(X) || !al16(workspace)) return XB_E_UNSUPPORTED;
    CUtensorMap mx;
    if (!xb_make_map_f32_2d(&mx, X, B, H_in, H_in, 32, 32, 2)) return XB_E_DRIVER;
    WBinParams p{};
    p.B = B;
    p.halves = H_out / 128;
    p.n_jobs = n_src * p.halves;
    p.H_out = H_out;
    p.dout[0] = dout0; p.nh[0] = nh0;
    p.dout[1] = dout1; p.nh[1] = dout1 ? nh1 : 0;
    p.signs = signs;
    p.sign_ld = sign_ld;
    const int grid = kNumSMs;
    p.part = workspace;
    p.head_part = workspace + (int64_t)grid * 128 * (H_in + 4);
    p.db2_part = p.head_part + (int64_t)grid * 256;
    return H_in == 128 ? launch_wgrad_bin<128>(mx, p, grid, (cudaStream_t)stream) : launch_wgrad_bin<256>(mx, p, grid, (cudaStream_t)stream);
}

extern "C" int xb_mlp_backward_tail_bin(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1,
                                        float* dW0, float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1,
                                        float* dw2_1, float* db2_1, const float* trunk_ws, int trunk_parts, int obs_dim,
                                        float* dWt, float* dbt, const double* dls64, float* dls32, int A,
                                        double* norm_workspace, int64_t* step_dev, float lr0, float lr_end_factor,
                                        int64_t lr_total_iters, float beta1, float beta2, float max_norm, float grad_scale,
                                        float* lr_out, float* gnorm_out, const float* W0, const float* b0, const float* w2_0,
                                        const float* W1, const float* b1, const float* w2_1, float slope, xb_stream_t stream) {
    if (!W0 || !b0 || !w2_0 || (n_sources == 2 && (!W1 || !b1 || !w2_1))) return XB_E_BADARG;
    if (norm_workspace && (!step_dev || !trunk_ws)) return XB_E_BADARG;
    xb::AdamHyper h{lr0, lr_end_factor, beta1, beta2, 0.0f, max_norm, grad_scale, lr_total_iters};
    if (!norm_workspace) h.grad_scale = 1.0f;
    BinArgs bin{1, slope, {W0, W1}, {b0, b1}, {w2_0, w2_1}};
    return backward_tail_impl(wgrad_ws, H_out, H_in, n_sources, nh0, nh1, dW0, db0, dw2_0, db2_0, dW1, db1, dw2_1, db2_1,
                              trunk_ws, trunk_parts, obs_dim, dWt, dbt, dls64, dls32, A, norm_workspace, step_dev, h, lr_out,
                              gnorm_out, (cudaStream_t)stream, bin);
}


// The TRAINING forward with the trunk layer generated in the kernel (xb_mlp_fwd_from_obs) and everything xb_dense_fwd2_loss adds:
// the operand warps of the layer-0 CTAs also store h1 = leaky_relu(W0 obs + b0) (h1_out: wgrad's x operand, dgrad's mask), so the
// separate first-layer launch (xb_gather_trunk_fwd's second half) and the read of h1 by this launch disappear.
extern "C" int xb_mlp_fwd_from_obs_train(const float* obs, int ld, int obs_dim, const float* W0, const float* b0, int64_t M, int H,
                                         float slope, const float* Whi0, const float* Wlo0, const float* bias0, float* Y0,
                                         const float* head_w0, const float* head_b0, int n_head0, float* head_out0,
                                         const float* Whi1, const float* Wlo1, const float* bias1, float* Y1,
                                         const float* head_w1, const float* head_b1, int n_head1, float* head_out1, float* h1_out,
                                         const float* scal, const double* adv_stats, int64_t adv_count, float clip_range,
                                         float vf_coef, float ent_coef, float inv_batch, const float* logstd, float* dact,
                                         float* dv, double* loss_partials, uint32_t* loss_ticket, double* scalars, double* dlogstd,
                                         const float* prep_W0, const float* prep_W1, float* prep_thi, float* prep_tlo,
                                         uint32_t* sign_out, xb_stream_t stream) {
    if (!h1_out) return XB_E_BADARG;
    if (scal && (!dact || !dv || !loss_partials || !loss_ticket || !scalars || ((uintptr_t)scal & 15u))) return XB_E_BADARG;
    if (adv_stats && adv_count <= 0) return XB_E_BADARG;
    if (logstd && !dlogstd) return XB_E_BADARG;
    const float* Whi[2] = {Whi0, Whi1};
    const float* Wlo[2] = {Wlo0, Wlo1};
    const float* bias[2] = {bias0, bias1};
    float* Y[2] = {Y0, Y1};
    const float* hw[2] = {head_w0, head_w1};
    const float* hb[2] = {head_b0, head_b1};
    const int nh[2] = {n_head0, n_head1};
    float* ho[2] = {head_out0, head_out1};
    FusedLoss L{(const float4*)scal, adv_stats, adv_stats ? 1.0 / (double)adv_count : 0.0, clip_range, vf_coef, ent_coef,
                inv_batch, logstd ? 1 : 0, logstd, dact, dv, loss_partials, loss_ticket, scalars, dlogstd};
    const float* pw[2] = {prep_W0, prep_W1};
    TrunkArgs t{obs, ld, obs_dim, W0, b0, nullptr, nullptr, 0, 0.f, 0, h1_out};
    return dense_fwd_impl(nullptr, &t, M, H, H, slope, 2, Whi, Wlo, bias, Y, hw, hb, nh, ho, 1, stream, scal ? &L : nullptr, pw,
                          prep_thi, prep_tlo, sign_out);
}
