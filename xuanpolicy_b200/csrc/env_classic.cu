// env_classic.cu — batched CartPole-v1 / Pendulum-v1 / MountainCar-v0 (gym's, and the reference's 4-frame wrapper) /
// Acrobot-v1 step + auto-reset, one thread per environment.
//
// Replaces the per-env Python loop of DummyVecEnv_Gym.step_wait (xuance/environment/gym/gym_vec_env.py:201-212)
// over Gym_Env.step (xuance/environment/gym/gym_env.py:43-49) over gym 0.26.2's CartPoleEnv / PendulumEnv /
// TimeLimit (third party, not vendored; equations per SURVEY.md App. A, reset stream per App. B).
//
// Bit-exactness contract: fp64 state lives in registers for the whole step; every fp64 operation is an
// individually rounded __dadd_rn/__dmul_rn/__ddiv_rn (no FMA contraction — this TU is also built with
// -fmad=false); sin/cos are correctly rounded (crtrig.cuh); squares are v*v.  Under identical actions the
// fp64 states, float32 observations/rewards, flags, counters and reset draws equal the CPU oracle's bit for bit.
//
// Memory traffic per env-step (no reset): CartPole 4x8 R + 4x8 W state, 8 action, 4+4 elapsed, 8+8 score,
// 16 obs (+16 next_obs), 4 rew, 2 flags, 4+8 episode outputs; all accesses are SoA and fully coalesced,
// observations are one float4 per env.
#include "common.cuh"
#include "sample.cuh"
#include "crtrig.cuh"
#include "normalize.cuh"

namespace xb {

// ---------------------------------------------------------------- numpy PCG64 (XSL-RR 128/64) ----------------
struct Pcg64 {
    uint64_t hi, lo, inc_hi, inc_lo;
};

__device__ __forceinline__ uint64_t pcg64_next(Pcg64& g) {
    const uint64_t MH = 0x2360ED051FC65DA4ULL, ML = 0x4385DF649FCCF645ULL;
    // state = state * mult + inc  (mod 2^128)
    uint64_t lo = g.lo * ML;
    uint64_t hi = __umul64hi(g.lo, ML) + g.hi * ML + g.lo * MH;
    uint64_t nlo = lo + g.inc_lo;
    uint64_t carry = nlo < lo ? 1ULL : 0ULL;
    g.hi = hi + g.inc_hi + carry;
    g.lo = nlo;
    uint64_t x = g.hi ^ g.lo;
    unsigned rot = (unsigned)(g.hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}
// Generator.uniform: low + (high - low) * next_double, two roundings
__device__ __forceinline__ double pcg64_uniform(Pcg64& g, double low, double range) {
    double u = __dmul_rn((double)(pcg64_next(g) >> 11), 1.0 / 9007199254740992.0);
    return __dadd_rn(low, __dmul_rn(range, u));
}

constexpr double kPi = 3.141592653589793;

// ---------------------------------------------------------------- per-env dynamics ---------------------------
struct CartPole {
    static constexpr int kObsVec = 1;   // float4s per observation row
    static constexpr bool kTrigCache = false;
    static constexpr int S = 4;
    typedef int64_t action_t;
    static constexpr bool kDiscrete = true;
    static constexpr int kActions = 2;
    __device__ static void draw(double (&st)[4], Pcg64& g) {
#pragma unroll
        for (int k = 0; k < 4; ++k) st[k] = pcg64_uniform(g, -0.05, 0.05 - (-0.05));
    }
    __device__ static float4 observe(const double (&st)[4]) {
        return make_float4((float)st[0], (float)st[1], (float)st[2], (float)st[3]);
    }
    // returns reward (fp64); sets terminated
    __device__ static double step(double (&st)[4], action_t action, bool& terminated) {
        const double gravity = 9.8, masspole = 0.1, total_mass = 0.1 + 1.0, length = 0.5;
        const double polemass_length = 0.1 * 0.5, force_mag = 10.0, tau = 0.02;
        const double theta_thr = 12 * 2 * kPi / 360, x_thr = 2.4;
        double x = st[0], x_dot = st[1], theta = st[2], theta_dot = st[3];
        double force = action == 1 ? force_mag : -force_mag;
        double s, c;
        sincos_cr(theta, &s, &c);
        double td2 = __dmul_rn(theta_dot, theta_dot);
        double temp = __ddiv_rn(__dadd_rn(force, __dmul_rn(__dmul_rn(polemass_length, td2), s)), total_mass);
        double c2 = __dmul_rn(c, c);
        double denom = __dmul_rn(length, __dsub_rn(4.0 / 3.0, __ddiv_rn(__dmul_rn(masspole, c2), total_mass)));
        double thetaacc = __ddiv_rn(__dsub_rn(__dmul_rn(gravity, s), __dmul_rn(c, temp)), denom);
        double xacc = __dsub_rn(temp, __ddiv_rn(__dmul_rn(__dmul_rn(polemass_length, thetaacc), c), total_mass));
        x = __dadd_rn(x, __dmul_rn(tau, x_dot));
        x_dot = __dadd_rn(x_dot, __dmul_rn(tau, xacc));
        theta = __dadd_rn(theta, __dmul_rn(tau, theta_dot));
        theta_dot = __dadd_rn(theta_dot, __dmul_rn(tau, thetaacc));
        st[0] = x; st[1] = x_dot; st[2] = theta; st[3] = theta_dot;
        terminated = (x < -x_thr) || (x > x_thr) || (theta < -theta_thr) || (theta > theta_thr);
        return 1.0;
    }
};

struct Pendulum {
    static constexpr int kObsVec = 1;   // float4s per observation row
    static constexpr bool kTrigCache = true;   // sin/cos(theta) of the observation are the next step's dynamics inputs
    static constexpr int S = 2;
    typedef float action_t;
    static constexpr bool kDiscrete = false;
    static constexpr int kActions = 1;
    __device__ static void draw(double (&st)[2], Pcg64& g) {
        st[0] = pcg64_uniform(g, -kPi, kPi - (-kPi));
        st[1] = pcg64_uniform(g, -1.0, 1.0 - (-1.0));
    }
    __device__ static float4 observe_sc(const double (&st)[2], double s, double c) {   // s, c = sin, cos of st[0]
        return make_float4((float)c, (float)s, (float)st[1], 0.0f);
    }
    __device__ static float4 observe(const double (&st)[2]) {
        double s, c;
        sincos_cr(st[0], &s, &c);
        return observe_sc(st, s, c);
    }
    __device__ static double angle_normalize(double x) {
        const double two_pi = 2 * kPi;
        double r = fmod(__dadd_rn(x, kPi), two_pi);  // fmod is exact; then numpy's floor-mod sign fix
        if (r != 0.0) {
            if (r < 0.0) r = __dadd_rn(r, two_pi);
        } else {
            r = 0.0;
        }
        return __dsub_rn(r, kPi);
    }
    __device__ static double step(double (&st)[2], action_t action, bool& terminated) {
        double s, c;
        sincos_cr(st[0], &s, &c);
        return step_sc(st, action, terminated, s);
    }
    // the same step with sin(theta) supplied by the caller (the previous step's observation already evaluated it)
    __device__ static double step_sc(double (&st)[2], action_t action, bool& terminated, double s) {
        const double dt = 0.05;
        double th = st[0], thdot = st[1];
        float u32 = action < -2.0f ? -2.0f : (action > 2.0f ? 2.0f : action);
        double u = (double)u32;  // pinned numpy 1.21.6 promotion: float32 scalar (x) python float -> float64
        double an = angle_normalize(th);
        double costs = __dadd_rn(__dadd_rn(__dmul_rn(an, an), __dmul_rn(0.1, __dmul_rn(thdot, thdot))),
                                 __dmul_rn(0.001, __dmul_rn(u, u)));
        double newthdot = __dadd_rn(thdot, __dmul_rn(__dadd_rn(__dmul_rn(15.0, s), __dmul_rn(3.0, u)), dt));
        newthdot = newthdot < -8.0 ? -8.0 : (newthdot > 8.0 ? 8.0 : newthdot);
        double newth = __dadd_rn(th, __dmul_rn(newthdot, dt));
        st[0] = newth; st[1] = newthdot;
        terminated = false;
        return -costs;
    }
};


// gym 0.26.2 MountainCarEnv (gym/envs/classic_control/mountain_car.py; xuance config
// xuance/configs/ppo/classic_control/MountainCar-v0.yaml), TimeLimit 200.  Operation order of step():
//   velocity += (action - 1) * force + math.cos(3 * position) * (-gravity)
//   velocity = clip(velocity, -max_speed, max_speed); position += velocity; position = clip(position, min, max)
//   if position == min_position and velocity < 0: velocity = 0
//   terminated = position >= goal_position and velocity >= goal_velocity; reward = -1.0
// reset(): state = [uniform(-0.6, -0.4), 0].
struct MountainCar {
    static constexpr int kObsVec = 1;   // float4s per observation row
    static constexpr bool kTrigCache = false;
    static constexpr int S = 2;
    typedef int64_t action_t;
    static constexpr bool kDiscrete = true;
    static constexpr int kActions = 3;
    __device__ static void draw(double (&st)[2], Pcg64& g) {
        st[0] = pcg64_uniform(g, -0.6, -0.4 - (-0.6));
        st[1] = 0.0;
    }
    __device__ static float4 observe(const double (&st)[2]) { return make_float4((float)st[0], (float)st[1], 0.0f, 0.0f); }
    __device__ static double step(double (&st)[2], action_t action, bool& terminated) {
        const double force = 0.001, gravity = 0.0025, max_speed = 0.07, min_pos = -1.2, max_pos = 0.6, goal_pos = 0.5;
        double position = st[0], velocity = st[1];
        double s, c;
        sincos_cr(__dmul_rn(3.0, position), &s, &c);
        const double push = __dmul_rn((double)(action - 1), force);
        velocity = __dadd_rn(velocity, __dadd_rn(push, __dmul_rn(c, -gravity)));
        velocity = velocity < -max_speed ? -max_speed : (velocity > max_speed ? max_speed : velocity);
        position = __dadd_rn(position, velocity);
        position = position < min_pos ? min_pos : (position > max_pos ? max_pos : position);
        if (position == min_pos && velocity < 0.0) velocity = 0.0;
        st[0] = position; st[1] = velocity;
        terminated = position >= goal_pos && velocity >= 0.0;
        return -1.0;
    }
};

// MountainCar-v0 AS THE REFERENCE DEFINES IT: `make_envs` wraps every env id containing "MountainCar" in
// xuance/environment/gym/gym_env.py:50-83 `MountainCar(Gym_Env)` (selected at xuance/environment/__init__.py:66-67): the
// observation is the concatenation of the last FOUR frames, oldest first (`LazyFrames(list(self.frames))`, deque maxlen 4,
// gym_env.py:227-254), shape (8,); `reset()` fills all four frames with the reset observation (:67-68).  The three previous
// float32 frames ride in the fp64 state slots 2..7 (exact), so the generic step / reset / rollout kernels need no extra
// argument; slots 0..1 are gym's (position, velocity) with the physics of `MountainCar` above, bit for bit.
struct MountainCarStack {
    static constexpr int kObsVec = 2;
    static constexpr bool kTrigCache = false;
    static constexpr int S = 8;
    typedef int64_t action_t;
    static constexpr bool kDiscrete = true;
    static constexpr int kActions = 3;
    __device__ static void draw(double (&st)[8], Pcg64& g) {
        double b[2];
        MountainCar::draw(b, g);
        st[0] = b[0]; st[1] = b[1];
#pragma unroll
        for (int k = 0; k < 3; ++k) {           // for i in range(num_stack): frames.append(obs)
            st[2 + 2 * k] = (double)(float)b[0];
            st[3 + 2 * k] = (double)(float)b[1];
        }
    }
    __device__ static void observe(const double (&st)[8], float4 (&o)[2]) {
        o[0] = make_float4((float)st[2], (float)st[3], (float)st[4], (float)st[5]);
        o[1] = make_float4((float)st[6], (float)st[7], (float)st[0], (float)st[1]);
    }
    __device__ static double step(double (&st)[8], action_t action, bool& terminated) {
        double b[2] = {st[0], st[1]};
        const float fp = (float)b[0], fv = (float)b[1];       // the frame appended by the previous step / reset
        const double r = MountainCar::step(b, action, terminated);
        st[2] = st[4]; st[3] = st[5]; st[4] = st[6]; st[5] = st[7];
        st[6] = (double)fp; st[7] = (double)fv;
        st[0] = b[0]; st[1] = b[1];
        return r;
    }
};

// gym 0.26.2 AcrobotEnv (gym/envs/classic_control/acrobot.py; xuance config xuance/configs/ppo/classic_control/Acrobot-v1.yaml),
// "book" dynamics, TimeLimit 500, restated from the published algorithm (operation order = Python's left-to-right):
//   s_augmented = append(state, AVAIL_TORQUE[a]);  ns = rk4(_dsdt, s_augmented, [0, 0.2])   (one RK4 step, dt = 0.2)
//   ns[0], ns[1] = wrap(., -pi, pi);  ns[2] = bound(., -4pi, 4pi);  ns[3] = bound(., -9pi, 9pi)
//   terminated = -cos(s0) - cos(s1 + s0) > 1.0;  reward = -1.0 (0.0 on termination)
//   obs = float32([cos s0, sin s0, cos s1, sin s1, s2, s3]);  reset: uniform(-0.1, 0.1, 4).astype(float32)
// With m1 = m2 = l1 = I1 = I2 = 1, lc1 = lc2 = 0.5, g = 9.8 the constant sub-products of _dsdt fold exactly
// (x*1.0, x*0.5 and 0.5*9.8 are exact), which leaves the roundings written out below.
struct Acrobot {
    static constexpr int kObsVec = 2;
    static constexpr bool kTrigCache = false;
    static constexpr int S = 4;
    typedef int64_t action_t;
    static constexpr bool kDiscrete = true;
    static constexpr int kActions = 3;
    __device__ static void draw(double (&st)[4], Pcg64& g) {
#pragma unroll
        for (int k = 0; k < 4; ++k) st[k] = (double)(float)pcg64_uniform(g, -0.1, 0.1 - (-0.1));   // .astype(np.float32)
    }
    __device__ static void observe(const double (&st)[4], float4 (&o)[2]) {
        double s0, c0, s1, c1;
        sincos_cr(st[0], &s0, &c0);
        sincos_cr(st[1], &s1, &c1);
        o[0] = make_float4((float)c0, (float)s0, (float)c1, (float)s1);
        o[1] = make_float4((float)st[2], (float)st[3], 0.0f, 0.0f);
    }
    // _dsdt: (theta1, theta2, dtheta1, dtheta2, a) -> (dtheta1, dtheta2, ddtheta1, ddtheta2)
    __device__ static void dsdt(const double (&y)[4], double a, double (&k)[4]) {
        const double theta1 = y[0], theta2 = y[1], dtheta1 = y[2], dtheta2 = y[3];
        const double half_pi = kPi / 2.0;
        double s2, c2, sn, cphi2, cphi1;
        sincos_cr(theta2, &s2, &c2);
        sincos_cr(__dsub_rn(__dadd_rn(theta1, theta2), half_pi), &sn, &cphi2);
        sincos_cr(__dsub_rn(theta1, half_pi), &sn, &cphi1);
        // d1 = m1*lc1**2 + m2*(l1**2 + lc2**2 + 2*l1*lc2*cos(theta2)) + I1 + I2
        const double d1 = __dadd_rn(__dadd_rn(__dadd_rn(0.25, __dadd_rn(1.25, c2)), 1.0), 1.0);
        // d2 = m2*(lc2**2 + l1*lc2*cos(theta2)) + I2
        const double d2 = __dadd_rn(__dadd_rn(0.25, __dmul_rn(0.5, c2)), 1.0);
        const double phi2 = __dmul_rn(0.5 * 9.8, cphi2);                       // m2*lc2*g*cos(theta1 + theta2 - pi/2)
        // phi1 = -m2*l1*lc2*dtheta2**2*sin(theta2) - 2*m2*l1*lc2*dtheta2*dtheta1*sin(theta2) + (m1*lc1 + m2*l1)*g*cos(theta1 - pi/2) + phi2
        const double tA = __dmul_rn(__dmul_rn(-0.5, __dmul_rn(dtheta2, dtheta2)), s2);
        const double tB = __dmul_rn(__dmul_rn(dtheta2, dtheta1), s2);
        const double tC = __dmul_rn(1.5 * 9.8, cphi1);
        const double phi1 = __dadd_rn(__dadd_rn(__dsub_rn(tA, tB), tC), phi2);
        // book: ddtheta2 = (a + d2/d1*phi1 - m2*l1*lc2*dtheta1**2*sin(theta2) - phi2) / (m2*lc2**2 + I2 - d2**2/d1)
        const double num = __dsub_rn(__dsub_rn(__dadd_rn(a, __dmul_rn(__ddiv_rn(d2, d1), phi1)),
                                               __dmul_rn(__dmul_rn(0.5, __dmul_rn(dtheta1, dtheta1)), s2)), phi2);
        const double den = __dsub_rn(1.25, __ddiv_rn(__dmul_rn(d2, d2), d1));
        const double ddtheta2 = __ddiv_rn(num, den);
        const double ddtheta1 = __ddiv_rn(-__dadd_rn(__dmul_rn(d2, ddtheta2), phi1), d1);
        k[0] = dtheta1; k[1] = dtheta2; k[2] = ddtheta1; k[3] = ddtheta2;
    }
    __device__ static double wrap(double x, double m, double M) {
        const double diff = __dsub_rn(M, m);
        while (x > M) x = __dsub_rn(x, diff);
        while (x < m) x = __dadd_rn(x, diff);
        return x;
    }
    __device__ static double step(double (&st)[4], action_t action, bool& terminated) {
        const double a = (double)(action - 1);                                  // AVAIL_TORQUE = [-1.0, 0.0, +1]
        const double dt = 0.2, dt2 = 0.2 / 2.0, dt6 = 0.2 / 6.0;
        double k1[4], k2[4], k3[4], k4[4], y[4];
        dsdt(st, a, k1);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = __dadd_rn(st[i], __dmul_rn(dt2, k1[i]));
        dsdt(y, a, k2);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = __dadd_rn(st[i], __dmul_rn(dt2, k2[i]));
        dsdt(y, a, k3);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = __dadd_rn(st[i], __dmul_rn(dt, k3[i]));
        dsdt(y, a, k4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {   // y0 + dt / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)
            const double sum = __dadd_rn(__dadd_rn(__dadd_rn(k1[i], __dmul_rn(2.0, k2[i])), __dmul_rn(2.0, k3[i])), k4[i]);
            y[i] = __dadd_rn(st[i], __dmul_rn(dt6, sum));
        }
        y[0] = wrap(y[0], -kPi, kPi);
        y[1] = wrap(y[1], -kPi, kPi);
        const double v1 = 4 * kPi, v2 = 9 * kPi;
        y[2] = fmin(fmax(y[2], -v1), v1);
        y[3] = fmin(fmax(y[3], -v2), v2);
#pragma unroll
        for (int i = 0; i < 4; ++i) st[i] = y[i];
        double s0, c0, s10, c10;
        sincos_cr(st[0], &s0, &c0);
        sincos_cr(__dadd_rn(st[1], st[0]), &s10, &c10);
        terminated = __dsub_rn(-c0, c10) > 1.0;
        return terminated ? 0.0 : -1.0;
    }
};

// one-float4 observation rows: array form of observe() for the kernels below
template <class Env>
__device__ __forceinline__ void observe_row(const double (&st)[Env::S], float4 (&o)[Env::kObsVec]) {
    if constexpr (Env::kObsVec == 1) o[0] = Env::observe(st);
    else Env::observe(st, o);
}
template <class Env>
__device__ __forceinline__ void put_row(float4* dst, int64_t e, const float4 (&o)[Env::kObsVec]) {
#pragma unroll
    for (int v = 0; v < Env::kObsVec; ++v) dst[e * Env::kObsVec + v] = o[v];
}

// ---------------------------------------------------------------- kernels ------------------------------------
template <class Env>
__device__ __forceinline__ Pcg64 load_rng(const uint64_t* rng, int64_t N, int64_t e) {
    return Pcg64{rng[e], rng[N + e], rng[2 * N + e], rng[3 * N + e]};
}

template <class Env>
__global__ void __launch_bounds__(128) env_reset_kernel(double* __restrict__ state, uint64_t* __restrict__ rng,
                                                         int32_t* __restrict__ elapsed, double* __restrict__ ep_score,
                                                         float4* __restrict__ obs, int n_draws, int64_t N) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    Pcg64 g = load_rng<Env>(rng, N, e);
    double st[Env::S];
#pragma unroll
    for (int k = 0; k < Env::S; ++k) st[k] = state[k * N + e];
    for (int d = 0; d < n_draws; ++d) Env::draw(st, g);
#pragma unroll
    for (int k = 0; k < Env::S; ++k) state[k * N + e] = st[k];
    rng[e] = g.hi;
    rng[N + e] = g.lo;
    elapsed[e] = 0;
    ep_score[e] = 0.0;
    float4 o[Env::kObsVec];
    observe_row<Env>(st, o);
    put_row<Env>(obs, e, o);
}

template <class Env>
__global__ void __launch_bounds__(128)
    env_step_kernel(double* __restrict__ state, uint64_t* __restrict__ rng, int32_t* __restrict__ elapsed,
                    double* __restrict__ ep_score, const typename Env::action_t* __restrict__ actions,
                    float4* __restrict__ obs, float4* __restrict__ next_obs, float* __restrict__ rew,
                    uint8_t* __restrict__ term, uint8_t* __restrict__ trunc, float4* __restrict__ reset_obs,
                    int32_t* __restrict__ ep_step_out, double* __restrict__ ep_score_out,
                    double* __restrict__ ep_stats, int max_steps, int64_t N) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    double st[Env::S];
#pragma unroll
    for (int k = 0; k < Env::S; ++k) st[k] = state[k * N + e];
    typename Env::action_t a = actions[e];
    int32_t el = elapsed[e];
    double score = ep_score[e];

    bool terminated;
    double reward = Env::step(st, a, terminated);
    el += 1;                                   // TimeLimit.step / Gym_Env.step
    bool truncated = el >= max_steps;
    score = __dadd_rn(score, reward);          // Gym_Env._episode_score += reward (fp64)

    float4 o[Env::kObsVec];
    observe_row<Env>(st, o);
    put_row<Env>(obs, e, o);
    rew[e] = (float)reward;
    term[e] = terminated ? 1 : 0;
    trunc[e] = truncated ? 1 : 0;
    ep_step_out[e] = el;
    ep_score_out[e] = score;

    if (terminated || truncated) {             // gym_vec_env.py:207-209: immediate reset, reset obs travels aside
        if (ep_stats) {                        // running totals for the episode log (ppoclip_agent.py:102-109)
            atomicAdd(&ep_stats[0], 1.0);
            atomicAdd(&ep_stats[1], score);
            atomicAdd(&ep_stats[2], (double)el);
        }
        Pcg64 g = load_rng<Env>(rng, N, e);
        Env::draw(st, g);
        rng[e] = g.hi;
        rng[N + e] = g.lo;
        el = 0;
        score = 0.0;
        observe_row<Env>(st, o);
        put_row<Env>(reset_obs, e, o);
    }
    if (next_obs) put_row<Env>(next_obs, e, o);
#pragma unroll
    for (int k = 0; k < Env::S; ++k) state[k * N + e] = st[k];
    elapsed[e] = el;
    ep_score[e] = score;
}

// ------------------------------------------------------------------------------------------------ fused rollout step
// One launch per vector step of the device-resident rollout: sample the action + its log-prob from the policy outputs
// (PPOCLIP_Agent._action, ppoclip_agent.py:50-57), step the env (DummyVecEnv_Gym.step_wait, gym_vec_env.py:200-212) and
// store the transition into rollout row t (DummyOnPolicyBuffer.store, memory_tools.py:196-204) — the three per-env
// kernels sample_* / env_step / store back to back in one thread, the action never leaves registers.
struct RolloutStepArgs {
    // policy outputs for rows [0, N): logits [N][2] (Discrete(2)) or mu [N][1] + logstd [1]; value [N]
    const float* act_param;
    const float* logstd;
    const float* val;
    uint64_t seed;
    const uint64_t* counter_dev;
    uint64_t offset;
    // env state (SoA) and per-step outputs, as in env_step_kernel
    double* state;
    uint64_t* rng;
    int32_t* elapsed;
    double* ep_score;
    float4* obs;          // terminal-inclusive observation of this step
    float4* next_obs;     // reset-substituted observation the policy acts on next
    float* rew;
    uint8_t* term;
    uint8_t* trunc;
    float4* reset_obs;
    int32_t* ep_step_out;
    double* ep_score_out;
    double* ep_stats;
    int max_steps;
    // the observation the action was computed from, and the action / log-prob scratch the agent exposes
    const float4* x_in;
    void* act_out;
    float* logp_out;
    // rollout buffer row t
    float4* obs_row;
    float* act_row;
    float* rew_row;
    float* val_row;
    float* term_row;
    uint8_t* trunc_row;
    float* logp_row;
    const float* rew_scale;   // nullable: rewards are divided by *rew_scale and clipped to +-rew_clip (use_rewnorm)
    float rew_clip;
    // nullable pair: V(terminal obs of the previous step) [N] -> the previous rollout row's bootstrap values
    const float* boot_src;
    float* boot_row;
    // nullable, fp64 [3][N]: (theta, sin theta, cos theta) of the last observation this kernel produced.  sin/cos are pure
    // functions of theta, so a row is used only when its key equals the current theta bit for bit — a stale or
    // never-written row (key NaN) just means the values are recomputed.  Halves the correctly-rounded trig work of Pendulum.
    double* trig_cache;
    int64_t N;
    // optional (stats.partials != NULL): running statistics carried by this launch (normalize.cuh StepStats).  With
    // stats.obs_state_in set, x_in holds RAW observations and the stored row is their normalised form (the same arithmetic
    // as the forward kernel's, agent.py:112-113); the next observations' moments are merged into stats.obs_state_out.
    StepStats stats;
#ifdef XB_STEP_TS
    unsigned long long* ts;
#endif
};

template <class Env>
__global__ void __launch_bounds__(128) rollout_step_kernel(RolloutStepArgs a) {
    // launched with the programmatic-serialization attribute (common.cuh): resident early, starts when the forward before it
    // has completed; the next forward may then run its weight-only prologue underneath this kernel
#ifdef XB_STEP_TS
    unsigned long long* const ts = (blockIdx.x == 0 && threadIdx.x == 0) ? a.ts : nullptr;
    a.stats.ts = threadIdx.x == 0 ? a.ts : nullptr;
#endif
    XB_STEP_STAMP(ts, 100);
    pdl_wait();
    XB_STEP_STAMP(ts, 101);
    pdl_trigger();
    constexpr int V = Env::kObsVec, D = 4 * V;
    __shared__ double stat_smem[(2 * D + 3) * 32];
    __shared__ bool stat_flag;
    const bool with_stats = a.stats.partials != nullptr;
    double acc[2 * D + 3];
#pragma unroll
    for (int k = 0; k < 2 * D + 3; ++k) acc[k] = 0.0;
    const int64_t N = a.N;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < N) {
    // ---- sample (sample.cuh)
    const Philox ph = philox_setup(a.seed, a.counter_dev, a.offset);
    typename Env::action_t act;
    float logp;
    if (Env::kDiscrete) {
        act = (typename Env::action_t)sample_categorical_one(a.act_param + e * Env::kActions, Env::kActions, e, ph, &logp);
        ((int64_t*)a.act_out)[e] = (int64_t)act;
        a.act_row[e] = (float)act;
    } else {
        float x;
        logp = sample_gaussian_one(a.act_param + e, a.logstd, 1, e, ph, &x);
        act = (typename Env::action_t)x;
        ((float*)a.act_out)[e] = x;
        a.act_row[e] = x;
    }
    a.logp_out[e] = logp;
    a.logp_row[e] = logp;
    if (with_stats && a.stats.obs_state_in) {          // stored observation = the normalised one the policy acted on
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float4 q = a.x_in[e * V + v];
            const float in[4] = {q.x, q.y, q.z, q.w};
            float o4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int d = 4 * v + k;
                float mean, den;
                o4[k] = 0.f;
                if (d < a.stats.dim) {
                    norm_coeffs(a.stats.obs_state_in, D, d, mean, den);
                    o4[k] = norm_apply(in[k], mean, den, a.stats.obs_clip);
                }
            }
            a.obs_row[e * V + v] = make_float4(o4[0], o4[1], o4[2], o4[3]);
        }
    } else {
#pragma unroll
        for (int v = 0; v < V; ++v) a.obs_row[e * V + v] = a.x_in[e * V + v];
    }
    a.val_row[e] = a.val[e];
    if (a.boot_row) a.boot_row[e] = a.boot_src[e];   // V(terminal obs) for envs truncated at step t-1 (ppoclip_agent.py:99)
    // ---- env step (identical arithmetic to env_step_kernel)
    double st[Env::S];
#pragma unroll
    for (int k = 0; k < Env::S; ++k) st[k] = a.state[k * N + e];
    int32_t el = a.elapsed[e];
    double score = a.ep_score[e];
    bool terminated;
    double reward;
    float4 o[V];
    double sc_s = 0.0, sc_c = 0.0;
    if constexpr (Env::kTrigCache) {
        bool hit = false;
        if (a.trig_cache && a.trig_cache[e] == st[0]) {
            sc_s = a.trig_cache[N + e];
            hit = true;
        }
        if (!hit) sincos_cr(st[0], &sc_s, &sc_c);
        reward = Env::step_sc(st, act, terminated, sc_s);
        sincos_cr(st[0], &sc_s, &sc_c);            // of the NEW theta: this step's observation, the next step's dynamics
        o[0] = Env::observe_sc(st, sc_s, sc_c);
    } else {
        reward = Env::step(st, act, terminated);
        observe_row<Env>(st, o);
    }
    el += 1;
    const bool truncated = el >= a.max_steps;
    score = __dadd_rn(score, reward);
    put_row<Env>(a.obs, e, o);
    const float r32 = (float)reward;
    a.rew[e] = r32;
    a.term[e] = terminated ? 1 : 0;
    a.trunc[e] = truncated ? 1 : 0;
    a.ep_step_out[e] = el;
    a.ep_score_out[e] = score;
    if (terminated || truncated) {
        if (a.ep_stats) {
            atomicAdd(&a.ep_stats[0], 1.0);
            atomicAdd(&a.ep_stats[1], score);
            atomicAdd(&a.ep_stats[2], (double)el);
        }
        Pcg64 g = load_rng<Env>(a.rng, N, e);
        Env::draw(st, g);
        a.rng[e] = g.hi;
        a.rng[N + e] = g.lo;
        el = 0;
        score = 0.0;
        if constexpr (Env::kTrigCache) {
            sincos_cr(st[0], &sc_s, &sc_c);
            o[0] = Env::observe_sc(st, sc_s, sc_c);
        } else {
            observe_row<Env>(st, o);
        }
        put_row<Env>(a.reset_obs, e, o);
    }
    if (a.next_obs) put_row<Env>(a.next_obs, e, o);
    if constexpr (Env::kTrigCache) {
        if (a.trig_cache) {
            a.trig_cache[e] = st[0];
            a.trig_cache[N + e] = sc_s;
            a.trig_cache[2 * N + e] = sc_c;
        }
    }
#pragma unroll
    for (int k = 0; k < Env::S; ++k) a.state[k * N + e] = st[k];
    a.elapsed[e] = el;
    a.ep_score[e] = score;
    // ---- store the rest of the transition (store_kernel)
    float r = r32;
    if (a.rew_scale) {
        r = r / *a.rew_scale;
        r = fminf(fmaxf(r, -a.rew_clip), a.rew_clip);
    }
    a.rew_row[e] = r;
    a.term_row[e] = terminated ? 1.0f : 0.0f;
    if (a.trunc_row) a.trunc_row[e] = truncated ? 1 : 0;
    // ---- running statistics (normalize.cu returns_track_kernel / moments): this env's contributions
    if (with_stats) {
        if (a.stats.obs_state_in) {                     // moments of the observation the policy acts on NEXT
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const float in[4] = {o[v].x, o[v].y, o[v].z, o[v].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    acc[4 * v + k] = (double)in[k];
                    acc[D + 4 * v + k] = (double)in[k] * (double)in[k];
                }
            }
        }
        if (a.stats.returns) {
            // (1 - terminals) * gamma * returns + rewards (ppoclip_agent.py:87); A2C: gamma * returns + rewards (a2c_agent.py:85)
            double R = ((terminated && a.stats.mask_terminal) ? 0.0 : 1.0) * a.stats.gamma * a.stats.returns[e] + (double)r32;
            if (terminated || truncated) {
                acc[2 * D] = R;
                acc[2 * D + 1] = R * R;
                acc[2 * D + 2] = 1.0;
                R = 0.0;
            }
            a.stats.returns[e] = R;
        }
    }
    }   // e < N
    XB_STEP_STAMP(ts, 104);
    if (with_stats) step_stats_finish<D>(a.stats, acc, N, stat_smem, &stat_flag);
}

// ------------------------------------------------------------------------------------------------ evaluation step
// One launch per vector step of the evaluation loop (PPOCLIP_Agent.test, ppoclip_agent.py:113-165): sample the action from the
// policy outputs, step the env with auto-reset, append the scores of the episodes that ended to a queue in env order, and merge
// the moments of the observations the policy acts on next into the observation statistics (`obs_rms.update(obs)` at the top of
// the next loop iteration).  Sampling, env functors, trig cache and statistics are those of rollout_step_kernel; nothing is
// stored for training.
struct EvalStepArgs {
    const float* act_param;       // logits [N][A] or mu [N][1]
    const float* logstd;          // [1] (Gaussian)
    const uint64_t* key;          // Philox key of this evaluation
    uint64_t* step;               // evaluation step = the Philox counter's high half; +1 per step that runs
    double* state;
    uint64_t* rng;
    int32_t* elapsed;
    double* ep_score;
    float4* next_obs;             // reset-substituted observation the policy acts on next
    double* trig_cache;
    int max_steps;
    void* act_tape;               // nullable: [tape_steps][N] sampled actions, row = evaluation step
    int64_t tape_steps;
    double* scores;               // the episode queue, fp64 [cap]
    int64_t* count;               // entries in the queue
    const int64_t* test_episode;
    int64_t cap;
    uint64_t* ws;                 // [0] start ticket, [1] statistics ticket, [2, 2 + grid) look-back words
    int64_t N;
    StepStats stats;              // obs_state_in = the live statistics (nullable), obs_state_out = the merge candidate
};

__device__ __forceinline__ void st_release_u64(uint64_t* p, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_u64(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// look-back word of a CTA: status in the top two bits, a count of finished episodes in the low 32
constexpr uint64_t kLbAggregate = 1ull << 62, kLbInclusive = 2ull << 62, kLbValue = 0xffffffffull;

template <class Env>
__global__ void __launch_bounds__(128) eval_step_kernel(EvalStepArgs a) {
    constexpr int V = Env::kObsVec, D = 4 * V;
    __shared__ double stat_smem[(2 * D + 3) * 32];
    __shared__ bool stat_flag;
    __shared__ int64_t s_c0, s_base;
    __shared__ uint64_t s_step;
    __shared__ unsigned s_cta, s_warp[4];
    __shared__ bool s_active;
    // The stop rule reads the count the previous step left.  It is written only by this launch's last CTA, after every CTA
    // has taken its statistics ticket, so every CTA reads the same value.  A launch that finds the queue full changes nothing.
    if (threadIdx.x == 0) {
        s_c0 = *a.count;
        s_active = s_c0 < *a.test_episode;
        if (s_active) {
            s_step = *a.step;
            s_cta = ticket_take((unsigned int*)a.ws);     // CTAs take their place in env order in the order they start
        }
    }
    __syncthreads();
    if (!s_active) return;
    const int64_t N = a.N;
    const unsigned cta = s_cta;
    const uint64_t step = s_step;
    const int64_t e = (int64_t)cta * blockDim.x + threadIdx.x;
    double acc[2 * D + 3];
#pragma unroll
    for (int k = 0; k < 2 * D + 3; ++k) acc[k] = 0.0;
    bool done = false;
    double final_score = 0.0;
    if (e < N) {
        const Philox ph = philox_setup(*a.key, nullptr, step);
        typename Env::action_t act;
        float logp;
        if (Env::kDiscrete) {
            act = (typename Env::action_t)sample_categorical_one(a.act_param + e * Env::kActions, Env::kActions, e, ph, &logp);
            if (a.act_tape && (int64_t)step < a.tape_steps) ((int64_t*)a.act_tape)[(int64_t)step * N + e] = (int64_t)act;
        } else {
            float x;
            sample_gaussian_one(a.act_param + e, a.logstd, 1, e, ph, &x);
            act = (typename Env::action_t)x;
            if (a.act_tape && (int64_t)step < a.tape_steps) ((float*)a.act_tape)[(int64_t)step * N + e] = x;
        }
        // env step: the arithmetic of rollout_step_kernel / env_step_kernel
        double st[Env::S];
#pragma unroll
        for (int k = 0; k < Env::S; ++k) st[k] = a.state[k * N + e];
        int32_t el = a.elapsed[e];
        double score = a.ep_score[e];
        bool terminated;
        double reward;
        float4 o[V];
        double sc_s = 0.0, sc_c = 0.0;
        if constexpr (Env::kTrigCache) {
            bool hit = false;
            if (a.trig_cache && a.trig_cache[e] == st[0]) {
                sc_s = a.trig_cache[N + e];
                hit = true;
            }
            if (!hit) sincos_cr(st[0], &sc_s, &sc_c);
            reward = Env::step_sc(st, act, terminated, sc_s);
            sincos_cr(st[0], &sc_s, &sc_c);
            o[0] = Env::observe_sc(st, sc_s, sc_c);
        } else {
            reward = Env::step(st, act, terminated);
            observe_row<Env>(st, o);
        }
        el += 1;
        const bool truncated = el >= a.max_steps;
        score = __dadd_rn(score, reward);
        done = terminated || truncated;
        final_score = score;
        if (done) {
            Pcg64 g = load_rng<Env>(a.rng, N, e);
            Env::draw(st, g);
            a.rng[e] = g.hi;
            a.rng[N + e] = g.lo;
            el = 0;
            score = 0.0;
            if constexpr (Env::kTrigCache) {
                sincos_cr(st[0], &sc_s, &sc_c);
                o[0] = Env::observe_sc(st, sc_s, sc_c);
            } else {
                observe_row<Env>(st, o);
            }
        }
        put_row<Env>(a.next_obs, e, o);
        if constexpr (Env::kTrigCache) {
            if (a.trig_cache) {
                a.trig_cache[e] = st[0];
                a.trig_cache[N + e] = sc_s;
                a.trig_cache[2 * N + e] = sc_c;
            }
        }
#pragma unroll
        for (int k = 0; k < Env::S; ++k) a.state[k * N + e] = st[k];
        a.elapsed[e] = el;
        a.ep_score[e] = score;
        if (a.stats.obs_state_in) {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const float in[4] = {o[v].x, o[v].y, o[v].z, o[v].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    acc[4 * v + k] = (double)in[k];
                    acc[D + 4 * v + k] = (double)in[k] * (double)in[k];
                }
            }
        }
    }
    // ---- ordered compaction of the finished episodes: ballots within the CTA, decoupled look-back across CTAs
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, done);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t local = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            const unsigned c = s_warp[w];
            s_warp[w] = (unsigned)local;
            local += c;
        }
        uint64_t* words = a.ws + 2;
        uint64_t excl = 0;
        if (cta == 0) {
            st_release_u64(words, kLbInclusive | local);
        } else {
            st_release_u64(words + cta, kLbAggregate | local);
            for (int64_t j = (int64_t)cta - 1;;) {
                const uint64_t f = ld_acquire_u64(words + j);
                if (f == 0) continue;                       // CTA j has started (its place was taken before ours) but not published
                excl += f & kLbValue;
                if (f & kLbInclusive) break;
                --j;
            }
            st_release_u64(words + cta, kLbInclusive | (excl + local));
        }
        s_base = s_c0 + (int64_t)excl;
    }
    __syncthreads();
    if (done) {
        const int64_t pos = s_base + s_warp[warp] + __popc(m & ((1u << lane) - 1u));
        if (pos < a.cap) a.scores[pos] = final_score;
    }
    // ---- statistics (partials in CTA order), then the last CTA publishes the step
    step_stats_finish_at<D>(a.stats, acc, N, stat_smem, &stat_flag, (int)cta);
    if (!stat_flag || threadIdx.x >= 32) return;
    const uint64_t last = ld_acquire_u64(a.ws + 2 + (gridDim.x - 1));
    const int64_t c1 = s_c0 + (int64_t)(last & kLbValue);
    // the reference merges the next observations only when its loop goes round again (len(scores) < test_episode)
    if (a.stats.obs_state_in && c1 < *a.test_episode) {
        __syncwarp();
        double* live = const_cast<double*>(a.stats.obs_state_in);
        if (lane < 2 * D + 1) live[lane] = a.stats.obs_state_out[lane];
    }
    for (int64_t i = lane; i < (int64_t)gridDim.x; i += 32) a.ws[2 + i] = 0ull;
    if (lane == 0) {
        *a.count = c1;
        *a.step = step + 1;
        a.ws[0] = 0ull;
    }
}

__global__ void sincos_kernel(const double* __restrict__ x, double* __restrict__ s, double* __restrict__ c, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sincos_cr(x[i], &s[i], &c[i]);
}

static inline int env_block(int64_t N) {
    // small batches are latency bound: spread them over more SMs with narrower CTAs
    if (N <= (int64_t)kNumSMs * 32 * 2) return 32;
    if (N <= (int64_t)kNumSMs * 64 * 4) return 64;
    return 128;
}

}  // namespace xb

using namespace xb;

#ifdef XB_STEP_TS
unsigned long long* g_xb_step_ts = nullptr;
extern "C" int xb_debug_set_step_ts(void* buf) { g_xb_step_ts = (unsigned long long*)buf; return 0; }
#endif

extern "C" int xb_env_reset(int env_kind, double* state, uint64_t* rng, int32_t* elapsed, double* ep_score,
                            float* obs, int n_draws, int64_t N, xb_stream_t stream) {
    if (N <= 0 || n_draws < 0 || !state || !rng || !elapsed || !ep_score || !obs) return XB_E_BADARG;
    cudaStream_t s = (cudaStream_t)stream;
    int block = env_block(N), grid = ceil_div_i64(N, block);
    if (env_kind == XB_ENV_CARTPOLE)
        env_reset_kernel<CartPole><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (float4*)obs, n_draws, N);
    else if (env_kind == XB_ENV_PENDULUM)
        env_reset_kernel<Pendulum><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (float4*)obs, n_draws, N);
    else if (env_kind == XB_ENV_MOUNTAINCAR)
        env_reset_kernel<MountainCar><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (float4*)obs, n_draws, N);
    else if (env_kind == XB_ENV_ACROBOT)
        env_reset_kernel<Acrobot><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (float4*)obs, n_draws, N);
    else if (env_kind == XB_ENV_MOUNTAINCAR_STACK4)
        env_reset_kernel<MountainCarStack><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (float4*)obs, n_draws, N);
    else
        return XB_E_UNSUPPORTED;
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_env_step(int env_kind, double* state, uint64_t* rng, int32_t* elapsed, double* ep_score,
                           const void* actions, float* obs, float* next_obs, float* rew, uint8_t* term,
                           uint8_t* trunc, float* reset_obs, int32_t* ep_step_out, double* ep_score_out,
                           double* ep_stats, int max_episode_steps, int64_t N, xb_stream_t stream) {
    if (N <= 0 || !state || !rng || !elapsed || !ep_score || !actions || !obs || !rew || !term || !trunc ||
        !reset_obs || !ep_step_out || !ep_score_out)
        return XB_E_BADARG;
    cudaStream_t s = (cudaStream_t)stream;
    int block = env_block(N), grid = ceil_div_i64(N, block);
    if (env_kind == XB_ENV_CARTPOLE)
        env_step_kernel<CartPole><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (const int64_t*)actions,
                                                         (float4*)obs, (float4*)next_obs, rew, term, trunc,
                                                         (float4*)reset_obs, ep_step_out, ep_score_out, ep_stats,
                                                         max_episode_steps, N);
    else if (env_kind == XB_ENV_PENDULUM)
        env_step_kernel<Pendulum><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (const float*)actions,
                                                         (float4*)obs, (float4*)next_obs, rew, term, trunc,
                                                         (float4*)reset_obs, ep_step_out, ep_score_out, ep_stats,
                                                         max_episode_steps, N);
    else if (env_kind == XB_ENV_MOUNTAINCAR)
        env_step_kernel<MountainCar><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (const int64_t*)actions,
                                                            (float4*)obs, (float4*)next_obs, rew, term, trunc,
                                                            (float4*)reset_obs, ep_step_out, ep_score_out, ep_stats,
                                                            max_episode_steps, N);
    else if (env_kind == XB_ENV_ACROBOT)
        env_step_kernel<Acrobot><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (const int64_t*)actions,
                                                        (float4*)obs, (float4*)next_obs, rew, term, trunc,
                                                        (float4*)reset_obs, ep_step_out, ep_score_out, ep_stats,
                                                        max_episode_steps, N);
    else if (env_kind == XB_ENV_MOUNTAINCAR_STACK4)
        env_step_kernel<MountainCarStack><<<grid, block, 0, s>>>(state, rng, elapsed, ep_score, (const int64_t*)actions,
                                                                 (float4*)obs, (float4*)next_obs, rew, term, trunc,
                                                                 (float4*)reset_obs, ep_step_out, ep_score_out, ep_stats,
                                                                 max_episode_steps, N);
    else
        return XB_E_UNSUPPORTED;
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_sincos_f64(const double* x, double* s, double* c, int64_t n, xb_stream_t stream) {
    if (n <= 0 || !x || !s || !c) return XB_E_BADARG;
    sincos_kernel<<<ceil_div_i64(n, 128), 128, 0, (cudaStream_t)stream>>>(x, s, c, n);
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_rollout_step(int env_kind, const float* act_param, const float* logstd, const float* val, uint64_t seed,
                               const uint64_t* counter_dev, uint64_t offset, double* state, uint64_t* rng,
                               int32_t* elapsed, double* ep_score, float* obs, float* next_obs, float* rew, uint8_t* term,
                               uint8_t* trunc, float* reset_obs, int32_t* ep_step_out, double* ep_score_out,
                               double* ep_stats, int max_episode_steps, const float* x_in, void* act_out, float* logp_out,
                               float* obs_row, float* act_row, float* rew_row, float* val_row, float* term_row,
                               uint8_t* trunc_row, float* logp_row, const float* rew_scale, float rew_clip,
                               const float* boot_src, float* boot_row, double* trig_cache, const double* obs_state_in,
                               double* obs_state_out, int obs_dim, float obs_clip, double* ret_state, float* rew_std_io,
                               double* returns, double gamma, int mask_terminal, double* stat_partials, uint32_t* stat_ticket,
                               double* stat_sums_out, int64_t N, xb_stream_t stream) {
    if (N <= 0 || !act_param || !val || !state || !rng || !elapsed || !ep_score || !obs || !rew || !term || !trunc ||
        !reset_obs || !ep_step_out || !ep_score_out || !x_in || !act_out || !logp_out || !obs_row || !act_row ||
        !rew_row || !val_row || !term_row || !logp_row)
        return XB_E_BADARG;
    if (env_kind == XB_ENV_PENDULUM && !logstd) return XB_E_BADARG;
    if ((boot_row != nullptr) != (boot_src != nullptr)) return XB_E_BADARG;
    RolloutStepArgs a{act_param, logstd, val, seed, counter_dev, offset, state, rng, elapsed, ep_score, (float4*)obs,
                      (float4*)next_obs, rew, term, trunc, (float4*)reset_obs, ep_step_out, ep_score_out, ep_stats,
                      max_episode_steps, (const float4*)x_in, act_out, logp_out, (float4*)obs_row, act_row, rew_row,
                      val_row, term_row, trunc_row, logp_row, rew_scale, rew_clip, boot_src, boot_row, trig_cache, N, StepStats{}};
    if (stat_partials) {
        if (!stat_ticket || (!obs_state_in && !returns)) return XB_E_BADARG;
        if (obs_state_in && (obs_dim < 1 || obs_dim > 8)) return XB_E_BADARG;
        if (!stat_sums_out) {     // merged here: needs the destinations
            if (obs_state_in && (!obs_state_out || obs_state_in == obs_state_out)) return XB_E_BADARG;
            if ((ret_state != nullptr) != (returns != nullptr) || (ret_state && !rew_std_io)) return XB_E_BADARG;
        }
        a.stats = StepStats{obs_state_in, obs_state_out, obs_dim, obs_clip, ret_state, rew_std_io, returns, gamma, mask_terminal,
                            stat_partials, stat_ticket, stat_sums_out};
    }
#ifdef XB_STEP_TS
    a.ts = g_xb_step_ts;
#endif
    cudaStream_t s = (cudaStream_t)stream;
    int block = env_block(N), grid = ceil_div_i64(N, block);
    if (env_kind == XB_ENV_CARTPOLE) XB_CUDA(launch_pdl(rollout_step_kernel<CartPole>, dim3(grid), dim3(block), 0, s, true, a));
    else if (env_kind == XB_ENV_PENDULUM) XB_CUDA(launch_pdl(rollout_step_kernel<Pendulum>, dim3(grid), dim3(block), 0, s, true, a));
    else if (env_kind == XB_ENV_MOUNTAINCAR) XB_CUDA(launch_pdl(rollout_step_kernel<MountainCar>, dim3(grid), dim3(block), 0, s, true, a));
    else if (env_kind == XB_ENV_ACROBOT) XB_CUDA(launch_pdl(rollout_step_kernel<Acrobot>, dim3(grid), dim3(block), 0, s, true, a));
    else if (env_kind == XB_ENV_MOUNTAINCAR_STACK4) XB_CUDA(launch_pdl(rollout_step_kernel<MountainCarStack>, dim3(grid), dim3(block), 0, s, true, a));
    else return XB_E_UNSUPPORTED;
    XB_LAUNCH_CHECK();
    return 0;
}

extern "C" int xb_eval_step(int env_kind, const float* act_param, const float* logstd, const uint64_t* key, uint64_t* step,
                            double* state, uint64_t* rng, int32_t* elapsed, double* ep_score, float* next_obs, double* trig_cache,
                            int max_episode_steps, void* act_tape, int64_t tape_steps, double* scores, int64_t* count,
                            const int64_t* test_episode, int64_t cap, double* obs_state, double* obs_state_cand, int obs_dim,
                            double* partials, uint64_t* workspace, int64_t N, xb_stream_t stream) {
    if (N <= 0 || !act_param || !key || !step || !state || !rng || !elapsed || !ep_score || !next_obs || !scores || !count ||
        !test_episode || cap < 1 || !partials || !workspace || tape_steps < 0 || (act_tape && tape_steps == 0))
        return XB_E_BADARG;
    if (env_kind == XB_ENV_PENDULUM && !logstd) return XB_E_BADARG;
    if (obs_state && (!obs_state_cand || obs_state == obs_state_cand || obs_dim < 1 || obs_dim > 8)) return XB_E_BADARG;
    StepStats st{};
    st.obs_state_in = obs_state;
    st.obs_state_out = obs_state_cand;
    st.dim = obs_dim;
    st.partials = partials;
    st.ticket = (unsigned int*)(workspace + 1);
    EvalStepArgs a{act_param, logstd, key, step, state, rng, elapsed, ep_score, (float4*)next_obs, trig_cache, max_episode_steps,
                   act_tape, tape_steps, scores, count, test_episode, cap, workspace, N, st};
    cudaStream_t s = (cudaStream_t)stream;
    int block = env_block(N), grid = ceil_div_i64(N, block);
    if (env_kind == XB_ENV_CARTPOLE) eval_step_kernel<CartPole><<<grid, block, 0, s>>>(a);
    else if (env_kind == XB_ENV_PENDULUM) eval_step_kernel<Pendulum><<<grid, block, 0, s>>>(a);
    else if (env_kind == XB_ENV_MOUNTAINCAR) eval_step_kernel<MountainCar><<<grid, block, 0, s>>>(a);
    else if (env_kind == XB_ENV_ACROBOT) eval_step_kernel<Acrobot><<<grid, block, 0, s>>>(a);
    else if (env_kind == XB_ENV_MOUNTAINCAR_STACK4) eval_step_kernel<MountainCarStack><<<grid, block, 0, s>>>(a);
    else return XB_E_UNSUPPORTED;
    XB_LAUNCH_CHECK();
    return 0;
}
