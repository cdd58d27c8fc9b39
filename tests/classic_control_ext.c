/*
 * tests/classic_control_ext.c — C restatement of gym 0.26.2's Continuous_MountainCarEnv (MountainCarContinuous-v0), the
 * independent second oracle beside the Python restatement in tests/classic_control_ext.py.  Same conventions as
 * oracle/classic_control.c (whose PCG64 stream and trig flavours are repeated here): AoS fp64 state [n][2], rng [n][4],
 * one rounding per operation (built with -ffp-contract=off), flavour 0 = "cr" (libquadmath cosq rounded once), 1 = "libm".
 *
 * gym/envs/classic_control/continuous_mountain_car.py, restated from the published algorithm with the pinned numpy 1.21.6's
 * promotion (a float32 scalar with a Python float or int -> float64, so every operation of step() is fp64):
 *   force = min(max(action[0], -1.0), 1.0); velocity += force * 0.0015 - 0.0025 * math.cos(3 * position); clip to +-0.07;
 *   position += velocity; clip to [-1.2, 0.6]; if position == -1.2 and velocity < 0: velocity = 0;
 *   terminated = position >= 0.45 and velocity >= 0 (fp64); reward = (100.0 if terminated else 0) - math.pow(action[0], 2) * 0.1
 *   (the unclipped action); state = float32([position, velocity]).  reset: [U(-0.6, -0.4), 0] in fp64, obs = float32(state).
 * The state array holds fp64 values: the unrounded draw after a reset, (double)(float)x after a step.
 */
#include <math.h>
#include <quadmath.h>
#include <stdint.h>

typedef unsigned __int128 u128;

static inline double cos_f(double x, int flavour) { return flavour == 0 ? (double)cosq((__float128)x) : cos(x); }
static inline double sq_f(double v, int flavour) { return flavour == 0 ? v * v : pow(v, 2.0); }

/* numpy PCG64 (XSL-RR 128/64) and Generator.uniform, as oracle/classic_control.c */
static inline uint64_t pcg64_next(uint64_t* rng) {
    const u128 mult = ((u128)0x2360ED051FC65DA4ULL << 64) | 0x4385DF649FCCF645ULL;
    u128 st = ((u128)rng[0] << 64) | rng[1];
    u128 inc = ((u128)rng[2] << 64) | rng[3];
    st = st * mult + inc;
    rng[0] = (uint64_t)(st >> 64);
    rng[1] = (uint64_t)st;
    uint64_t x = rng[0] ^ rng[1];
    unsigned rot = (unsigned)(rng[0] >> 58);
    return (x >> rot) | (x << ((-rot) & 63));
}
static inline double pcg64_uniform(uint64_t* rng, double low, double range) {
    return low + range * ((double)(pcg64_next(rng) >> 11) * (1.0 / 9007199254740992.0));
}

static void draw(double* st, uint64_t* rng) {
    st[0] = pcg64_uniform(rng, -0.6, -0.4 - (-0.6));
    st[1] = 0.0;
}

void oc_mountaincar_continuous_reset(double* state /*[n][2]*/, uint64_t* rng, int32_t* elapsed, double* ep_score,
                                     float* obs /*[n][2]*/, int n_draws, long n) {
    for (long e = 0; e < n; ++e) {
        for (int d = 0; d < n_draws; ++d) draw(state + 2 * e, rng + 4 * e);
        elapsed[e] = 0; ep_score[e] = 0.0;
        obs[2 * e] = (float)state[2 * e]; obs[2 * e + 1] = (float)state[2 * e + 1];
    }
}

void oc_mountaincar_continuous_step(double* state, uint64_t* rng, int32_t* elapsed, double* ep_score,
                                    const float* actions, float* obs, float* rew, uint8_t* term, uint8_t* trunc,
                                    float* reset_obs, int32_t* ep_step_out, double* ep_score_out,
                                    int max_steps, long n, int flavour) {
    const double power = 0.0015, max_speed = 0.07, min_pos = -1.2, max_pos = 0.6, goal_pos = 0.45;
    for (long e = 0; e < n; ++e) {
        double* st = state + 2 * e;
        double position = st[0], velocity = st[1];
        const double a = (double)actions[e];
        const double force = fmin(fmax(a, -1.0), 1.0);
        velocity = velocity + (force * power - 0.0025 * cos_f(3.0 * position, flavour));
        velocity = velocity < -max_speed ? -max_speed : (velocity > max_speed ? max_speed : velocity);
        position = position + velocity;
        position = position < min_pos ? min_pos : (position > max_pos ? max_pos : position);
        if (position == min_pos && velocity < 0.0) velocity = 0.0;
        int terminated = position >= goal_pos && velocity >= 0.0;
        double reward = (terminated ? 100.0 : 0.0) - sq_f(a, flavour) * 0.1;
        st[0] = (double)(float)position; st[1] = (double)(float)velocity;
        elapsed[e] += 1;
        int truncated = elapsed[e] >= max_steps;
        ep_score[e] += reward;
        obs[2 * e] = (float)st[0]; obs[2 * e + 1] = (float)st[1];
        rew[e] = (float)reward; term[e] = (uint8_t)terminated; trunc[e] = (uint8_t)truncated;
        ep_step_out[e] = elapsed[e]; ep_score_out[e] = ep_score[e];
        if (terminated || truncated) {
            draw(st, rng + 4 * e);
            elapsed[e] = 0; ep_score[e] = 0.0;
            reset_obs[2 * e] = (float)st[0]; reset_obs[2 * e + 1] = (float)st[1];
        }
    }
}
