/*
 * swarm_b200.h -- C ABI of the B200-native swarm-environment hot path (libswarm_b200.so).
 *
 * The reference (allentran/golds-rl-gym) is pure Python and has NO FFI of its own; its
 * boundary for this path is three Python contracts (SURVEY.md section 8b).  Each entry point
 * below names the reference interface it stands in for.  A reference maintainer binds these
 * with ctypes (see INTEGRATION.md); the package `golds-rl-gym_b200/` is exactly that binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name starts with `host_`;
 *   - the library allocates nothing, never synchronises (except the *_host call) and launches
 *     on the caller's stream; all entry points are thread-safe for distinct buffers AND distinct
 *     streams (the two-kernel step keeps one internal side stream + fork/join event pair per
 *     (device, caller stream); two host threads must not step on the SAME stream concurrently);
 *   - return value: 0 = ok, negative = SwarmStatus error (swarm_strerror);
 *   - layouts are C order.  x:(E,N,2) f64, xa:(E,A,2) f64, actions:(E,A,2),
 *     grid:(E,G,G,2) f32 indexed [env][x_bin][y_bin][channel], positions:(E,A,2) u8.
 *     A grid must be 8-byte aligned (SWARM_ERR_FLAGS otherwise); 16-byte alignment is faster.
 *
 * Arithmetic: the O(N) integrator state is FP64 like the reference's numpy arrays
 * (fed_gym/envs/multiagent.py:30-86); the O(N^2) pair forces (multiagent.py:88-115) are FP32.
 */
#ifndef SWARM_B200_H
#define SWARM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWARM_ABI_VERSION 3

/* opaque: a cudaStream_t passed as a pointer-sized handle (0 = legacy default stream) */
typedef void* swarm_stream_t;

typedef enum SwarmStatus {
    SWARM_OK = 0,
    SWARM_ERR_NULL = -1,        /* a required pointer is NULL                          */
    SWARM_ERR_SIZE = -2,        /* unsupported E/N/A/G (see swarm_validate)            */
    SWARM_ERR_LAUNCH = -3,      /* CUDA launch / runtime error (swarm_last_cuda_error) */
    SWARM_ERR_FLAGS = -4        /* inconsistent flags / missing optional buffer        */
} SwarmStatus;

/* fed_gym/envs/multiagent.py:8-21 (class constants) + fed_gym/__init__.py:21-33 (TimeLimit 128)
 * + fed_gym/agents/state_processors.py:17-23 (box).  POD, passed by pointer, copied at call. */
typedef struct SwarmParams {
    int32_t n_envs;             /* E : envs in THIS shard                                   */
    int32_t n_locusts;          /* N : SwarmEnv.N_LOCUSTS (80)                              */
    int32_t n_agents;           /* A : SwarmEnv.N_AGENTS (10)                               */
    int32_t grid_size;          /* G : SwarmStateProcessor.grid_size (84 for PAAC)          */
    int32_t n_burn_in;          /* SwarmEnv.N_BURN_IN (10)                                  */
    int32_t max_episode_steps;  /* gym TimeLimit (128); 0 = raw SwarmEnv, no limit          */
    int32_t math_mode;          /* 0 = fast (MUFU rsqrt/ex2/rcp), 1 = precise (IEEE)        */
    int32_t tuning;             /* 0 = automatic launch shape.  Otherwise (results are bitwise the same for every
                                 * value): bits 4-5 = rasteriser placement (1 follower kernel, 2 raster warps in the
                                 * step kernel, 3 the step's own threads after the step);
                                 * bits 8-12 = the CLUSTER layout: 0 one CTA per env (N <= 2048), 1..16 one env per
                                 * thread-block cluster of K CTAs, 31 the library picks K.  It takes 512 < N <= 8192
                                 * (SWARM_ERR_FLAGS for N <= 512, K > 16, K above the env's force warps, or with
                                 * placement bits; SWARM_ERR_SIZE when the layout does not fit the device) and
                                 * applies to swarm_step / _reset / _forces / _rasterize;
                                 * all other bits must be 0                                                   */
    double noise;               /* NOISE 1e-4   */
    double gravity;             /* GRAVITY -1   */
    double wind;                /* WIND_SPEED 1 */
    double F;                   /* 0.5          */
    double L;                   /* 10           */
    double dt;                  /* 0.05         */
    double box_width;           /* WIDTH 3  -> x range [mean-1.5, mean+1.5]                 */
    double box_height;          /* HEIGHT 3 -> y range [0, 2*HEIGHT]                        */
    uint64_t seed;              /* Philox key                                               */
    int64_t env_id_offset;      /* global id of local env 0 (shard-invariant RNG streams)   */
} SwarmParams;

/* The env batch's persistent state (SwarmEnv.states / .agent_noise[t] / .particle_noise[t] /
 * TimeLimit._elapsed_steps).  noise_* hold the FROZEN row N_BURN_IN that every post-reset step
 * re-uses because SwarmEnv._step never advances self.t (multiagent.py:38,40; SURVEY Q1).  They are
 * written at every reset; a step with SWARM_STEP_FRESH_NOISE does not read them. */
typedef struct SwarmState {
    double* x;                  /* (E,N,2) */
    double* xa;                 /* (E,A,2) */
    double* noise_x;            /* (E,N,2) unscaled N(0,1) */
    double* noise_a;            /* (E,A,2) unscaled N(0,1) */
    int32_t* elapsed;           /* (E) steps since reset   */
    uint32_t* episode;          /* (E) resets so far (Philox counter word) */
    uint32_t* work;             /* nullable (work_words uint32): scratch words, ZERO when handed over and zero again
                                 * after every call.  With at least 2 + E of them swarm_step may produce the
                                 * observation with a second kernel that follows the step on an internal
                                 * higher-priority stream (per-env ready flags in work[2..2+E)); with fewer (>= 2) it
                                 * only uses the work queue work[0..1]; with none, static env assignment and raster
                                 * warps inside the step kernel.  Not shared between concurrently running calls. */
    uint64_t work_words;        /* number of uint32 words behind `work` (0 if work == NULL); checked, never trusted */
} SwarmState;

/* The reference's random draws of one reset (multiagent.py:51-56), injected for parity tests.
 * Only rows 0..n_burn_in of the 138-row noise tables are ever read by the reference. */
typedef struct SwarmInjectedDraws {
    const double* x0;             /* (E,N,2)              np.random.rand            */
    const double* xa0;            /* (E,A,2)                                        */
    const double* burn_actions;   /* (E,n_burn_in,A,2)    N(0,1), unclipped         */
    const double* agent_noise;    /* (E,n_burn_in+1,A,2)                            */
    const double* particle_noise; /* (E,n_burn_in+1,N,2)                            */
} SwarmInjectedDraws;

#define SWARM_STEP_AUTO_RESET   1u  /* SwarmRunner._run: on done, reset and observe the new episode */
#define SWARM_STEP_CLIP_ACTIONS 2u  /* SwarmRunner.transform_actions_for_env, in place on actions   */
#define SWARM_STEP_ACTIONS_F64  4u  /* actions_f64 is used instead of actions_f32                   */
#define SWARM_STEP_NO_ACTION_WIND 8u  /* SwarmEnv._step(add_wind=False), multiagent.py:30,35-36: the step's
                                       * actions are used as they are (burn-in steps of an auto-reset still
                                       * add the wind, like the reference's _reset -> step)                */
#define SWARM_STEP_INKERNEL_RASTER 16u /* never use the follower kernel (see swarm_step); same results     */
#define SWARM_STEP_FRESH_NOISE  32u /* the reference with SURVEY Q1 fixed (self.t advances): env e's step uses
                                     * Philox row n_burn_in + elapsed[e] of noise streams 3 and 4 of its current
                                     * episode (episode word st->episode[e] - 1), drawn inside the step kernel,
                                     * instead of the frozen row st->noise_*.  The first step after a Philox
                                     * reset is the same in both modes.  io->noise_a / io->noise_x still
                                     * override their own row when given.  Without the flag nothing changes. */

typedef struct SwarmStepIO {
    float* actions_f32;         /* (E,A,2) PAAC shared_actions dtype (paac.py:269); in/out if CLIP  */
    double* actions_f64;        /* (E,A,2) gym-facade dtype; used when SWARM_STEP_ACTIONS_F64        */
    const double* noise_a;      /* nullable (E,A,2): per-step override of the frozen (or fresh) row */
    const double* noise_x;      /* nullable (E,N,2)                                                 */
    float* reward;              /* (E)  = -mean_j |v_j|^2                                           */
    uint8_t* done;              /* (E)  reward >= 0 || ++elapsed >= max_episode_steps               */
    float* grid;                /* nullable (E,G,G,2): fused rasterise of the post-step state       */
    uint8_t* positions;         /* nullable (E,A,2); required iff grid != NULL                      */
    float* v_out;               /* nullable (E,N,2): pre-cutoff locust velocities (diagnostics)     */
    uint32_t flags;
    uint32_t reserved;
} SwarmStepIO;

/* What an auto-resetting step overwrites, kept for the caller (swarm_step_final).  Every pointer is nullable.
 * terminated / truncated are written for every env on every step (done == terminated | truncated; both may be 1);
 * x / xa / grid / positions only for envs with done[e] -- the rows of the other envs keep their bytes.  The
 * terminal state is the post-step state BEFORE the auto-reset (without SWARM_STEP_AUTO_RESET: the returned state). */
typedef struct SwarmStepFinal {
    double* x;                  /* (E,N,2) nullable: terminal locust positions of envs with done[e]               */
    double* xa;                 /* (E,A,2) nullable                                                                */
    uint8_t* terminated;        /* (E) nullable: reward >= 0                                                       */
    uint8_t* truncated;         /* (E) nullable: max_episode_steps > 0 && elapsed >= max_episode_steps              */
    float* grid;                /* (E,G,G,2) nullable: process_state of the terminal state (done envs); needs x, xa */
    uint8_t* positions;         /* (E,A,2) required iff grid                                                       */
} SwarmStepFinal;

/* Per-env physics (swarm_reset_physics / swarm_step_physics / swarm_forces_physics): env e takes noise, gravity, wind, F,
 * L and dt from row e of a device table instead of SwarmParams, with the same roundings (F, 1/L, wind and gravity to
 * FP32 for the pair forces; noise, wind and dt FP64), so a row equal to SwarmParams gives their bits exactly.
 * With SWARM_PHYSICS_RESAMPLE every reset of env e (explicit or auto-reset) first draws a new row:
 *   column c = lo[c] + (hi[c] - lo[c]) u   (each operation rounded once; lo == hi gives lo exactly)
 * u = the .x (even c) or .y (odd c) of the uniform pair c / 2 of Philox stream 5 of the reset (seed, global env id,
 * episode counter before the reset's increment) -- always Philox, also with injected draws.  The row is written to
 * table[e] and governs the reset's burn-in and every step of the new episode.  Without the flag the table is only read
 * (once per step / reset / forces call), so the caller may edit rows between calls.
 * Before any CUDA call: phys or table NULL -> SWARM_ERR_NULL; table not 16-byte aligned, unknown flag bits or
 * reserved != 0 -> SWARM_ERR_FLAGS; with RESAMPLE a non-finite bound, lo > hi, a non-finite hi - lo or lo[4] (L) <= 0
 * -> SWARM_ERR_SIZE.  The table's values are device data and are not checked. */
#define SWARM_PHYSICS_RESAMPLE 1u
typedef struct SwarmPhysics {
    double* table;              /* (E,6) f64 device, 16-byte aligned: env e's {noise, gravity, wind, F, L, dt}         */
    uint32_t flags;             /* SWARM_PHYSICS_RESAMPLE                                                               */
    uint32_t reserved;          /* must be 0                                                                            */
    double lo[6], hi[6];        /* per-column uniform range of SWARM_PHYSICS_RESAMPLE                                   */
} SwarmPhysics;

int swarm_abi_version(void);
const char* swarm_strerror(int status);
const char* swarm_last_cuda_error(void);

/* Size / resource check for a parameter set; SWARM_OK, SWARM_ERR_SIZE or SWARM_ERR_FLAGS.  No GPU work (whether a
 * cluster can be scheduled is checked by the calls themselves, before they launch anything). */
int swarm_validate(const SwarmParams* p);

/* SwarmEnv._reset (multiagent.py:46-63): draws + n_burn_in burn-in steps; elapsed=0; episode+=1.
 * mask: nullable (E) u8, only envs with mask!=0 are reset.  draws: nullable -> Philox4x32-10
 * keyed by (seed, env_id_offset+e, episode) as documented in csrc/swarm_philox.cuh. */
int swarm_reset(const SwarmParams* p, const SwarmState* st, const uint8_t* mask,
                const SwarmInjectedDraws* draws, swarm_stream_t stream);

/* SwarmEnv._step (multiagent.py:30-44) + TimeLimit + (optionally) the SwarmRunner._run
 * auto-reset (emulator_runner.py:126-135) and SwarmStateProcessor.process_state
 * (state_processors.py:29-42) of the resulting state: one kernel, or -- for large swarms when
 * st->work is given -- the step kernel plus a rasteriser kernel that follows it concurrently on
 * an internal stream (joined back into `stream` before the call returns its work to it).
 * The call can be captured into a CUDA graph; instantiate such a graph with
 * cudaGraphInstantiateFlagUseNodePriority (PyTorch does), or the follower loses its priority
 * and runs after the step instead of next to it.
 * The follower spins on per-env flags the step kernel raises, so the two kernels must be able to
 * run side by side or step-first.  Eager launches guarantee it (the step is launched first); a tool
 * that re-orders or isolates graph nodes (graph-node profiling, some debuggers) does not: pass
 * SWARM_STEP_INKERNEL_RASTER or set the environment variable SWARM_B200_NO_FOLLOWER=1 there.  The
 * spin is bounded (a follower that sees no progress for ~20 s traps: the call then fails with a
 * CUDA launch error at the next synchronisation instead of hanging).
 * reset_draws: nullable; injected draws used by auto-reset instead of Philox. */
int swarm_step(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io,
               const SwarmInjectedDraws* reset_draws, swarm_stream_t stream);

/* swarm_step that also keeps the terminal step of every env whose episode ends (gymnasium's terminated / truncated
 * and final observation): the step kernel splits done into fin->terminated / fin->truncated and copies a done env's
 * post-step state to fin->x / fin->xa before the auto-reset overwrites it.  With fin->grid the standalone rasteriser
 * then runs once more, after the step, over the done envs only (fin->x / fin->xa as its source, io->done as its mask;
 * the other envs' CTAs read one byte and leave): bit for bit swarm_rasterize of the terminal state.  One or two
 * more launches than swarm_step, on `stream`; capturable like it.  fin == NULL is exactly swarm_step.
 * SWARM_ERR_FLAGS, before any launch: fin->grid without fin->positions, fin->x or fin->xa; fin->positions without
 * fin->grid; fin->grid not 8-byte aligned. */
int swarm_step_final(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                     const SwarmInjectedDraws* reset_draws, swarm_stream_t stream);

/* swarm_reset / swarm_step_final / swarm_forces with per-env physics (SwarmPhysics above).  fin is nullable like
 * swarm_step_final's.  Separate kernel instantiations: the kernels of swarm_reset / swarm_step / swarm_step_final /
 * swarm_forces are unchanged. */
int swarm_reset_physics(const SwarmParams* p, const SwarmState* st, const SwarmPhysics* phys, const uint8_t* mask,
                        const SwarmInjectedDraws* draws, swarm_stream_t stream);
int swarm_step_physics(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                       const SwarmPhysics* phys, const SwarmInjectedDraws* reset_draws, swarm_stream_t stream);
int swarm_forces_physics(const SwarmParams* p, const SwarmPhysics* phys, const double* x, const double* xa, float* v,
                         float* reward, swarm_stream_t stream);
/* swarm_step_plan for swarm_step_physics (its kernels hold the physics rows in shared memory). */
int swarm_step_plan_physics(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmPhysics* phys,
                            int32_t out[8]);

/* Action repeat (frame skip): one call makes up to `repeat` env steps per env with the call's actions, each exactly the
 * step swarm_step makes (actions converted and, with SWARM_STEP_CLIP_ACTIONS, clipped and written back once; elapsed
 * advances per substep; fresh noise draws row n_burn_in + elapsed for each substep; io->noise_a / io->noise_x overrides
 * serve every substep).  An env stops at its first done substep; then the auto-reset (if requested) runs once.
 * reward[e] is the FP32 sum, in substep order, of the stepped substeps' rewards; done, fin->terminated / truncated /
 * x / xa and v_out are the last stepped substep's; grid / positions are the observation of the state the call returns.
 * Bit for bit: one swarm_step* call with the call's flags, then up to repeat - 1 calls without SWARM_STEP_CLIP_ACTIONS
 * and SWARM_STEP_AUTO_RESET, each env stopping at its first done, a masked swarm_reset* of the done envs (with
 * auto-reset), and the observation of the final state.
 * fin and phys are nullable: with both NULL this is swarm_step, with one of them swarm_step_final / swarm_step_physics.
 * repeat == 1 launches exactly the kernels of those calls.  The argument checks are theirs; repeat < 1 is
 * SWARM_ERR_SIZE, before any CUDA call.  swarm_step_host has no repeat. */
int swarm_step_repeat(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                      const SwarmPhysics* phys, int32_t repeat, const SwarmInjectedDraws* reset_draws, swarm_stream_t stream);
/* swarm_step_plan for swarm_step_repeat (phys nullable). */
int swarm_step_plan_repeat(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmPhysics* phys,
                           int32_t repeat, int32_t out[8]);

/* The launch shape swarm_step would use for these arguments (no launch; needs the device for occupancy queries):
 * out = { force mode, filler warp (0/1), rasteriser placement (0 none, 1 follower kernel, 2 raster warps, 3 the step's
 * own threads, 4 the env's thread-block cluster), threads per CTA, CTAs (E K in the cluster layout), dynamic shared
 * memory bytes, follower CTAs (the cluster layout: K), kernel launches }. */
int swarm_step_plan(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, int32_t out[8]);

/* Same call with HOST buffers for the per-step inputs/results; synchronises the stream before
 * returning.  With PINNED host buffers (cudaHostAlloc / torch pin_memory: device-visible under
 * UVA) the kernel reads host_actions and writes host_reward / host_done directly over PCIe --
 * no staging copies (io->actions_f32 / io->reward / io->done are then left untouched).  With
 * pageable memory it copies host_actions to io->actions_f32, runs swarm_step and copies
 * io->reward / io->done back.
 * host_grid / host_positions: nullable (both or neither; need io->grid): the compact observation
 * (E,G,G,2) f32 + (E,A,2) u8 is also copied back to the host (copy engine, after the step) -- the
 * numpy-out case of the reference's process_state.
 * One env step per call, with the class-wide physics: no per-env physics and no action repeat (swarm_step_physics,
 * swarm_step_repeat). */
int swarm_step_host(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io,
                    const float* host_actions, float* host_reward, uint8_t* host_done,
                    float* host_grid, uint8_t* host_positions, swarm_stream_t stream);

/* Debug only, and only in a library built with -DSWARM_TRACE (the production build compiles the hooks out: they cost
 * 0.5-2.5 %): from now on every step / rasteriser kernel of this process records phase timestamps of each CTA's first
 * env into device_words (n_words uint64, zeroed by the caller; 32 words per record: for phase ph < 16 the global
 * timer in ns at [2 ph] and the SM cycle counter at [2 ph + 1]; record = CTA index of the step kernel, E + env for
 * the follower kernel; phases: see scripts/trace_step.py).  NULL switches it off.  Not thread-safe. */
void swarm_debug_trace(uint64_t* device_words, int64_t n_words);

/* Destroys the CUDA graphs swarm_step_host caches for the CALLING host thread (one per argument
 * set, at most 32).  They are also destroyed when the thread exits. */
void swarm_step_host_clear(void);

/* SwarmStateProcessor.process_state (state_processors.py:25-42): grid + uint8 agent cells.
 * box: nullable (E,4) f64 = [lo_x, hi_x, lo_y, hi_y], i.e. _get_bounding_box (:25-27) of
 * vstack([x, xa]).  n_agents may be 0 here (then xa/positions may be NULL): the box/grid of a
 * bare point set, as tests/env_tests.py:39 uses _get_bounding_box(state[0]).
 * The observation is numpy's bit for bit either way; with a box the window's centre is always taken by numpy's
 * sequential FP64 sum (the box reports it), without one -- and inside swarm_step -- by a parallel sum that is verified
 * against a rigorous error bound and replaced by the sequential one only when a point sits within that bound of a bin edge. */
int swarm_rasterize(const SwarmParams* p, const double* x, const double* xa,
                    float* grid, uint8_t* positions, double* box, swarm_stream_t stream);

/* SwarmRunner.get_local_states (emulator_runner.py:98-111) for the whole batch:
 * expanded (E,A,G,G,3) f32 = grid channels + one-hot at positions[e][a]. */
int swarm_expand_obs(const SwarmParams* p, const float* grid, const uint8_t* positions,
                     float* expanded, swarm_stream_t stream);

/* SwarmEnv.v_calculate (multiagent.py:88-115): v (E,N,2) f32 and reward (E) f32 from x, xa. */
int swarm_forces(const SwarmParams* p, const double* x, const double* xa,
                 float* v, float* reward, swarm_stream_t stream);

/* SwarmEnv.x_update (multiagent.py:70-75) on n particles, in place on x AND v like the
 * reference (v gets the ground cutoff); noise is the already-scaled additive term. */
int swarm_x_update(double* x, double* v, const double* noise, int64_t n, double dt, swarm_stream_t stream);

/* SwarmEnv.xv_cutoff (multiagent.py:77-86) on n particles, in place. */
int swarm_xv_cutoff(double* x, double* v, int64_t n, swarm_stream_t stream);

/* SwarmEnv.s (multiagent.py:65-68): out[i] = F exp(-r[i]/L) - exp(-r[i]), FP64. */
int swarm_s_potential(const double* r, double* out, int64_t n, double F, double L, swarm_stream_t stream);

/* SwarmRunner.transform_actions_for_env (emulator_runner.py:113-118), in place, n rows of 2. */
int swarm_clip_actions(float* actions, int64_t n_rows, float max_norm, swarm_stream_t stream);

/* Materialise the Philox draws that swarm_reset would use for each env's CURRENT episode
 * counter (st->episode), in the SwarmInjectedDraws layout, so a test can inject the very
 * same numbers into the reference.  Output pointers are the (non-const) draws buffers. */
int swarm_philox_draws(const SwarmParams* p, const SwarmState* st, double* x0, double* xa0,
                       double* burn_actions, double* agent_noise, double* particle_noise,
                       swarm_stream_t stream);

/* Materialise rows row0 .. row0+n_rows-1 of the noise streams 3 and 4 of every env's CURRENT
 * episode (episode word st->episode[e] - 1, i.e. the episode the last reset started): the rows a
 * SWARM_STEP_FRESH_NOISE step draws (row n_burn_in + elapsed) and the reset's own rows 0..n_burn_in,
 * bit for bit.  agent_noise (E,n_rows,A,2), particle_noise (E,n_rows,N,2), unscaled N(0,1).
 * SWARM_ERR_NULL / SWARM_ERR_SIZE (row0 < 0, n_rows <= 0) are returned before any CUDA call. */
int swarm_philox_noise_rows(const SwarmParams* p, const SwarmState* st, int32_t row0, int32_t n_rows,
                            double* agent_noise, double* particle_noise, swarm_stream_t stream);

/* Raw Philox4x32-10 blocks for known-answer tests: out[i] = philox(ctr[i], key[i]). */
int swarm_philox_raw(const uint32_t* ctr /*(n,4)*/, const uint32_t* key /*(n,2)*/,
                     uint32_t* out /*(n,4)*/, int64_t n, swarm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SWARM_B200_H */
