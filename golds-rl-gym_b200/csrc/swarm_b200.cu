// libswarm_b200.so -- kernels + the extern "C" ABI declared in include/swarm_b200.h.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -shared
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <stdlib.h>

#include <cmath>
#include <map>
#include <mutex>
#include <tuple>
#include <utility>

#include "swarm_kernels.cuh"
#include "swarm_cluster.cuh"

using namespace swarm;

namespace {

// ------------------------------------------------------------------------------------------ kernels

// Issue the cp.async copies of everything env e's step reads from HBM into stage buffer sg (PHYS: and its physics row
// into sg.ph).
template <bool PHYS>
__device__ __forceinline__ void prefetch_env(const Stage& sg, const KP& kp, const SwarmState& st, const SwarmStepIO& io,
                                             const int e, const Grp& g, const SwarmPhysics& phys) {
    const int N = kp.N, A = kp.A;
    const double2* gx = reinterpret_cast<const double2*>(st.x) + (size_t)e * N;
    for (int i = g.tid; i < N; i += g.n) cp_async<16>(sg.xs + i, gx + i);
    const double2* ga = reinterpret_cast<const double2*>(st.xa) + (size_t)e * A;
    const double2* gna = reinterpret_cast<const double2*>(io.noise_a ? io.noise_a : st.noise_a) + (size_t)e * A;
    const bool fetch_an = !kp.fresh || io.noise_a;     // fresh noise: the step draws the agent row itself
    for (int k = g.tid; k < A; k += g.n) {
        cp_async<16>(sg.as + k, ga + k);
        if (fetch_an) cp_async<16>(sg.an + k, gna + k);
        if (io.flags & SWARM_STEP_ACTIONS_F64)
            cp_async<16>(sg.araw + 16 * k, reinterpret_cast<const double2*>(io.actions_f64) + (size_t)e * A + k);
        else
            cp_async<8>(sg.araw + 16 * k, reinterpret_cast<const float2*>(io.actions_f32) + (size_t)e * A + k);
    }
    if (g.tid == g.n - 1) {
        cp_async<4>(sg.misc, st.elapsed + e);
        if (kp.fresh) cp_async<4>(sg.misc + 1, st.episode + e);
    }
    if constexpr (PHYS) {
        if (g.tid < 3) cp_async<16>(sg.ph + 2 * g.tid, phys.table + (size_t)e * kPhysCols + 2 * g.tid);
    }
}

// PHYS kernels: the physics rows of the n_stage stage buffers, behind the smem_bytes(...) of the kernel's carve
__device__ __forceinline__ double* phys_rows(unsigned char* smem_raw, size_t smem) {
    return reinterpret_cast<double*>(smem_raw + smem);
}

// SwarmEnv._step + TimeLimit + SwarmRunner auto-reset + process_state for the whole batch.
// Persistent CTAs (env e = blockIdx.x, += gridDim.x), two warp-specialised groups per CTA:
//   threads [0, n_force)          FORCE group : prefetch the next env (cp.async), step, done /
//                                               auto-reset, write the state back, hand the
//                                               post-step positions over in sm.rx[it & 1]
//   threads [n_force, blockDim.x) RASTER group: zero-fill the env's grid (before the positions even
//                                               exist), wait for them, histogram + scatter
// so that the rasteriser of env e (latency chains + 56 KB of stores) and the HBM reads of env
// e + gridDim.x both run under a force phase.  Hand-over: named barriers FULL[b] (force arrives,
// raster waits) and EMPTY[b] (raster arrives, force waits before re-using rx[b] two envs later).
// PLACE (compile time, so that every instantiation only carries the code it runs -- the kernel is instruction-cache
// sensitive): 0 no rasteriser in this kernel (none wanted, or k_raster_follow trails it), 2 a raster GROUP rides along,
// 3 the force group rasterises its own env after the step (SELF; optionally with a filler warp for the TMA zero fill).
// FIN (swarm_step_final; fin's pointers nullable): the done split of every env and the terminal state of the done ones,
// copied out of the stage buffer in the (rare) done branch before the auto-reset overwrites it.  Compile time, so that
// swarm_step's kernels (FIN = false) stay exactly what they were: the same code behind a runtime branch re-schedules
// the whole kernel and was measured to cost 2.8 % of the C4 step with the feature off (0.1703 -> 0.1751 ms).
// PHYS (swarm_step_physics): per-env physics.  Env e's row is prefetched with the env into its stage buffer's row, and
// an auto-reset with SWARM_PHYSICS_RESAMPLE draws the new episode's row into it (and the table) before the burn-in.
// Compile time for the same reason as FIN.
// REP (swarm_step_repeat, with either FIN): action repeat.  The step proper runs up to `repeat` substeps with
// the same actions through the one env_step call site, summing the FP32 rewards in order and stopping at the first done
// substep; the done / auto-reset / write-back / rasterise tail then runs once.  `repeat` is a kernel parameter rather
// than a KP field: a longer KP would move every later parameter of every kernel and change the default kernels' code.
template <int MODE, bool PRECISE, int PLACE, bool FIN, bool PHYS, bool REP>
__global__ void __maxnreg__(64) k_step(const KP kp, const SwarmState st, const SwarmStepIO io,
                                       const SwarmInjectedDraws dr, const int has_draws, const int n_force,
                                       const SwarmStepFinal fin, const SwarmPhysics phys, const int repeat) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = kp.N, A = kp.A;
    const int n_all = blockDim.x, n_raster = n_all - n_force;
    constexpr bool raster = PLACE == 2;            // a raster GROUP rides along
    constexpr bool self_raster = PLACE == 3;       // the force group rasterises its own env after the step
    const bool filler = self_raster && kp.filler;  // ... while one extra warp issues / awaits the TMA zero fill
    Smem sm = carve(smem_raw, N, A, kp.G, kp.n_stage, true, ModeT<MODE>::SYM, raster ? 1 : (self_raster ? 2 : 0));
    double* prow = nullptr;
    if constexpr (PHYS)
        prow = phys_rows(smem_raw, smem_bytes(N, A, kp.G, kp.n_stage, true, raster ? 1 : (self_raster ? 2 : 0), ModeT<MODE>::SYM));
    // stage buffer b with its physics row
    auto stage = [&](const int b) {
        Stage s = stage_at(smem_raw, N, A, b);
        if constexpr (PHYS) s.ph = prow + kPhysCols * b;
        return s;
    };

    // Env assignment: the first two envs of a CTA are static (blockIdx.x, + gridDim.x); with a work queue the
    // later ones are drawn from an atomic counter (index 2 * gridDim.x + ticket), which evens out the CTAs'
    // finishing times; without, the static stride continues.
    uint32_t* const work = st.work;
    const bool dyn = raster && kp.dynamic != 0;

    if ((int)threadIdx.x < n_force) {
        const Grp g = {(int)threadIdx.x, n_force};
        constexpr int T = ModeT<MODE>::T;
        int e = blockIdx.x, e1 = blockIdx.x + gridDim.x;   // the env of this iteration and of the next one
        const int cells = kp.G * kp.G;
        if constexpr (self_raster) {       // shared-memory prologue: independent of the previous kernel's results
            raster_table_clear(sm, (int)(smem_table_bytes(N, A, kp.G) / 4), g);
            raster_lut_fill(sm, kp, g.tid, g.n);
            if (filler) bar_arrive<BAR_FULL>(n_all);       // the table is clean: the filler warp may read its zeros
        }
        pdl_wait();                        // from here on the previous kernels' writes (state, actions, grid) are visible
        if (e < kp.E) prefetch_env<PHYS>(stage(0), kp, st, io, e, g, phys);
        cp_async_commit();
        int it = 0;
        if (g.tid == 0) trace_mark(kp, blockIdx.x, TR_ENTRY);
        for (; e < kp.E; ++it) {
            int grabbed = 0;                       // the env after next: asked for now, needed an iteration later
            if (dyn && g.tid == 0) grabbed = 2 * (int)gridDim.x + (int)atomicAdd(work, 1u);
            sm.st = stage(it & 1);
            cp_async_wait_all();
            g.sync();      // this env's stage buffer has landed; the other one and sm.nx are free again
            if (it == 0 && g.tid == 0) trace_mark(kp, blockIdx.x, TR_LOADED);
            if (it == 0) pdl_launch_dependents();       // the next kernel's CTAs may take free SM slots from now on
            if constexpr (self_raster) {
                // Without a filler warp (odd grid sizes, or no room for its 32 threads) the group streams the env's zeros
                // out itself with plain stores -- AFTER the env's inputs have landed: a burst of 56 KB per env from every
                // CTA at once would otherwise sit in front of those loads.  (Issuing TMA bulk stores from a force thread was
                // measured and dropped: the issue blocks for microseconds when every CTA does it at once.)
                if (!filler) raster_zero_fill(io.grid + (size_t)e * cells * 2, cells, g.tid, g.n);
            }
            if (dyn && it > 0) e1 = sm.mail[1];
            // Fresh noise: the step uses row n_burn + elapsed of noise streams 3 / 4 of the env's current episode (the last
            // reset was keyed with the counter's value before its increment), drawn below instead of read from HBM
            DrawCtx nd;
            nd.key = kp.key;
            nd.env = kp.env_off + (uint32_t)e;
            nd.episode = (uint32_t)sm.st.misc[1] - 1u;
            const uint32_t nrow = (uint32_t)kp.n_burn + (uint32_t)sm.st.misc[0];
            {   // this env's locust noise row: each thread fetches (or draws) the rows of its own targets, so that its
                // own wait (before the integration) is all the synchronisation it needs
                if (kp.fresh && !io.noise_x) {
#pragma unroll
                    for (int t = 0; t < T; ++t) {
                        const int j = target_index<MODE>(g, t, kp);
                        if (j < N) sm.nx[j] = draw_normal2(nd, STREAM_NOISE_X, nrow, (uint32_t)j);
                    }
                } else {
                    const double2* gnx = reinterpret_cast<const double2*>(io.noise_x ? io.noise_x : st.noise_x) + (size_t)e * N;
#pragma unroll
                    for (int t = 0; t < T; ++t) {
                        const int j = target_index<MODE>(g, t, kp);
                        if (j < N) cp_async<16>(sm.nx + j, gnx + j);
                    }
                }
                cp_async_commit();      // (an empty group with fresh noise: env_step's wait counts groups)
            }
            if (e1 < kp.E) prefetch_env<PHYS>(stage((it + 1) & 1), kp, st, io, e1, g, phys);
            cp_async_commit();     // (possibly empty) group of the next env: env_step waits for all but this one

            // actions: HBM dtype -> FP64, optional clip (the owner thread of agent k also moves it)
            for (int k = g.tid; k < A; k += g.n) {
                double2 a;
                if (io.flags & SWARM_STEP_ACTIONS_F64) {
                    a = *reinterpret_cast<const double2*>(sm.st.araw + 16 * k);
                } else {
                    const float2 f = *reinterpret_cast<const float2*>(sm.st.araw + 16 * k);
                    a = make_double2((double)f.x, (double)f.y);
                }
                if (io.flags & SWARM_STEP_CLIP_ACTIONS) {
                    // emulator_runner.py:113-118: rows with |a| >= MAX_MOVE_NORM(1) are divided by |a|, in place
                    if (io.flags & SWARM_STEP_ACTIONS_F64) {
                        const double d = sqrt(__dadd_rn(__dmul_rn(a.x, a.x), __dmul_rn(a.y, a.y)));
                        if (d >= 1.0) {
                            a.x = a.x / d; a.y = a.y / d;
                            reinterpret_cast<double2*>(io.actions_f64)[(size_t)e * A + k] = a;
                        }
                    } else {
                        const float fx = (float)a.x, fy = (float)a.y;
                        const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy)));
                        if (d >= 1.0f) {
                            const float2 c = make_float2(__fdiv_rn(fx, d), __fdiv_rn(fy, d));
                            reinterpret_cast<float2*>(io.actions_f32)[(size_t)e * A + k] = c;
                            a = make_double2((double)c.x, (double)c.y);
                        }
                    }
                }
                sm.act[k] = a;
                // fresh noise: the agent's row, by the thread that moves the agent in env_step
                if (kp.fresh && !io.noise_a) sm.st.an[k] = draw_normal2(nd, STREAM_NOISE_A, nrow, (uint32_t)k);
            }

            // One env_step call site serves the step proper and, if the episode ends here, the burn-in
            // steps of the auto-reset (emulator_runner.py:127-132: the terminal reward/done are reported,
            // the state -- and therefore the observation -- is the freshly reset episode's).
            int elapsed = 0;
            ResetCtx rc;
            uint32_t ep = 0;
            int r = -1;                              // -1: the step proper; >= 0: burn-in row being stepped
            float* v_out = io.v_out ? io.v_out + (size_t)e * N * 2 : nullptr;
            int sub = 0;                             // REP: substep of the step proper
            float rsum = 0.0f;                       // REP: FP32 sum of the substeps' rewards
            for (;;) {
                // multiagent.py:30,35-36: _step(add_wind=False) leaves the action alone; the burn-in steps of a reset
                // always go through step() with the default add_wind=True (multiagent.py:59-61)
                const double reward = env_step<MODE, PRECISE, self_raster, PHYS>(sm, kp, g, v_out,
                                                                                  (r < 0 && !kp.wind_step) ? 0.0 : (PHYS ? sm.st.ph[2] : kp.wind),
                                                                                  (r < 0 && it == 0) ? (long long)blockIdx.x : -1);
                if (r < 0) {
                    // multiagent.py:44 done = reward >= 0; gym TimeLimit: done |= ++elapsed >= max_episode_steps
                    elapsed = sm.st.misc[0] + 1;
                    if constexpr (REP) elapsed += sub;
                    const bool done = (reward >= 0.0) || (kp.max_steps > 0 && elapsed >= kp.max_steps);
                    if constexpr (REP) {
                        // in substep order from the first substep's reward (not 0.0f): repeat 1 and -0.0 keep their bits
                        rsum = sub == 0 ? (float)reward : __fadd_rn(rsum, (float)reward);
                        if (!done && ++sub < repeat) {
                            // Fresh noise: substep sub uses row nrow + sub, drawn with the prologue's owner mappings (targets
                            // of this thread into sm.nx, agents k = tid mod n into sm.st.an).  env_step reads each of these
                            // elements only with the thread that writes it here, and the previous substep's reads of them
                            // were by this same thread: no barrier.  Frozen rows and overrides stay where they are.
                            if (kp.fresh) {
                                const uint32_t row = nrow + (uint32_t)sub;
                                if (!io.noise_x) {
#pragma unroll
                                    for (int t = 0; t < T; ++t) {
                                        const int j = target_index<MODE>(g, t, kp);
                                        if (j < N) sm.nx[j] = draw_normal2(nd, STREAM_NOISE_X, row, (uint32_t)j);
                                    }
                                }
                                if (!io.noise_a)
                                    for (int k = g.tid; k < A; k += g.n) sm.st.an[k] = draw_normal2(nd, STREAM_NOISE_A, row, (uint32_t)k);
                            }
                            continue;
                        }
                    }
                    if (g.tid == 0) {
                        io.reward[e] = REP ? rsum : (float)reward;
                        io.done[e] = done ? 1 : 0;
                        if constexpr (FIN) {
                            if (fin.terminated) fin.terminated[e] = reward >= 0.0 ? 1 : 0;
                            if (fin.truncated) fin.truncated[e] = (kp.max_steps > 0 && elapsed >= kp.max_steps) ? 1 : 0;
                        }
                    }
                    if constexpr (FIN) {
                        // the terminal state, final since env_step's closing barrier; reset_begin's leading barrier
                        // orders these reads before its writes
                        if (done && fin.x) {
                            double2* fx = reinterpret_cast<double2*>(fin.x) + (size_t)e * N;
                            for (int i = g.tid; i < N; i += g.n) fx[i] = sm.st.xs[i];
                        }
                        if (done && fin.xa) {
                            double2* fa = reinterpret_cast<double2*>(fin.xa) + (size_t)e * A;
                            for (int k = g.tid; k < A; k += g.n) fa[k] = sm.st.as[k];
                        }
                    }
                    if (!(done && (io.flags & SWARM_STEP_AUTO_RESET))) break;      // group-uniform
                    ep = st.episode[e];
                    // the new episode's physics: written after env_step's closing barrier (nobody reads the row any more),
                    // visible after reset_begin's leading one -- before the first burn-in step moves anything
                    if constexpr (PHYS) {
                        if (phys.flags & SWARM_PHYSICS_RESAMPLE) phys_reset_row(sm.st.ph, phys, kp, e, ep, g.tid, true);
                    }
                    rc = reset_begin(sm, kp, g, e, ep, has_draws != 0, dr);
                    v_out = nullptr;
                    elapsed = 0;
                }
                if (reset_row(sm, kp, g, rc, ++r, dr, st)) {
                    if (g.tid == 0) st.episode[e] = ep + 1;
                    break;
                }
            }
            if (g.tid == 0) {
                st.elapsed[e] = elapsed;
                if (dyn) sm.mail[1] = grabbed;          // read by everybody after the next iteration's barrier
                if (it == 0) trace_mark(kp, blockIdx.x, TR_STEPPED);
            }

            if (raster && it >= 1) bar_sync<BAR_EMPTY>(n_all);   // the raster group has read the previous env's points
            double2* ox = reinterpret_cast<double2*>(st.x) + (size_t)e * N;
            double2* oa = reinterpret_cast<double2*>(st.xa) + (size_t)e * A;
            double2* rx = sm.rx;
            const Stage stg = sm.st;
            // the write-back of the new state: by everybody here, or -- when this group rasterises its own env -- as
            // the first thing inside env_raster
            auto write_back = [&](const int tid, const int n) {
                for (int i = tid; i < N; i += n) {
                    const double2 q = stg.xs[i];
                    ox[i] = q;
                    if (raster) rx[i] = q;
                }
                for (int k = tid; k < A; k += n) {
                    const double2 q = stg.as[k];
                    oa[k] = q;
                    if (raster) rx[N + k] = q;
                }
            };
            if constexpr (!self_raster) write_back(g.tid, g.n);
            // bar.arrive / bar.sync order the shared-memory writes above for the threads that complete
            // the barrier (PTX ISA, producer/consumer example of barrier.arrive): no extra fence
            if constexpr (raster) {
                if (g.tid == 0) sm.mail[0] = e;
                bar_arrive<BAR_FULL>(n_all);
            }
            if (PLACE == 0 && kp.publish) {   // tell the concurrently running k_raster_follow that env e's new state is in memory
                g.sync();
                if (g.tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(work + 2 + e), "r"(1u) : "memory");
            }
            if (it == 0 && g.tid == 0) trace_mark(kp, blockIdx.x, TR_STORED);
            if constexpr (self_raster) {
                // state_processors.py:29-42 of the new state, straight from the stage buffer: [xs | as] are contiguous
                // = vstack([x, xa]), final and visible since env_step's closing barrier
                env_raster<false>(sm, stg.xs, kp, g, io.grid + (size_t)e * cells * 2, io.positions + (size_t)e * A * 2, filler,
                                 ZeroSelf{filler, n_all}, NoRelease(), write_back, it == 0 ? (long long)blockIdx.x : -1);
                if (filler && e1 < kp.E) bar_arrive<BAR_FULL>(n_all);   // clean again: the next env's zero fill may start
            }
            e = e1;
            if (!dyn) e1 = e + gridDim.x;
        }
        if constexpr (raster) {      // tell the raster group that nothing more is coming
            if (it >= 1) bar_sync<BAR_EMPTY>(n_all);
            if (g.tid == 0) sm.mail[0] = -1;
            bar_arrive<BAR_FULL>(n_all);
        }
        if (dyn && g.tid == 0) {   // the last CTA to leave puts the queue back to zero for the next call
            __threadfence();
            if (atomicAdd(work + 1, 1u) == gridDim.x - 1) {
                work[0] = 0u;
                work[1] = 0u;
            }
        }
    } else if constexpr (self_raster) {
        // The filler warp of the SELF shape: streams out the zeros of the CTA's envs (TMA bulk stores fed from the clean
        // counter table) while the force group computes, and tells it when the table may be written (BAR_ZREAD) and
        // when the zeros have landed (BAR_ZDONE).
        const int lane = (int)threadIdx.x - n_force;
        const int cells = kp.G * kp.G;
        const uint32_t table_bytes = (uint32_t)smem_table_bytes(N, A, kp.G);
        pdl_wait();                                        // the grid may still be read / written by the previous kernels
        pdl_launch_dependents();
        for (int e = blockIdx.x; e < kp.E; e += gridDim.x) {
            bar_sync<BAR_FULL>(n_all);                     // the force group has (re)cleaned the table
            if (lane == 0) {
                tma_zero_fill_issue(io.grid + (size_t)e * cells * 2, sm.table, cells, table_bytes);
                if (e == (int)blockIdx.x) trace_mark(kp, blockIdx.x, TR_ZFILL);
                tma_zero_fill_wait_read();
            }
            __syncwarp();
            bar_arrive<BAR_ZREAD>(n_all);
            if (lane == 0) tma_zero_fill_wait_done();
            __syncwarp();
            bar_arrive<BAR_ZDONE>(n_all);
        }
    } else if constexpr (raster) {
        const RGrp g = {(int)threadIdx.x - n_force, n_raster};
        const int cells = kp.G * kp.G;
        const bool tma = tma_zero_fill_ok(io.grid, cells);
        const uint32_t table_bytes = (uint32_t)smem_table_bytes(N, A, kp.G);
        raster_table_clear(sm, (int)(table_bytes / 4), g);
        raster_lut_fill(sm, kp, g.tid, g.n);
        g.sync();
        pdl_wait();                                        // the grid may still be read / written by the previous kernels
        pdl_launch_dependents();
        auto zero_fill = [&](int e) {
            // The observation is ~99 % zeros: stream them out first (TMA bulk stores fed from the clean counter
            // table, else plain stores); the non-zero cells are scattered over them afterwards.
            float* grid_e = io.grid + (size_t)e * cells * 2;
            if (tma) {
                if (g.tid == 0) tma_zero_fill_issue(grid_e, sm.table, cells, table_bytes);
            } else {
                raster_zero_fill(grid_e, cells, g.tid, g.n);
            }
        };
        for (int it = 0;; ++it) {
            // statically assigned envs are known in advance: their zeros go out while the force group still
            // computes; envs drawn from the work queue are only known at the hand-over
            const int predicted = (!dyn || it < 2) ? (int)(blockIdx.x + it * gridDim.x) : -1;
            const bool early = predicted >= 0 && predicted < kp.E;
            if (early) zero_fill(predicted);
            bar_sync<BAR_FULL>(n_all);
            const int e = sm.mail[0];
            if (e < 0) break;
            if (!early) zero_fill(e);
            auto release = [n_all]() { bar_arrive<BAR_EMPTY>(n_all); };   // the force group always waits for it
            env_raster<false>(sm, sm.rx, kp, g, io.grid + (size_t)e * cells * 2, io.positions + (size_t)e * A * 2, tma,
                              ZeroOwn{tma, 0}, release, NoOverlap(), it == 0 ? (long long)blockIdx.x : -1);
        }
    }
}

// SwarmEnv._reset for the masked envs (one CTA per env).  PHYS: the env's row (drawn, with SWARM_PHYSICS_RESAMPLE)
// governs the burn-in.
template <int MODE, bool PRECISE, bool PHYS>
__global__ void __maxnreg__(64) k_reset(const KP kp, const SwarmState st, const uint8_t* __restrict__ mask,
                                        const SwarmInjectedDraws dr, const int has_draws, const SwarmPhysics phys) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int e = blockIdx.x;
    if (mask && !mask[e]) return;
    Smem sm = carve(smem_raw, kp.N, kp.A, kp.G, 1, true, ModeT<MODE>::SYM, 0);
    const Grp g = {(int)threadIdx.x, (int)blockDim.x};
    const uint32_t ep = st.episode[e];
    if constexpr (PHYS) {     // visible after reset_begin's leading barrier
        sm.st.ph = phys_rows(smem_raw, smem_bytes(kp.N, kp.A, kp.G, 1, true, 0, ModeT<MODE>::SYM));
        phys_reset_row(sm.st.ph, phys, kp, e, ep, g.tid, true);
    }
    const ResetCtx rc = reset_begin(sm, kp, g, e, ep, has_draws != 0, dr);
    for (int r = 0; !reset_row(sm, kp, g, rc, r, dr, st); ++r)
        env_step<MODE, PRECISE, false, PHYS>(sm, kp, g, nullptr, PHYS ? sm.st.ph[2] : kp.wind);
    double2* ox = reinterpret_cast<double2*>(st.x) + (size_t)e * kp.N;
    double2* oa = reinterpret_cast<double2*>(st.xa) + (size_t)e * kp.A;
    for (int i = g.tid; i < kp.N; i += g.n) ox[i] = sm.st.xs[i];
    for (int k = g.tid; k < kp.A; k += g.n) oa[k] = sm.st.as[k];
    if (g.tid == 0) {
        st.elapsed[e] = 0;
        st.episode[e] = ep + 1;
    }
}

// SwarmStateProcessor.process_state of the state k_step is producing RIGHT NOW: a persistent kernel on a second,
// higher-priority stream that runs concurrently with a rasteriser-less k_step.  It streams out an env's zeros,
// waits for k_step to publish the env (ready[e], release/acquire), reads the fresh positions from L2, rasterises
// and clears the flag again.  k_step then runs in its fastest shape (one hardware-scheduled CTA per env) and the
// rasteriser's latency chains cost it no shared memory, registers or barriers.
constexpr unsigned long long kFollowTimeoutNs = 20ull * 1000 * 1000 * 1000;

__global__ void __launch_bounds__(128) k_raster_follow(const KP kp, const double* __restrict__ x,
                                                       const double* __restrict__ xa, float* __restrict__ grid,
                                                       uint8_t* __restrict__ positions, uint32_t* ready) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = kp.N, A = kp.A, cells = kp.G * kp.G;
    const Smem sm = carve(smem_raw, N, A, kp.G, 0, false, 0, 1);
    const RGrp g = {(int)threadIdx.x, (int)blockDim.x};
    const bool tma = tma_zero_fill_ok(grid, cells);
    const uint32_t table_bytes = (uint32_t)smem_table_bytes(N, A, kp.G);
    raster_table_clear(sm, (int)(table_bytes / 4), g);
    raster_lut_fill(sm, kp, g.tid, g.n);
    g.sync();
    double2* pts = sm.rx;
    for (int e = blockIdx.x; e < kp.E; e += gridDim.x) {
        float* grid_e = grid + (size_t)e * cells * 2;
        if (tma) {
            if (g.tid == 0) tma_zero_fill_issue(grid_e, sm.table, cells, table_bytes);
        } else {
            raster_zero_fill(grid_e, cells, g.tid, g.n);
        }
        if (g.tid == 0) {
            // Bounded spin: the step kernel normally publishes within microseconds.  If it never does (it faulted, or a
            // tool serialised the two kernels follower-first) this kernel traps after kFollowTimeoutNs instead of hanging
            // the device: the caller sees a CUDA error (SWARM_ERR_LAUNCH) at its next synchronisation.
            uint32_t v;
            unsigned long long t0 = 0;
            for (unsigned spins = 0;; ++spins) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ready + e) : "memory");
                if (v) break;
                __nanosleep(200);
                if ((spins & 1023u) == 1023u) {
                    unsigned long long now;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                    if (t0 == 0) t0 = now;
                    else if (now - t0 > kFollowTimeoutNs) __trap();
                }
            }
        }
        g.sync();
        const double2* gx = reinterpret_cast<const double2*>(x) + (size_t)e * N;     // fresh data: L2, not L1
        const double2* ga = reinterpret_cast<const double2*>(xa) + (size_t)e * A;
        for (int i = g.tid; i < N; i += g.n) pts[i] = __ldcg(gx + i);
        for (int k = g.tid; k < A; k += g.n) pts[N + k] = __ldcg(ga + k);
        g.sync();
        env_raster<false>(sm, pts, kp, g, grid_e, positions + (size_t)e * A * 2, tma, ZeroOwn{tma, 0}, NoRelease(), NoOverlap(),
                          (long long)kp.E + e);
        if (g.tid == 0) ready[e] = 0u;          // consumed: the next step's k_step raises it again
    }
}

// SwarmStateProcessor.process_state for the batch (standalone: one CTA per env).  EXACT: the caller wants the bounding
// box (_get_bounding_box), so numpy's sequential mean is always walked; otherwise the same verified parallel mean as the step.
// mask: nullable (E) u8, only envs with mask != 0 are rasterised (the terminal observations of swarm_step_final).
template <bool EXACT>
__global__ void __launch_bounds__(256) k_rasterize(const KP kp, const double* __restrict__ x,
                                                   const double* __restrict__ xa, float* __restrict__ grid,
                                                   uint8_t* __restrict__ positions, double* __restrict__ box,
                                                   const uint8_t* __restrict__ mask) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int e = blockIdx.x;
    if (mask && !mask[e]) return;
    const int cells = kp.G * kp.G;
    const Smem sm = carve(smem_raw, kp.N, kp.A, kp.G, 0, false, 0, 1);
    const RGrp g = {(int)threadIdx.x, (int)blockDim.x};
    float* grid_e = grid + (size_t)e * cells * 2;
    const double2* gx = reinterpret_cast<const double2*>(x) + (size_t)e * kp.N;
    const double2* ga = reinterpret_cast<const double2*>(xa) + (size_t)e * kp.A;
    double2* pts = sm.rx;
    for (int i = g.tid; i < kp.N; i += g.n) pts[i] = gx[i];
    for (int k = g.tid; k < kp.A; k += g.n) pts[kp.N + k] = ga[k];
    raster_zero_fill(grid_e, cells, g.tid, g.n);
    raster_table_clear(sm, (int)(smem_table_bytes(kp.N, kp.A, kp.G) / 4), g);
    raster_lut_fill(sm, kp, g.tid, g.n);
    g.sync();
    env_raster<EXACT>(sm, pts, kp, g, grid_e, positions + (size_t)e * kp.A * 2, false, ZeroOwn{false, 0}, NoRelease(), NoOverlap());
    if (EXACT && box && g.tid == 0) {
        const double m = sm.box[0];
        box[4 * e + 0] = m - kp.half_w;
        box[4 * e + 1] = m + kp.half_w;
        box[4 * e + 2] = 0.0;
        box[4 * e + 3] = kp.y_hi;
    }
}

// SwarmEnv.v_calculate for the batch (no integration; one CTA per env).  PHYS: F, L, wind and gravity of the env's row.
template <int MODE, bool PRECISE, bool PHYS>
__global__ void __maxnreg__(64) k_forces(const KP kp, const double* __restrict__ x,
                                         const double* __restrict__ xa, float* __restrict__ v,
                                         float* __restrict__ reward, const SwarmPhysics phys) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int e = blockIdx.x;
    constexpr int T = ModeT<MODE>::T;
    const Smem sm = carve(smem_raw, kp.N, kp.A, kp.G, 1, true, ModeT<MODE>::SYM, 0);
    const Grp g = {(int)threadIdx.x, (int)blockDim.x};
    const double2* gx = reinterpret_cast<const double2*>(x) + (size_t)e * kp.N;
    const double2* ga = reinterpret_cast<const double2*>(xa) + (size_t)e * kp.A;
    for (int i = g.tid; i < kp.N; i += g.n) sm.st.xs[i] = gx[i];
    float4* ag = agent_sources<MODE>(sm, kp);
    for (int k = g.tid; k < kp.A; k += g.n) ag[k] = split_hilo(ga[k], kp.cscale);
    stage_locusts<MODE>(sm, kp, g);
    g.sync();
    float vx[T], vy[T];
    if constexpr (PHYS) pair_forces<MODE, PRECISE>(sm, phys_kp(kp, phys.table + (size_t)e * kPhysCols), g, vx, vy);
    else pair_forces<MODE, PRECISE>(sm, kp, g, vx, vy);
    energy_put<MODE>(sm, kp, g, vx, vy);
    if (v) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const int j = target_index<MODE>(g, t, kp);
            if (j < kp.N) reinterpret_cast<float2*>(v)[(size_t)e * kp.N + j] = make_float2(vx[t], vy[t]);
        }
    }
    g.sync();
    const double r = energy_get<MODE>(sm, kp, g);
    if (reward && g.tid == 0) reward[e] = (float)r;
}

// SwarmRunner.get_local_states for the batch: (E,A,G,G,3) from (E,G,G,2) + (E,A,2).
__global__ void __launch_bounds__(256) k_expand(const int E, const int A, const int G,
                                                const float2* __restrict__ grid, const uint8_t* __restrict__ pos,
                                                float* __restrict__ out) {
    const int cells = G * G;
    const int ea = blockIdx.y;             // e*A + a
    const int e = ea / A;
    const int hot = (int)pos[2 * ea] * G + (int)pos[2 * ea + 1];
    const float2* g = grid + (size_t)e * cells;
    float* o = out + (size_t)ea * cells * 3;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += gridDim.x * blockDim.x) {
        const float2 q = __ldg(g + c);
        __stcs(o + 3 * c + 0, q.x);
        __stcs(o + 3 * c + 1, q.y);
        __stcs(o + 3 * c + 2, c == hot ? 1.0f : 0.0f);
    }
}

__global__ void k_clip(float2* __restrict__ a, const int64_t n, const float max_norm) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 q = a[i];
    const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(q.x, q.x), __fmul_rn(q.y, q.y)));
    if (d >= max_norm) a[i] = make_float2(__fdiv_rn(q.x, d), __fdiv_rn(q.y, d));
}

// SwarmEnv.x_update / xv_cutoff / s as standalone element-wise helpers (static methods of the facade)
__global__ void k_x_update(double2* __restrict__ x, double2* __restrict__ v, const double2* __restrict__ noise,
                           const int64_t n, const double dt, const int move) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double2 p = x[i], w = v[i];
    if (p.y <= 0.0) {                      // multiagent.py:77-86, v is mutated like the reference
        p.y = 0.0; w.x = 0.0;
        if (w.y <= 0.0) w.y = 0.0;
    }
    v[i] = w;
    if (move) move_particle(p, w, noise[i], dt, 1.0);
    x[i] = p;
}

__global__ void k_s_potential(const double* __restrict__ r, double* __restrict__ out, const int64_t n,
                              const double F, const double L) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __dadd_rn(__dmul_rn(F, exp(-r[i] / L)), -exp(-r[i]));
}

__global__ void k_philox_draws(const KP kp, const SwarmState st, double2* __restrict__ x0, double2* __restrict__ xa0,
                               double2* __restrict__ burn, double2* __restrict__ an, double2* __restrict__ pn) {
    const int e = blockIdx.x;
    const int N = kp.N, A = kp.A, rows = kp.n_burn + 1;
    DrawCtx ctx;
    ctx.key = kp.key;
    ctx.env = kp.env_off + (uint32_t)e;
    ctx.episode = st.episode[e];
    for (int i = threadIdx.x; i < N; i += blockDim.x) x0[(size_t)e * N + i] = draw_uniform2(ctx, STREAM_X0, i);
    for (int k = threadIdx.x; k < A; k += blockDim.x) xa0[(size_t)e * A + k] = draw_uniform2(ctx, STREAM_XA0, k);
    for (int r = 0; r < rows; ++r) {
        for (int k = threadIdx.x; k < A; k += blockDim.x) {
            if (r < kp.n_burn) burn[((size_t)e * kp.n_burn + r) * A + k] = draw_normal2(ctx, STREAM_BURN, r, k);
            an[((size_t)e * rows + r) * A + k] = draw_normal2(ctx, STREAM_NOISE_A, r, k);
        }
        for (int i = threadIdx.x; i < N; i += blockDim.x)
            pn[((size_t)e * rows + r) * N + i] = draw_normal2(ctx, STREAM_NOISE_X, r, i);
    }
}

// rows row0.. of noise streams 3 / 4 of every env's current episode (what a SWARM_STEP_FRESH_NOISE step draws);
// blockIdx.y strides over the rows
__global__ void k_philox_noise_rows(const KP kp, const SwarmState st, const int row0, const int n_rows,
                                    double2* __restrict__ an, double2* __restrict__ pn) {
    const int e = blockIdx.x;
    const int N = kp.N, A = kp.A;
    DrawCtx ctx;
    ctx.key = kp.key;
    ctx.env = kp.env_off + (uint32_t)e;
    ctx.episode = st.episode[e] - 1u;
    for (int r = blockIdx.y; r < n_rows; r += gridDim.y) {
        const uint32_t row = (uint32_t)row0 + (uint32_t)r;
        for (int k = threadIdx.x; k < A; k += blockDim.x)
            an[((size_t)e * n_rows + r) * A + k] = draw_normal2(ctx, STREAM_NOISE_A, row, k);
        for (int i = threadIdx.x; i < N; i += blockDim.x)
            pn[((size_t)e * n_rows + r) * N + i] = draw_normal2(ctx, STREAM_NOISE_X, row, i);
    }
}

__global__ void k_philox_raw(const uint4* __restrict__ ctr, const uint2* __restrict__ key, uint4* __restrict__ out,
                             const int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = philox4x32_10(ctr[i], key[i]);
}

// ---- CLUSTER layout (swarm_cluster.cuh, DESIGN 3.4): env blockIdx.x / K on the K CTAs of one thread-block cluster.
// nf = the one-CTA kernel's force threads (the virtual mapping); launched with cudaLaunchKernelEx and a cluster
// dimension.

// Noise row r of the env's locust j: r < 0 the step proper's row (override, frozen or fresh), else reset row r.
struct ClNoise {
    const KP& kp;
    const SwarmState& st;
    const SwarmStepIO* io;
    const SwarmInjectedDraws& dr;
    DrawCtx fresh_d, reset_d;
    uint32_t fresh_row;
    int e;
    bool inj;
    __device__ __forceinline__ double2 operator()(const int r, const int j) const {
        if (r < 0) {
            if (kp.fresh && !io->noise_x) return draw_normal2(fresh_d, STREAM_NOISE_X, fresh_row, (uint32_t)j);
            return reinterpret_cast<const double2*>(io->noise_x ? io->noise_x : st.noise_x)[(size_t)e * kp.N + j];
        }
        return inj ? reinterpret_cast<const double2*>(dr.particle_noise)[((size_t)e * (kp.n_burn + 1) + r) * kp.N + j]
                   : draw_normal2(reset_d, STREAM_NOISE_X, (uint32_t)r, (uint32_t)j);
    }
};

// reset_begin of the cluster: every CTA draws its own targets' initial positions (into global memory) and all agents'
__device__ __forceinline__ void cl_reset_begin(const CSmem& sm, const KP& kp, const CMap& m, const int e, double2* xe,
                                               const ClNoise& nz) {
    const int N = kp.N, A = kp.A, tid = (int)threadIdx.x;
    if (m.active) {
        for (int j = m.vtid; j < N; j += m.nf)
            xe[j] = nz.inj ? reinterpret_cast<const double2*>(nz.dr.x0)[(size_t)e * N + j] : draw_uniform2(nz.reset_d, STREAM_X0, j);
    }
    if (tid < A)
        sm.as[tid] = nz.inj ? reinterpret_cast<const double2*>(nz.dr.xa0)[(size_t)e * A + tid] : draw_uniform2(nz.reset_d, STREAM_XA0, tid);
}

// reset_row of the cluster: agent noise row r and burn-in action r (every CTA); for r == n_burn the frozen rows are
// stored (own targets; rank 0 the agents') and true is returned
__device__ __forceinline__ bool cl_reset_row(const CSmem& sm, const KP& kp, const CMap& m, const int e, const int r,
                                             const SwarmState& st, const ClNoise& nz) {
    const int N = kp.N, A = kp.A, tid = (int)threadIdx.x, rows = kp.n_burn + 1;
    const bool last = r >= kp.n_burn;
    if (tid < A) {
        const double2 z = nz.inj ? reinterpret_cast<const double2*>(nz.dr.agent_noise)[((size_t)e * rows + r) * A + tid]
                                 : draw_normal2(nz.reset_d, STREAM_NOISE_A, r, tid);
        sm.an[tid] = z;
        if (last) {
            if (m.rank == 0) reinterpret_cast<double2*>(st.noise_a)[(size_t)e * A + tid] = z;
        } else {
            sm.act[tid] = nz.inj ? reinterpret_cast<const double2*>(nz.dr.burn_actions)[((size_t)e * kp.n_burn + r) * A + tid]
                                 : draw_normal2(nz.reset_d, STREAM_BURN, r, tid);
        }
    }
    if (last && m.active)
        for (int j = m.vtid; j < N; j += m.nf) reinterpret_cast<double2*>(st.noise_x)[(size_t)e * N + j] = nz(r, j);
    return last;
}

// One SwarmEnv._step of the cluster's env up to the new positions in pn (nothing written yet); v_out: this env's.
template <int MODE, bool PRECISE>
__device__ __forceinline__ void cl_step_forces(const CSmem& sm, const KP& kp, const CMap& m, const double2* xe,
                                               const double2* xae, const double wind_a, const int r, const ClNoise& nz,
                                               float* v_out, double2 (&pn)[ModeT<MODE>::T]) {
    constexpr int T = ModeT<MODE>::T;
    cl_stage<true>(sm, kp, xe, xae, wind_a);
    if (m.active) {
        float vx[T], vy[T];
        cl_forces<MODE, PRECISE>(sm, kp, m, vx, vy);
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const int j = m.vtid + t * m.nf;
            double2 p = make_double2(0.0, 0.0);
            if (j < kp.N) {
                if (v_out) reinterpret_cast<float2*>(v_out)[j] = make_float2(vx[t], vy[t]);
                p = __ldcg(xe + j);
                move_particle(p, make_double2((double)vx[t], (double)vy[t]), nz(r, j), kp.dt, kp.sigma);
            }
            pn[t] = p;
        }
    }
}

template <int T>
__device__ __forceinline__ void cl_store(const KP& kp, const CMap& m, double2* xe, const double2 (&pn)[T]) {
    if (m.active) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const int j = m.vtid + t * m.nf;
            if (j < kp.N) xe[j] = pn[t];
        }
    }
}

// SwarmEnv._step + TimeLimit + auto-reset + process_state (k_step's contract) for the cluster layout.
// FIN: k_step's; each CTA copies its own targets' terminal positions from pn[], rank 0 the agents' from sm.as.
// PHYS: k_step's; every CTA reads (or draws) the env's row into its own shared memory, rank 0 writes a drawn row back.
// REP: k_step's; the reward is cluster-uniform, and so is the early stop.
template <int MODE, bool PRECISE, bool FIN, bool PHYS, bool REP>
__global__ void __maxnreg__(64) k_step_cluster(const KP kp, const SwarmState st, const SwarmStepIO io,
                                               const SwarmInjectedDraws dr, const int has_draws, const int nf,
                                               const SwarmStepFinal fin, const SwarmPhysics phys, const int repeat) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int T = ModeT<MODE>::T;
    const int N = kp.N, A = kp.A, tid = (int)threadIdx.x;
    const CMap m = cl_map(nf);
    const CSmem sm = cl_carve(smem_raw, N, A, kp.G, m.K, true);
    const int e = (int)blockIdx.x / m.K;
    const bool lead = m.rank == 0;
    double2* xe = reinterpret_cast<double2*>(st.x) + (size_t)e * N;
    double2* xae = reinterpret_cast<double2*>(st.xa) + (size_t)e * A;
    const int elapsed0 = st.elapsed[e];
    const uint32_t episode0 = st.episode[e];
    double* ph = nullptr;
    if constexpr (PHYS) {       // the row, visible after the barrier in front of the first agent move
        ph = phys_rows(smem_raw, cl_smem_bytes(N, A, kp.G, m.K, true));
        if (tid < kPhysCols) ph[tid] = phys.table[(size_t)e * kPhysCols + tid];
    }
    ClNoise nz{kp, st, &io, dr, {}, {}, 0u, e, has_draws != 0};
    nz.fresh_d.key = kp.key;
    nz.fresh_d.env = kp.env_off + (uint32_t)e;
    nz.fresh_d.episode = episode0 - 1u;      // the episode the last reset started
    nz.fresh_row = (uint32_t)kp.n_burn + (uint32_t)elapsed0;
    nz.reset_d = nz.fresh_d;
    nz.reset_d.episode = episode0;
    // the agents, in every CTA: state, noise row, actions (HBM dtype -> FP64, optional clip; rank 0 writes the clipped
    // actions back once every CTA has read them)
    bool clipped = false;
    double2 aclip = make_double2(0.0, 0.0);
    if (tid < A) {
        const int k = tid;
        sm.as[k] = xae[k];
        if (kp.fresh && !io.noise_a) sm.an[k] = draw_normal2(nz.fresh_d, STREAM_NOISE_A, nz.fresh_row, (uint32_t)k);
        else sm.an[k] = reinterpret_cast<const double2*>(io.noise_a ? io.noise_a : st.noise_a)[(size_t)e * A + k];
        double2 a;
        if (io.flags & SWARM_STEP_ACTIONS_F64) {
            a = reinterpret_cast<const double2*>(io.actions_f64)[(size_t)e * A + k];
        } else {
            const float2 f = reinterpret_cast<const float2*>(io.actions_f32)[(size_t)e * A + k];
            a = make_double2((double)f.x, (double)f.y);
        }
        if (io.flags & SWARM_STEP_CLIP_ACTIONS) {
            if (io.flags & SWARM_STEP_ACTIONS_F64) {
                const double d = sqrt(__dadd_rn(__dmul_rn(a.x, a.x), __dmul_rn(a.y, a.y)));
                if (d >= 1.0) {
                    a.x = a.x / d; a.y = a.y / d;
                    clipped = true;
                }
            } else {
                const float fx = (float)a.x, fy = (float)a.y;
                const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy)));
                if (d >= 1.0f) {
                    a = make_double2((double)__fdiv_rn(fx, d), (double)__fdiv_rn(fy, d));
                    clipped = true;
                }
            }
        }
        sm.act[k] = a;
        aclip = a;
    }
    if constexpr (PHYS) __syncthreads();
    float* v_out = io.v_out ? io.v_out + (size_t)e * N * 2 : nullptr;
    int elapsed = 0;
    int sub = 0;                // REP: substep of the step proper
    float rsum = 0.0f;          // REP: FP32 sum of the substeps' rewards
    for (int r = -1;;) {
        double2 pn[T];
        if constexpr (PHYS)
            cl_step_forces<MODE, PRECISE>(sm, phys_kp(kp, ph), m, xe, xae, (r < 0 && !kp.wind_step) ? 0.0 : ph[2], r, nz, v_out, pn);
        else
            cl_step_forces<MODE, PRECISE>(sm, kp, m, xe, xae, (r < 0 && !kp.wind_step) ? 0.0 : kp.wind, r, nz, v_out, pn);
        cluster_sync();     // every CTA has read the old state (and its actions): the new one may be written
        cl_store(kp, m, xe, pn);
        const double reward = cl_reward(sm, kp, m);
        if (r < 0) {
            elapsed = elapsed0 + 1;
            if constexpr (REP) elapsed += sub;
            const bool done = (reward >= 0.0) || (kp.max_steps > 0 && elapsed >= kp.max_steps);
            if constexpr (REP) {
                rsum = sub == 0 ? (float)reward : __fadd_rn(rsum, (float)reward);
                if (!done && ++sub < repeat) {
                    // the next substep's fresh rows: the locusts' are drawn inside cl_step_forces from nz.fresh_row, the
                    // agents' here, where cl_reset_row writes a burn-in row (read after the barrier below)
                    ++nz.fresh_row;
                    if (kp.fresh && !io.noise_a && tid < A)
                        sm.an[tid] = draw_normal2(nz.fresh_d, STREAM_NOISE_A, nz.fresh_row, (uint32_t)tid);
                    cluster_sync();     // the new state is in memory before any CTA reads it again
                    continue;
                }
            }
            if (lead && tid == 0) {
                io.reward[e] = REP ? rsum : (float)reward;
                io.done[e] = done ? 1 : 0;
                if constexpr (FIN) {
                    if (fin.terminated) fin.terminated[e] = reward >= 0.0 ? 1 : 0;
                    if (fin.truncated) fin.truncated[e] = (kp.max_steps > 0 && elapsed >= kp.max_steps) ? 1 : 0;
                }
            }
            if constexpr (FIN) {
                if (done && fin.x) cl_store(kp, m, reinterpret_cast<double2*>(fin.x) + (size_t)e * N, pn);
                if (done && fin.xa && lead && tid < A) reinterpret_cast<double2*>(fin.xa)[(size_t)e * A + tid] = sm.as[tid];
            }
            if (!(done && (io.flags & SWARM_STEP_AUTO_RESET))) break;      // cluster-uniform
            // the new episode's row: nobody reads the old one since the cluster barrier above; published by the one
            // that closes this iteration
            if constexpr (PHYS) {
                if (phys.flags & SWARM_PHYSICS_RESAMPLE) phys_reset_row(ph, phys, kp, e, episode0, tid, lead);
            }
            cl_reset_begin(sm, kp, m, e, xe, nz);
            v_out = nullptr;
            elapsed = 0;
        }
        if (cl_reset_row(sm, kp, m, e, ++r, st, nz)) {
            if (lead && tid == 0) st.episode[e] = episode0 + 1;
            break;
        }
        cluster_sync();     // the new state is in memory before any CTA reads it again
    }
    if (lead) {
        if (tid == 0) st.elapsed[e] = elapsed;
        if (tid < A) {
            xae[tid] = sm.as[tid];
            if (clipped) {
                const double2 a = aclip;
                if (io.flags & SWARM_STEP_ACTIONS_F64) reinterpret_cast<double2*>(io.actions_f64)[(size_t)e * A + tid] = a;
                else reinterpret_cast<float2*>(io.actions_f32)[(size_t)e * A + tid] = make_float2((float)a.x, (float)a.y);
            }
        }
    }
    if (io.grid)
        cl_raster<T, false>(sm, kp, m, xe, xae, io.grid + (size_t)e * kp.G * kp.G * 2, io.positions + (size_t)e * A * 2, nullptr);
    cluster_sync();         // no CTA leaves while a peer may still read its shared memory
}

// SwarmEnv._reset for the masked envs, cluster layout.  PHYS: k_reset's (rank 0 writes a drawn row back).
template <int MODE, bool PRECISE, bool PHYS>
__global__ void __maxnreg__(64) k_reset_cluster(const KP kp, const SwarmState st, const uint8_t* __restrict__ mask,
                                                const SwarmInjectedDraws dr, const int has_draws, const int nf,
                                                const SwarmPhysics phys) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int T = ModeT<MODE>::T;
    const int N = kp.N, A = kp.A, tid = (int)threadIdx.x;
    const CMap m = cl_map(nf);
    const int e = (int)blockIdx.x / m.K;
    if (mask && !mask[e]) return;            // the whole cluster
    const CSmem sm = cl_carve(smem_raw, N, A, kp.G, m.K, true);
    double2* xe = reinterpret_cast<double2*>(st.x) + (size_t)e * N;
    double2* xae = reinterpret_cast<double2*>(st.xa) + (size_t)e * A;
    const uint32_t ep = st.episode[e];
    double* ph = nullptr;
    if constexpr (PHYS) {       // visible after the cluster barrier in front of the first burn-in step
        ph = phys_rows(smem_raw, cl_smem_bytes(N, A, kp.G, m.K, true));
        phys_reset_row(ph, phys, kp, e, ep, tid, m.rank == 0);
    }
    ClNoise nz{kp, st, nullptr, dr, {}, {}, 0u, e, has_draws != 0};
    nz.reset_d.key = kp.key;
    nz.reset_d.env = kp.env_off + (uint32_t)e;
    nz.reset_d.episode = ep;
    cl_reset_begin(sm, kp, m, e, xe, nz);
    for (int r = 0; !cl_reset_row(sm, kp, m, e, r, st, nz); ++r) {
        cluster_sync();     // the state is in memory before any CTA reads it
        double2 pn[T];
        if constexpr (PHYS) cl_step_forces<MODE, PRECISE>(sm, phys_kp(kp, ph), m, xe, xae, ph[2], r, nz, nullptr, pn);
        else cl_step_forces<MODE, PRECISE>(sm, kp, m, xe, xae, kp.wind, r, nz, nullptr, pn);
        cluster_sync();     // every CTA has read the old state
        cl_store(kp, m, xe, pn);
    }
    cluster_sync();         // every CTA has read the episode counter
    if (m.rank == 0) {
        if (tid == 0) {
            st.elapsed[e] = 0;
            st.episode[e] = ep + 1;
        }
        if (tid < A) xae[tid] = sm.as[tid];
    }
}

// SwarmEnv.v_calculate for the batch, cluster layout.  PHYS: k_forces'.
template <int MODE, bool PRECISE, bool PHYS>
__global__ void __maxnreg__(64) k_forces_cluster(const KP kp, const double* __restrict__ x, const double* __restrict__ xa,
                                                 float* __restrict__ v, float* __restrict__ reward, const int nf,
                                                 const SwarmPhysics phys) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int T = ModeT<MODE>::T;
    const CMap m = cl_map(nf);
    const CSmem sm = cl_carve(smem_raw, kp.N, kp.A, kp.G, m.K, true);
    const int e = (int)blockIdx.x / m.K;
    const double2* xe = reinterpret_cast<const double2*>(x) + (size_t)e * kp.N;
    const double2* xae = reinterpret_cast<const double2*>(xa) + (size_t)e * kp.A;
    cl_stage<false>(sm, kp, xe, xae, 0.0);
    if (m.active) {
        float vx[T], vy[T];
        if constexpr (PHYS) cl_forces<MODE, PRECISE>(sm, phys_kp(kp, phys.table + (size_t)e * kPhysCols), m, vx, vy);
        else cl_forces<MODE, PRECISE>(sm, kp, m, vx, vy);
        if (v) {
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int j = m.vtid + t * m.nf;
                if (j < kp.N) reinterpret_cast<float2*>(v)[(size_t)e * kp.N + j] = make_float2(vx[t], vy[t]);
            }
        }
    }
    cluster_sync();         // every energy slot is in place
    const double r = cl_reward(sm, kp, m);
    if (reward && m.rank == 0 && threadIdx.x == 0) reward[e] = (float)r;
    cluster_sync();
}

// SwarmStateProcessor.process_state for the batch, cluster layout (k_rasterize's contract).
template <int T, bool EXACT>
__global__ void __launch_bounds__(1024) k_rasterize_cluster(const KP kp, const double* __restrict__ x,
                                                            const double* __restrict__ xa, float* __restrict__ grid,
                                                            uint8_t* __restrict__ positions, double* __restrict__ box,
                                                            const int nf, const uint8_t* __restrict__ mask) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const CMap m = cl_map(nf);
    const int e = (int)blockIdx.x / m.K;
    if (mask && !mask[e]) return;            // the whole cluster
    const CSmem sm = cl_carve(smem_raw, kp.N, kp.A, kp.G, m.K, false);
    cl_raster<T, EXACT>(sm, kp, m, reinterpret_cast<const double2*>(x) + (size_t)e * kp.N,
                        reinterpret_cast<const double2*>(xa) + (size_t)e * kp.A, grid + (size_t)e * kp.G * kp.G * 2,
                        positions + (size_t)e * kp.A * 2, box ? box + 4 * (size_t)e : nullptr);
    cluster_sync();
}

// ------------------------------------------------------------------------------------------ host side

thread_local char g_cuda_err[256] = "";

// debug timeline buffer (swarm_debug_trace); process-wide, nullptr in production
unsigned long long* g_trace = nullptr;
long long g_trace_slots = 0;

int cuda_fail(cudaError_t err, const char* what) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(err));
    return SWARM_ERR_LAUNCH;
}

constexpr size_t kMaxSmem = 227 * 1024;
constexpr int kMaxLocusts = 2048;
constexpr int kMaxThreads = 1024;

// N <= 512: unordered pairs -- MODE 3 (64-wide super-tiles, two targets per lane) when N pads to a
// multiple of 64 anyway, else MODE 1 (32-wide tiles, one target per lane); N > 512: ordered pairs
// with 2 or 4 targets per thread (MODE 2/4).
int force_mode(int N) {
    if (N <= kSymMaxLocusts) return ((N + 63) / 64) * 64 == ((N + 31) / 32) * 32 ? 3 : 1;
    return N <= 1024 ? 2 : 4;
}
int force_sym(int mode) { return mode == 1 ? 1 : (mode == 3 ? 2 : 0); }

// threads of the force group
int block_threads(int N, int mode) {
    if (mode == 3) return ((N + 63) / 64) * 32;
    const int per = (N + mode - 1) / mode;
    return ((per + 31) / 32) * 32;
}

// threads of the raster group riding along with the force group in k_step
// measured: 64 raster threads beat 32 for small swarms (1024 x 64: 14.2 vs 17.6 us per step)
// threads of the raster group that rides along in k_step (WARPS shape).  64 as a rule; 96 bin a small swarm's points in ONE
// round (N + A <= 96) -- taken when the CTA stays small (a single force warp: N = 64) or the batch has fewer CTAs than SMs,
// i.e. when the extra registers cost no resident CTA (measured, profiles/r02_shapes.md: 1024 x 64 13.1 -> 12.8 us,
// 4096 x 64 46.7 -> 45.1, 32 x 80 9.75 -> 9.0; but 4096 x 80 48.1 -> 55.9 with its three force warps)
int raster_threads(int N, int A, int nf, int E, int sms) {
    if (N + A <= 96 && (nf <= 32 || E <= sms)) return 96;
    return (N + A) <= 1024 ? 64 : 128;
}

// raster: 0 none, 1 raster group (own point buffer), 2 the force group rasterises
size_t step_smem(const SwarmParams* p, int raster, int n_stage, int mode) {
    return smem_bytes(p->n_locusts, p->n_agents, p->grid_size, n_stage, true, raster, force_sym(mode));
}

// The kernels read and write a grid cell's two channels as one float2: the grid must be 8-byte aligned.  (Any further
// alignment is optional: 16 bytes enables the TMA zero fill, the filler warp and 16-byte stores.)
bool grid_aligned(const void* grid) { return (reinterpret_cast<uintptr_t>(grid) & 7) == 0; }

// ---- CLUSTER layout: SwarmParams::tuning bits 8-12 = K (1..16 CTAs per env), kClusterAuto = the library picks K
constexpr int kClusterShift = 8, kClusterAuto = 31;
int tuning_cluster(const SwarmParams* p) { return p->tuning > 0 ? (p->tuning >> kClusterShift) & 31 : 0; }
// virtual warps of the env (the one-CTA kernel's force warps) and the cluster sizes they allow: at most one CTA per
// warp and kClusterMaxK; at least as many CTAs as it takes to keep a CTA within kMaxThreads
int cl_warps(int N) { return block_threads(N, force_mode(N)) >> 5; }
int cl_kmin(int N) { return (cl_warps(N) * 32 + kMaxThreads - 1) / kMaxThreads; }
int cl_kmax(int N) { return cl_warps(N) < kClusterMaxK ? cl_warps(N) : kClusterMaxK; }
bool cl_fits(const SwarmParams* p, int K, bool force) {
    return K >= cl_kmin(p->n_locusts) && cl_smem_bytes(p->n_locusts, p->n_agents, p->grid_size, K, force) <= kMaxSmem;
}
int validate_cluster(const SwarmParams* p, int cl) {
    if ((p->tuning & 0x30) || (cl > kClusterMaxK && cl != kClusterAuto)) return SWARM_ERR_FLAGS;
    // N <= 512: the one-CTA kernels take unordered pairs, which a cluster cannot reproduce bit for bit
    if (p->n_locusts < kClusterMinLocusts) return SWARM_ERR_FLAGS;
    if (cl != kClusterAuto) {
        if (cl > cl_kmax(p->n_locusts)) return SWARM_ERR_FLAGS;        // a CTA without a warp
        return cl_fits(p, cl, true) ? SWARM_OK : SWARM_ERR_SIZE;
    }
    for (int K = cl_kmin(p->n_locusts); K <= cl_kmax(p->n_locusts); ++K)
        if (cl_fits(p, K, true)) return SWARM_OK;
    return SWARM_ERR_SIZE;
}

int validate(const SwarmParams* p, int min_agents = 1) {
    if (!p) return SWARM_ERR_NULL;
    const int cl = tuning_cluster(p);
    if (p->n_envs < 1 || p->n_locusts < 1 || p->n_locusts > (cl ? kClusterMaxLocusts : kMaxLocusts)) return SWARM_ERR_SIZE;
    if (p->n_agents < min_agents || p->n_agents > 32) return SWARM_ERR_SIZE;
    if (p->grid_size < 2 || p->grid_size > 255) return SWARM_ERR_SIZE;      // positions are uint8
    if (p->n_burn_in < 0 || p->max_episode_steps < 0) return SWARM_ERR_SIZE;
    if (p->math_mode != 0 && p->math_mode != 1) return SWARM_ERR_FLAGS;
    if (p->tuning < 0 || (p->tuning & ~(0x30 | (31 << kClusterShift)))) return SWARM_ERR_FLAGS;
    if (cl) {
        if (int rc = validate_cluster(p, cl)) return rc;
    } else if (step_smem(p, 1, 2, force_mode(p->n_locusts)) > kMaxSmem) {
        return SWARM_ERR_SIZE;
    }
    if (p->env_id_offset < 0 || p->env_id_offset + p->n_envs > (int64_t)0xffffffffLL) return SWARM_ERR_SIZE;
    return SWARM_OK;
}

KP make_kp(const SwarmParams* p, int mode = 0) {
    KP k;
    memset(&k, 0, sizeof(k));
    if (!mode) mode = force_mode(p->n_locusts);
    k.E = p->n_envs; k.N = p->n_locusts; k.A = p->n_agents; k.G = p->grid_size;
    k.n_burn = p->n_burn_in; k.max_steps = p->max_episode_steps;
    k.sigma = p->noise; k.wind = p->wind; k.dt = p->dt;
    k.half_w = p->box_width / 2.0; k.y_hi = 2.0 * p->box_height;
    k.cscale = 1.4426950408889634;                 // log2(e): exp(-r) == exp2(-c r)
    k.F = (float)p->F;
    k.nInvL = (float)(-1.0 / p->L);
    k.U = (float)p->wind; k.Gv = (float)p->gravity;
    k.eps_s = (float)(1e-6 * 1.4426950408889634);  // multiagent.py:103 "+ 0.000001", scaled
    k.ri_max = 0.000244140625f / k.eps_s;          // eps / r <= 2^-12 (inv_r_eps)
    k.key = make_uint2((uint32_t)(p->seed & 0xffffffffu), (uint32_t)(p->seed >> 32));
    k.env_off = (uint32_t)p->env_id_offset;
    k.dynamic = 0;
    k.publish = 0;
    k.n_stage = 2;
    k.raster = 0;
    k.wind_step = 1;
    // numpy: linspace(0, 2 HEIGHT, G + 1) has step (hi - lo) / G, rounded once (state_processors.py:31-32)
    k.step_y = (k.y_hi - 0.0) / (double)k.G;
    k.inv_y = 1.0 / k.step_y;
    k.inv_x = (double)k.G / (2.0 * k.half_w);
    k.inv_P = 1.0 / (double)(k.N + k.A);
    k.inv_G = 1.0 / (double)k.G;
    k.inv_N = 1.0 / (double)k.N;
    k.trace = g_trace;
    k.trace_slots = g_trace_slots;
    return k;
}

// Per (device, kernel) launch cache: the opt-in shared-memory ceiling already granted and the
// occupancy (CTAs/SM) of the configurations seen, so that the steady-state cost of an entry
// point is one cudaGetDevice + one launch.
// Side stream (higher priority) + fork/join events of the two-kernel step: one set per (device, caller stream), so
// that calls on different streams -- from one host thread or several -- never share an event or serialise their
// followers, and a stream that is being captured only ever pulls ITS side stream into the capture.
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};

struct KernelCache {
    std::mutex mu;
    std::map<std::pair<int, cudaStream_t>, SideStream> side;
    std::map<std::pair<int, const void*>, size_t> smem_set;
    std::map<std::tuple<int, const void*, int, size_t>, int> occupancy;
    std::map<std::pair<int, const void*>, int> regs;
    std::map<int, int> sms;
};
KernelCache& cache() {
    static KernelCache c;
    return c;
}

int current_device(int* dev) {
    cudaError_t err = cudaGetDevice(dev);
    return err == cudaSuccess ? SWARM_OK : cuda_fail(err, "cudaGetDevice");
}

template <typename K>
int prep(K kernel, size_t smem) {
    int dev = 0;
    if (int rc = current_device(&dev)) return rc;
    KernelCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    auto key = std::make_pair(dev, (const void*)kernel);
    const bool first = c.smem_set.find(key) == c.smem_set.end();
    size_t& have = c.smem_set[key];
    if (first) {
        // every kernel asks for the same (maximal) shared-memory carve-out: an SM cannot change its L1/shared split
        // while a CTA is resident, and the step and its follower must be able to share SMs
        cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                               (int)cudaSharedmemCarveoutMaxShared);
        if (err != cudaSuccess) return cuda_fail(err, "cudaFuncSetAttribute(carveout)");
    }
    if (smem > 48 * 1024 && smem > have) {
        cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return cuda_fail(err, "cudaFuncSetAttribute");
        have = smem;
    }
    return SWARM_OK;
}

// occupancy (CTAs per SM) of a launch shape and the SM count of the current device
template <typename K>
int occupancy(K kernel, int threads, size_t smem, int* per_sm_out, int* n_sms = nullptr) {
    int dev = 0;
    if (int rc = current_device(&dev)) return rc;
    KernelCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    auto s = c.sms.find(dev);
    if (s == c.sms.end()) {
        int n = 0;
        cudaError_t err = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (err != cudaSuccess) return cuda_fail(err, "cudaDeviceGetAttribute");
        s = c.sms.emplace(dev, n).first;
    }
    const auto key = std::make_tuple(dev, (const void*)kernel, threads, smem);
    auto o = c.occupancy.find(key);
    if (o == c.occupancy.end()) {
        int per_sm = 0;
        cudaFuncAttributes fa;
        cudaError_t err = cudaFuncGetAttributes(&fa, kernel);        // also forces the (lazily loaded) kernel in
        if (err == cudaSuccess) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
        if (err != cudaSuccess) return cuda_fail(err, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
        c.regs[std::make_pair(dev, (const void*)kernel)] = fa.numRegs;
        o = c.occupancy.emplace(key, per_sm).first;
    }
    *per_sm_out = o->second;
    if (n_sms) *n_sms = s->second;
    return SWARM_OK;
}

// grid of a persistent kernel: every SM filled to its occupancy, never more CTAs than envs
template <typename K>
int persistent_grid(K kernel, int threads, size_t smem, int n_envs, int* grid, int* n_sms = nullptr) {
    int per_sm = 0, sms = 1;
    if (int rc = occupancy(kernel, threads, smem, &per_sm, &sms)) return rc;
    if (per_sm < 1) per_sm = 1;
    const long long slots = (long long)sms * per_sm;
    *grid = (int)(n_envs < slots ? n_envs : slots);
    if (n_sms) *n_sms = sms;
    return SWARM_OK;
}

// registers per thread of a kernel occupancy() has seen on the current device (0 if unknown)
int kernel_regs(const void* kernel) {
    int dev = 0;
    if (current_device(&dev)) return 0;
    KernelCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    auto r = c.regs.find(std::make_pair(dev, kernel));
    return r == c.regs.end() ? 0 : r->second;
}

int check_launch(const char* what) {
    cudaError_t err = cudaGetLastError();
    return err == cudaSuccess ? SWARM_OK : cuda_fail(err, what);
}

// ---- CLUSTER layout: shape and launch ------------------------------------------------------------------------------
struct ClusterShape {
    int K, nf, nt;
    size_t smem;
};

// clusters of K CTAs of this kernel that the device can hold at once (0: unschedulable), cached per device
template <typename Kern>
int cluster_occupancy(Kern kernel, int K, int nt, size_t smem, int* out) {
    int dev = 0;
    if (int rc = current_device(&dev)) return rc;
    KernelCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    const auto key = std::make_tuple(dev, (const void*)kernel, nt * 32 + K, smem);
    auto o = c.occupancy.find(key);
    if (o == c.occupancy.end()) {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3((unsigned)K);
        cfg.blockDim = dim3((unsigned)nt);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)K;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int n = 0;
        const cudaError_t err = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
        if (err != cudaSuccess) {
            cudaGetLastError();
            n = 0;                     // e.g. a cluster size the device does not support: refused, not a failure
        }
        o = c.occupancy.emplace(key, n).first;
    }
    *out = o->second;
    return SWARM_OK;
}

// The cluster size of a call and its launch shape.  Refuses (SWARM_ERR_SIZE) a size whose shared memory or cluster does
// not fit the device -- before anything is launched.  The library's choice (kClusterAuto) is the largest K whose clusters
// the device can hold for the whole batch at once (cudaOccupancyMaxActiveClusters >= E: one wave), else the smallest K.
// Measured (profiles/r04_cluster.md): K beyond one wave costs a second wave (8192 x 16: K = 6 2.18 ms, K = 7 4.32 ms),
// and in multi-wave batches more CTAs per env only add the per-CTA work (N = 2048, E = 148: K = 1 0.67 ms, K = 4 0.95).
// phys_bytes: the PHYS kernels' physics row behind the carve
template <typename Kern>
int cluster_shape(const SwarmParams* p, Kern kernel, bool force, ClusterShape* out, size_t phys_bytes = 0) {
    const int N = p->n_locusts, cl = tuning_cluster(p);
    const int nf = block_threads(N, force_mode(N)), nw = nf >> 5;
    const bool pick = cl == kClusterAuto;
    const int k_hi = pick ? cl_kmax(N) : cl, k_lo = pick ? cl_kmin(N) : cl;
    ClusterShape fallback = {0, 0, 0, 0};
    for (int K = k_hi; K >= k_lo; --K) {
        if (!cl_fits(p, K, force)) continue;
        const int nt = cl_threads(nw, K);
        const size_t smem = cl_smem_bytes(N, p->n_agents, p->grid_size, K, force) + phys_bytes;
        if (smem > kMaxSmem) continue;
        int rc = prep(kernel, smem);
        if (rc) return rc;
        if (K > 8) {
            const cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (err != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
        }
        int n = 0;
        if ((rc = cluster_occupancy(kernel, K, nt, smem, &n))) return rc;
        if (n < 1) continue;
        const ClusterShape sh = {K, nf, nt, smem};
        if (!pick || n >= p->n_envs) {
            *out = sh;
            return SWARM_OK;
        }
        fallback = sh;                 // the smallest schedulable K so far
    }
    if (fallback.K == 0) return SWARM_ERR_SIZE;
    *out = fallback;
    return SWARM_OK;
}

template <typename Kern, typename... Args>
int launch_cluster(Kern kernel, const ClusterShape& sh, int n_envs, cudaStream_t s, const char* what, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)((long long)n_envs * sh.K));
    cfg.blockDim = dim3((unsigned)sh.nt);
    cfg.dynamicSmemBytes = sh.smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)sh.K;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t err = cudaLaunchKernelEx(&cfg, kernel, args...);
    if (err != cudaSuccess) return cuda_fail(err, what);
    return check_launch(what);
}

#define DISPATCH_T(T_, ...)              \
    switch (T_) {                        \
        case 1: { constexpr int TT = 1; __VA_ARGS__; } break; \
        case 2: { constexpr int TT = 2; __VA_ARGS__; } break; \
        case 3: { constexpr int TT = 3; __VA_ARGS__; } break; \
        default: { constexpr int TT = 4; __VA_ARGS__; } break; \
    }

// swarm_step_host keeps the launches of its last argument sets as instantiated graphs (per host thread)
struct HostStepKey {
    SwarmParams p;
    SwarmState st;
    SwarmStepIO io;
    float* host_grid;
    uint8_t* host_positions;
    int device;
};
constexpr int kHostGraphs = 32;     // distinct (params, state, buffers) argument sets kept per host thread
struct HostStepCache {
    struct Entry {
        HostStepKey key;
        cudaGraphExec_t exec = nullptr;
    } entries[kHostGraphs];
    unsigned next_victim = 0;
    bool capture_failure_reported = false;
    void clear() {
        for (Entry& e : entries)
            if (e.exec) {
                cudaGraphExecDestroy(e.exec);
                e.exec = nullptr;
            }
    }
    ~HostStepCache() { clear(); }       // thread exit: the graphs go with the thread
};
HostStepCache& host_cache() {
    static thread_local HostStepCache c;
    return c;
}

// device-visible alias of a pinned (page-locked, UVA-mapped) host pointer, or nullptr
template <typename T>
T* mapped_host(T* host) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return a.type == cudaMemoryTypeHost ? static_cast<T*>(a.devicePointer) : nullptr;
}

typedef void (*StepKernel)(const KP, const SwarmState, const SwarmStepIO, const SwarmInjectedDraws, const int, const int,
                           const SwarmStepFinal, const SwarmPhysics, const int);

template <int PLACE, bool FIN, bool PHYS, bool REP>
StepKernel step_kernel_p(int mode, bool precise) {
    switch (mode) {
        case 1: return precise ? k_step<1, true, PLACE, FIN, PHYS, REP> : k_step<1, false, PLACE, FIN, PHYS, REP>;
        case 2: return precise ? k_step<2, true, PLACE, FIN, PHYS, REP> : k_step<2, false, PLACE, FIN, PHYS, REP>;
        case 3: return precise ? k_step<3, true, PLACE, FIN, PHYS, REP> : k_step<3, false, PLACE, FIN, PHYS, REP>;
        default: return precise ? k_step<4, true, PLACE, FIN, PHYS, REP> : k_step<4, false, PLACE, FIN, PHYS, REP>;
    }
}
template <bool FIN, bool PHYS, bool REP = false>
StepKernel step_kernel_f(int mode, bool precise, int place) {
    return place == 2 ? step_kernel_p<2, FIN, PHYS, REP>(mode, precise)
                      : (place == 3 ? step_kernel_p<3, FIN, PHYS, REP>(mode, precise)
                                    : step_kernel_p<0, FIN, PHYS, REP>(mode, precise));
}
// place: RasterPlace (NONE / FOLLOW share the rasteriser-less kernel); fin: the swarm_step_final variant; phys: the
// swarm_step_physics one; rep: the swarm_step_repeat one (with and without FIN: a FIN kernel whose fin pointers are all
// null was measured 2.8 % slower than the FIN = false one on the C4 step, profiles/r07_action_repeat.md)
StepKernel step_kernel(int mode, bool precise, int place, bool fin, bool phys, bool rep) {
    if (rep && phys) return fin ? step_kernel_f<true, true, true>(mode, precise, place) : step_kernel_f<false, true, true>(mode, precise, place);
    if (rep) return fin ? step_kernel_f<true, false, true>(mode, precise, place) : step_kernel_f<false, false, true>(mode, precise, place);
    if (phys) return fin ? step_kernel_f<true, true>(mode, precise, place) : step_kernel_f<false, true>(mode, precise, place);
    return fin ? step_kernel_f<true, false>(mode, precise, place) : step_kernel_f<false, false>(mode, precise, place);
}

template <bool FIN, bool PHYS, bool REP = false>
StepKernel step_kernel_cluster_f(int mode, bool precise) {
    return mode == 2 ? (precise ? k_step_cluster<2, true, FIN, PHYS, REP> : k_step_cluster<2, false, FIN, PHYS, REP>)
                     : (precise ? k_step_cluster<4, true, FIN, PHYS, REP> : k_step_cluster<4, false, FIN, PHYS, REP>);
}
StepKernel step_kernel_cluster(int mode, bool precise, bool fin, bool phys, bool rep) {
    if (rep && phys) return fin ? step_kernel_cluster_f<true, true, true>(mode, precise) : step_kernel_cluster_f<false, true, true>(mode, precise);
    if (rep) return fin ? step_kernel_cluster_f<true, false, true>(mode, precise) : step_kernel_cluster_f<false, false, true>(mode, precise);
    if (phys) return fin ? step_kernel_cluster_f<true, true>(mode, precise) : step_kernel_cluster_f<false, true>(mode, precise);
    return fin ? step_kernel_cluster_f<true, false>(mode, precise) : step_kernel_cluster_f<false, false>(mode, precise);
}

const SwarmInjectedDraws kNoDraws = {nullptr, nullptr, nullptr, nullptr, nullptr};
const SwarmStepFinal kNoFinal = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
const SwarmPhysics kNoPhysics = {nullptr, 0u, 0u, {0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0}};

// SwarmPhysics' host checks (before any CUDA call)
int check_physics(const SwarmPhysics* ph) {
    if (!ph || !ph->table) return SWARM_ERR_NULL;
    if ((reinterpret_cast<uintptr_t>(ph->table) & 15) || (ph->flags & ~SWARM_PHYSICS_RESAMPLE) || ph->reserved)
        return SWARM_ERR_FLAGS;
    if (ph->flags & SWARM_PHYSICS_RESAMPLE) {
        for (int c = 0; c < kPhysCols; ++c) {
            const double lo = ph->lo[c], hi = ph->hi[c];
            if (!std::isfinite(lo) || !std::isfinite(hi) || !(lo <= hi) || !std::isfinite(hi - lo)) return SWARM_ERR_SIZE;
        }
        if (!(ph->lo[4] > 0.0)) return SWARM_ERR_SIZE;       // L: the pair force divides by it
    }
    return SWARM_OK;
}

bool draws_complete(const SwarmInjectedDraws* d) {
    return d->x0 && d->xa0 && d->burn_actions && d->agent_noise && d->particle_noise;
}

// ---- launch shape of swarm_step ------------------------------------------------------------------------------
// WHERE the observation is produced (same results every way):
//   FOLLOW  k_raster_follow on the side stream trails a rasteriser-less, one-env-per-CTA k_step (needs 2 + E flags)
//   WARPS   a raster warp group inside persistent k_step CTAs, one env behind the force group
//   SELF    the step's own threads rasterise their env right after stepping it (one env per CTA)
//   CLUSTER the env's K CTAs of a thread-block cluster rasterise it after the step (the cluster layout, tuning bits 8-12)
enum RasterPlace { RASTER_NONE = 0, RASTER_FOLLOW = 1, RASTER_WARPS = 2, RASTER_SELF = 3, RASTER_CLUSTER = 4 };

struct StepShape {
    int mode;        // force mode (1..6)
    int place;       // RasterPlace
    int follow_threads, follow_per_sm;
    size_t follow_smem;
};

bool env_flag(const char* name) {
    const char* v = getenv(name);
    return v && v[0] && v[0] != '0';
}

}  // namespace

// ------------------------------------------------------------------------------------------ C ABI

extern "C" {

int swarm_abi_version(void) { return SWARM_ABI_VERSION; }

const char* swarm_strerror(int status) {
    switch (status) {
        case SWARM_OK: return "ok";
        case SWARM_ERR_NULL: return "required pointer is NULL";
        case SWARM_ERR_SIZE:
            return "unsupported size (E>=1, 1<=N<=2048 in one CTA per env or 513<=N<=8192 in the cluster layout, 1<=A<=32, "
                   "2<=G<=255, shared memory <= 227 KB, a cluster the device can schedule)";
        case SWARM_ERR_LAUNCH: return "CUDA launch/runtime error (see swarm_last_cuda_error)";
        case SWARM_ERR_FLAGS:
            return "inconsistent flags or missing optional buffer (the cluster layout: N > 512, K <= 16 and at most one CTA "
                   "per force warp, no raster placement)";
        default: return "unknown status";
    }
}

const char* swarm_last_cuda_error(void) { return g_cuda_err; }

int swarm_validate(const SwarmParams* p) { return validate(p); }

}  // extern "C"

namespace {

// swarm_reset's launches (PHYS: the k_reset* variants with per-env physics)
template <bool PHYS>
int reset_launch(const SwarmParams* p, const SwarmState* st, const SwarmPhysics& phys, const uint8_t* mask,
                 const SwarmInjectedDraws* draws, swarm_stream_t stream) {
    int rc = 0;
    if (!st || !st->x || !st->xa || !st->noise_x || !st->noise_a || !st->elapsed || !st->episode) return SWARM_ERR_NULL;
    if (draws && !draws_complete(draws)) return SWARM_ERR_NULL;
    const int mode = force_mode(p->n_locusts);
    const KP kp = make_kp(p, mode);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t phys_bytes = PHYS ? kPhysRowBytes : 0;
    if (tuning_cluster(p)) {
        const SwarmInjectedDraws dr = draws ? *draws : kNoDraws;
        const int has = draws ? 1 : 0;
        ClusterShape sh;
        auto go = [&](auto kernel) {
            int r = cluster_shape(p, kernel, true, &sh, phys_bytes);
            return r ? r : launch_cluster(kernel, sh, kp.E, s, "swarm_reset", kp, *st, mask, dr, has, sh.nf, phys);
        };
        if (mode == 2) return p->math_mode ? go(k_reset_cluster<2, true, PHYS>) : go(k_reset_cluster<2, false, PHYS>);
        return p->math_mode ? go(k_reset_cluster<4, true, PHYS>) : go(k_reset_cluster<4, false, PHYS>);
    }
    const size_t smem = step_smem(p, 0, 1, mode) + phys_bytes;
    if (smem > kMaxSmem) return SWARM_ERR_SIZE;
    const int nt = block_threads(kp.N, mode);
    if (nt > kMaxThreads) return SWARM_ERR_SIZE;
    DISPATCH_T(mode,
        if (p->math_mode) {
            if ((rc = prep(k_reset<TT, true, PHYS>, smem))) return rc;
            k_reset<TT, true, PHYS><<<kp.E, nt, smem, s>>>(kp, *st, mask, draws ? *draws : kNoDraws, draws ? 1 : 0, phys);
        } else {
            if ((rc = prep(k_reset<TT, false, PHYS>, smem))) return rc;
            k_reset<TT, false, PHYS><<<kp.E, nt, smem, s>>>(kp, *st, mask, draws ? *draws : kNoDraws, draws ? 1 : 0, phys);
        })
    return check_launch("swarm_reset");
}

}  // namespace

extern "C" {

int swarm_reset(const SwarmParams* p, const SwarmState* st, const uint8_t* mask, const SwarmInjectedDraws* draws,
                swarm_stream_t stream) {
    const int rc = validate(p);
    return rc ? rc : reset_launch<false>(p, st, kNoPhysics, mask, draws, stream);
}

int swarm_reset_physics(const SwarmParams* p, const SwarmState* st, const SwarmPhysics* phys, const uint8_t* mask,
                        const SwarmInjectedDraws* draws, swarm_stream_t stream) {
    int rc = validate(p);
    if (!rc) rc = check_physics(phys);
    return rc ? rc : reset_launch<true>(p, st, *phys, mask, draws, stream);
}

}  // extern "C"

namespace {

struct StepPlan {
    int mode, place;              // force mode (1..4), RasterPlace
    int nf, nt, grid;             // force threads, threads per CTA, CTAs
    int n_stage, dynamic, raster, filler; // KP fields
    int follow_threads, rgrid;    // follower launch (place == RASTER_FOLLOW)
    size_t smem, follow_smem;
    StepKernel kernel;
    int cluster;                  // CTAs per env (place == RASTER_CLUSTER)
};

// Validates the arguments of swarm_step and decides its launch shape (automatic, or forced through
// SwarmParams::tuning).  Touches the GPU only for attribute / occupancy queries (cached per device).
// phys: the PHYS kernels, with the physics rows of their stage buffers behind their shared memory.  repeat > 1: the REP
// kernels.
int plan_step(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmInjectedDraws* reset_draws,
              StepPlan* out, const bool fin = false, const bool phys = false, const int repeat = 1) {
    int rc = validate(p);
    if (rc) return rc;
    if (!st || !io) return SWARM_ERR_NULL;
    if (!st->x || !st->xa || !st->noise_x || !st->noise_a || !st->elapsed || !st->episode) return SWARM_ERR_NULL;
    if (!io->reward || !io->done) return SWARM_ERR_NULL;
    if ((io->flags & SWARM_STEP_ACTIONS_F64) ? !io->actions_f64 : !io->actions_f32) return SWARM_ERR_NULL;
    if ((io->grid != nullptr) != (io->positions != nullptr)) return SWARM_ERR_FLAGS;
    if (!grid_aligned(io->grid)) return SWARM_ERR_FLAGS;
    if (io->flags & ~(SWARM_STEP_AUTO_RESET | SWARM_STEP_CLIP_ACTIONS | SWARM_STEP_ACTIONS_F64 | SWARM_STEP_NO_ACTION_WIND |
                      SWARM_STEP_INKERNEL_RASTER | SWARM_STEP_FRESH_NOISE))
        return SWARM_ERR_FLAGS;
    if (reset_draws && !draws_complete(reset_draws)) return SWARM_ERR_NULL;
    if (st->work_words && !st->work) return SWARM_ERR_NULL;
    const int N = p->n_locusts, A = p->n_agents, E = p->n_envs;
    const bool want_grid = io->grid != nullptr;
    const bool have_queue = st->work != nullptr && st->work_words >= 2;
    const bool have_flags = st->work != nullptr && st->work_words >= 2 + (uint64_t)E;
    int sms = 148;
    {
        int dev = 0;
        if ((rc = current_device(&dev))) return rc;
        KernelCache& c = cache();
        std::lock_guard<std::mutex> lk(c.mu);
        auto it = c.sms.find(dev);
        if (it == c.sms.end()) {
            int n = 0;
            cudaError_t err = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
            if (err != cudaSuccess) return cuda_fail(err, "cudaDeviceGetAttribute");
            it = c.sms.emplace(dev, n).first;
        }
        sms = it->second;
    }
    const int filler_threads = 32;                           // the SELF shape's TMA zero-fill warp
    const int mode = force_mode(N);
    const int nf = block_threads(N, mode);
    const bool rep = repeat > 1;
    out->cluster = 0;
    if (tuning_cluster(p)) {
        // one env per thread-block cluster; the observation (if any) comes from the cluster itself, st->work is not used
        ClusterShape sh;
        out->kernel = step_kernel_cluster(mode, p->math_mode != 0, fin, phys, rep);
        if ((rc = cluster_shape(p, out->kernel, true, &sh, phys ? kPhysRowBytes : 0))) return rc;
        out->mode = mode; out->place = RASTER_CLUSTER;
        out->raster = 0; out->n_stage = 0; out->filler = 0; out->dynamic = 0;
        out->nf = sh.nf; out->nt = sh.nt; out->smem = sh.smem; out->cluster = sh.K;
        out->grid = (int)((long long)E * sh.K);
        out->follow_threads = 0; out->follow_smem = 0; out->rgrid = 0;
        return SWARM_OK;
    }
    if (nf > kMaxThreads) return SWARM_ERR_SIZE;
    // With the per-env flags the observation can be produced by a second kernel that follows the step on a higher-priority
    // stream (k_raster_follow).  The follower spins until the step publishes an env, so the step must always be able to get
    // onto an SM next to it: shared memory, threads AND registers of both have to fit (checked below).
    const int follow_threads = (N + A) <= 128 ? 32 : 128;
    const size_t follow_smem = smem_bytes(N, A, p->grid_size, 0, false, 1, 0);
    // raster CTAs per SM that keep pace with the step (measured at 4096 envs: N = 160: 4 -> 0.110 ms, 2 -> 0.118; N = 192 and up: 2)
    int follow_per_sm = (N + A) <= 128 ? 6 : (N < 192 ? 4 : 2);
    while (follow_per_sm > 0 &&
           follow_per_sm * (follow_smem + 1024) + step_smem(p, 0, 1, mode) + (phys ? kPhysRowBytes : 0) + 1024 > kMaxSmem)
        --follow_per_sm;
    const bool no_follower = (io->flags & SWARM_STEP_INKERNEL_RASTER) || env_flag("SWARM_B200_NO_FOLLOWER");
    const StepKernel kernel = step_kernel(mode, p->math_mode != 0, RASTER_FOLLOW, fin, phys, rep);     // the rasteriser-less kernel
    bool follow_fits = have_flags && !no_follower && follow_per_sm > 0 && follow_per_sm * follow_threads + nf <= 2048;
    int rgrid = 0;
    if (want_grid && follow_fits) {
        // registers: follow_per_sm follower CTAs must leave room for at least one step CTA on every SM
        const size_t smem0 = step_smem(p, 0, 1, mode) + (phys ? kPhysRowBytes : 0);
        int o = 0;
        if ((rc = prep(kernel, smem0)) || (rc = occupancy(kernel, nf, smem0, &o))) return rc;
        if ((rc = prep(k_raster_follow, follow_smem))) return rc;
        if ((rc = persistent_grid(k_raster_follow, follow_threads, follow_smem, E, &rgrid))) return rc;
        const long long rs = kernel_regs((const void*)kernel), rf = kernel_regs((const void*)k_raster_follow);
        while (follow_per_sm > 1 && follow_per_sm * follow_threads * rf + nf * rs > 65536) --follow_per_sm;
        if (follow_per_sm * follow_threads * rf + nf * rs > 65536) follow_fits = false;
        if (rgrid > sms * follow_per_sm) rgrid = sms * follow_per_sm;
    }
    const bool warps_fit = nf + raster_threads(N, A, nf, E, sms) <= kMaxThreads &&
                           step_smem(p, 1, 2, mode) + (phys ? 2 * kPhysRowBytes : 0) <= kMaxSmem;
    int place = RASTER_NONE;
    if (want_grid) {
        const int forced = (p->tuning >> 4) & 3;
        // Measured (B200, 4096 envs): the follower wins for large swarms in multi-wave batches (N = 256: 0.181 vs 0.199 ms,
        // N = 192: 0.123 vs 0.135), the raster warps for small swarms, where the rasteriser -- not the forces -- is the
        // critical path (N = 128: 0.080 vs 0.108 ms, N = 64: 0.052 vs 0.069).  Batches of at most about one wave of
        // one-env CTAs have nothing to hide the rasteriser under: there the step's own threads rasterise (SELF).
        const int per_sm = 65536 / (64 * (nf + filler_threads)) > 0 ? 65536 / (64 * (nf + filler_threads)) : 1;
        // ... measured (profiles/r02_shapes.md): SELF wins from 96 force threads up (1024 x 80: 17.8 vs 19.5 us, 512 x 256: 37.0
        // vs 39.3); with one or two force warps per env the dedicated raster warps stay ahead (1024 x 64: 13.9 vs 20.2),
        // and so they do when there are fewer CTAs than SMs (32 x 80: 10.4 vs 11.0).
        if (forced) place = forced;
        // Large swarms (N >= 160, where the alternative is the follower kernel) keep SELF up to 4 CTAs per SM: beyond that the
        // batch is XU-bound like a multi-wave one and the follower overlaps better (1024 x 192: 43.5 vs 46.0 us).
        else if (E > sms && nf >= 96 && E <= (long long)sms * (N >= 160 && per_sm > 4 ? 4 : per_sm)) place = RASTER_SELF;
        else if (N >= 160) place = RASTER_FOLLOW;
        // Action repeat keeps each env K times longer in its step CTA.  Measured (profiles/r07_action_repeat.md): in
        // multi-wave batches with three or more force warps the follower then overtakes the raster warps (4096 x 80:
        // K = 2 85.3 vs 89.7 us per decision, K = 4 140.7 vs 154.1, K = 8 252.3 vs 284.6); with one force warp it does
        // not (1024 x 64, K = 4: 40.4 vs 32.4).  K = 1 keeps its choice.
        else if (rep && E > sms && nf >= 96) place = RASTER_FOLLOW;
        else place = RASTER_WARPS;
        if (place == RASTER_FOLLOW && !follow_fits) place = RASTER_WARPS;
        if (place == RASTER_WARPS && !warps_fit) place = RASTER_SELF;
    }
    const bool warps = place == RASTER_WARPS, self = place == RASTER_SELF;
    out->mode = mode; out->place = place;
    out->raster = warps ? 1 : (self ? 2 : 0);
    out->n_stage = warps ? 2 : 1;         // one env per CTA (no raster warps): nothing to prefetch into a second buffer
    out->smem = step_smem(p, out->raster, out->n_stage, mode) + (phys ? out->n_stage * kPhysRowBytes : 0);
    if (out->smem > kMaxSmem) return SWARM_ERR_SIZE;
    out->nf = nf;
    // SELF: one extra warp issues / awaits the TMA zero fill (possible when the grid is a whole number of 16-byte words
    // per table-sized piece: cells % 8 == 0, 16-byte aligned base)
    // ... as long as its 32 threads do not push the batch out of a single wave of CTAs (registers)
    out->filler = (self && ((p->grid_size * p->grid_size) & 7) == 0 && (reinterpret_cast<uintptr_t>(io->grid) & 15) == 0 &&
                   nf + 32 <= kMaxThreads && E <= (long long)sms * (65536 / (64 * (nf + 32)))) ? 1 : 0;
    out->nt = nf + (warps ? raster_threads(N, A, nf, E, sms) : 0) + (out->filler ? 32 : 0);
    out->kernel = step_kernel(mode, p->math_mode != 0, place, fin, phys, rep);
    if ((rc = prep(out->kernel, out->smem))) return rc;
    int grid = 0;
    if ((rc = persistent_grid(out->kernel, out->nt, out->smem, E, &grid))) return rc;
    // without raster warps to overlap there is nothing to gain from persistence, and hardware-scheduled one-env
    // CTAs measure 8 % faster (C4: 0.154 vs 0.166 ms)
    if (!warps) grid = E;
    out->grid = grid;
    // the work queue pays off when every CTA has several large envs to work through (one contended atomic per env)
    out->dynamic = (warps && have_queue && E >= 3 * grid && (long long)N * (N + A) >= 16384) ? 1 : 0;
    out->follow_threads = follow_threads;
    out->follow_smem = follow_smem;
    out->rgrid = rgrid;
    return SWARM_OK;
}

}  // namespace

extern "C" {

static int step_plan_out(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const bool phys, int32_t out[8],
                         const int repeat = 1) {
    if (!out) return SWARM_ERR_NULL;
    StepPlan pl;
    const int rc = plan_step(p, st, io, nullptr, &pl, false, phys, repeat);
    if (rc) return rc;
    out[0] = pl.mode; out[1] = pl.filler; out[2] = pl.place; out[3] = pl.nt; out[4] = pl.grid;
    out[5] = (int32_t)pl.smem; out[6] = pl.place == RASTER_FOLLOW ? pl.rgrid : (pl.place == RASTER_CLUSTER ? pl.cluster : 0);
    out[7] = pl.place == RASTER_FOLLOW ? 2 : 1;
    return SWARM_OK;
}

int swarm_step_plan(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, int32_t out[8]) {
    return step_plan_out(p, st, io, false, out);
}

int swarm_step_plan_physics(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmPhysics* phys,
                            int32_t out[8]) {
    int rc = validate(p);
    if (!rc) rc = check_physics(phys);
    return rc ? rc : step_plan_out(p, st, io, true, out);
}

int swarm_step_plan_repeat(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmPhysics* phys,
                           int32_t repeat, int32_t out[8]) {
    int rc = validate(p);
    if (!rc && repeat < 1) rc = SWARM_ERR_SIZE;
    if (!rc && phys) rc = check_physics(phys);
    return rc ? rc : step_plan_out(p, st, io, phys != nullptr, out, repeat);
}

// SwarmStateProcessor.process_state of the batch (or of the envs with mask[e] != 0): swarm_rasterize's launches.
static int rasterize_launch(const SwarmParams* p, const double* x, const double* xa, float* grid, uint8_t* positions,
                            double* box, const uint8_t* mask, swarm_stream_t stream) {
    int rc = 0;
    const KP kp = make_kp(p);
    if (tuning_cluster(p)) {
        const cudaStream_t s = (cudaStream_t)stream;
        ClusterShape sh;
        auto go = [&](auto kernel) {
            int r = cluster_shape(p, kernel, false, &sh);
            return r ? r : launch_cluster(kernel, sh, kp.E, s, "swarm_rasterize", kp, x, xa, grid, positions, box, sh.nf, mask);
        };
        if (force_mode(kp.N) == 2) return box ? go(k_rasterize_cluster<2, true>) : go(k_rasterize_cluster<2, false>);
        return box ? go(k_rasterize_cluster<4, true>) : go(k_rasterize_cluster<4, false>);
    }
    const size_t smem = smem_bytes(kp.N, kp.A, kp.G, 0, false, 1, 0);
    const int nt = (kp.N + kp.A) <= 128 ? 64 : 128;
    if (box) {
        if ((rc = prep(k_rasterize<true>, smem))) return rc;
        k_rasterize<true><<<kp.E, nt, smem, (cudaStream_t)stream>>>(kp, x, xa, grid, positions, box, mask);
    } else {
        if ((rc = prep(k_rasterize<false>, smem))) return rc;
        k_rasterize<false><<<kp.E, nt, smem, (cudaStream_t)stream>>>(kp, x, xa, grid, positions, box, mask);
    }
    return check_launch("swarm_rasterize");
}

// swarm_step's launches; with terminal outputs (fin_out != NULL) the FIN variants of the step kernels, with per-env
// physics (phys_in != NULL, checked) the PHYS ones, with repeat > 1 the REP ones
static int step_launch(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin_out,
                       const SwarmInjectedDraws* reset_draws, swarm_stream_t stream, const SwarmPhysics* phys_in = nullptr,
                       const int repeat = 1) {
    StepPlan pl;
    int rc = plan_step(p, st, io, reset_draws, &pl, fin_out != nullptr, phys_in != nullptr, repeat);
    const SwarmStepFinal fin = fin_out ? *fin_out : kNoFinal;
    const SwarmPhysics phys = phys_in ? *phys_in : kNoPhysics;
    if (rc) return rc;
    KP kp = make_kp(p, pl.mode);
    kp.raster = pl.raster;
    kp.filler = pl.filler;
    kp.n_stage = pl.n_stage;
    kp.dynamic = pl.dynamic;
    kp.wind_step = (io->flags & SWARM_STEP_NO_ACTION_WIND) ? 0 : 1;
    kp.fresh = (io->flags & SWARM_STEP_FRESH_NOISE) ? 1 : 0;
    const SwarmInjectedDraws dr = reset_draws ? *reset_draws : kNoDraws;
    const int has = reset_draws ? 1 : 0;
    cudaStream_t s = (cudaStream_t)stream;
    const StepKernel kernel = pl.kernel;
    const int grid = pl.grid, nt = pl.nt, nf = pl.nf, rgrid = pl.rgrid, follow_threads = pl.follow_threads;
    const size_t smem = pl.smem, follow_smem = pl.follow_smem;
    if (pl.place == RASTER_CLUSTER) {      // no PDL: a cluster launch is an ordinary dependent of its predecessor
        const ClusterShape sh = {pl.cluster, nf, nt, smem};
        return launch_cluster(kernel, sh, p->n_envs, s, "swarm_step", kp, *st, *io, dr, has, nf, fin, phys, repeat);
    }
    if (pl.place != RASTER_FOLLOW) {
        // Single-kernel shapes are launched as programmatic dependents of whatever precedes them in the stream: when that is
        // the previous step (back-to-back env steps, a captured rollout graph) its tail overlaps with this kernel's launch
        // latency and shared-memory prologue; after any other kernel it is an ordinary launch.  SWARM_B200_NO_PDL=1 opts out.
        // Measured (profiles/r02_shapes.md): it pays for latency-bound batches -- small swarms (1024 x 80: 17.8 -> 16.5 us),
        // few CTAs per SM (256 x 256: 26.6 -> 25.3) -- and costs where the batch is XU-bound per SM, because the early-placed
        // CTAs of the next step unbalance the SMs (512 x 256: 36.8 -> 40.6 us), or where persistent raster-warp CTAs fill
        // the machine anyway.
        static const bool no_pdl = env_flag("SWARM_B200_NO_PDL");
        int sms = 148;
        {
            KernelCache& c = cache();
            std::lock_guard<std::mutex> lk(c.mu);
            int dev = 0;
            if (cudaGetDevice(&dev) == cudaSuccess && c.sms.count(dev)) sms = c.sms[dev];
        }
        const bool pdl = !no_pdl && (pl.place == RASTER_WARPS ? p->n_envs <= sms
                                                               : (p->n_locusts < 160 || p->n_envs <= 2 * sms));
        if (!pdl) {
            kernel<<<grid, nt, smem, s>>>(kp, *st, *io, dr, has, nf, fin, phys, repeat);
            return check_launch("swarm_step");
        }
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3((unsigned)nt);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, kp, *st, *io, dr, has, nf, fin, phys, repeat);
        if (le != cudaSuccess) return cuda_fail(le, "swarm_step (cudaLaunchKernelEx)");
        return check_launch("swarm_step");
    }
    // Step first, follower second: if anything serialises the two launches (a profiler, CUDA_LAUNCH_BLOCKING, a
    // device that cannot co-schedule them) the step simply finishes before the follower starts and finds every
    // flag raised -- slower, never dead-locked.  Run concurrently, the follower's CTAs (higher-priority stream)
    // take the first SM slots the step's one-env CTAs free up and then trail it by one env.
    kp.publish = 1;
    int dev = 0;
    if ((rc = current_device(&dev))) return rc;
    KernelCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);          // fork, both launches and join of one call are never interleaved with another's
    SideStream& ss = c.side[std::make_pair(dev, s)];
    cudaError_t err = cudaSuccess;
    if (!ss.stream) {
        // first call on this stream; it may be inside a stream capture (the caller warmed up on another stream):
        // creating a stream / events is harmless there, so step out of the capture's API restrictions for it
        cudaStreamCaptureMode cm = cudaStreamCaptureModeRelaxed;
        cudaThreadExchangeStreamCaptureMode(&cm);
        int lo = 0, hi = 0;
        err = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (err == cudaSuccess) err = cudaStreamCreateWithPriority(&ss.stream, cudaStreamNonBlocking, hi);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming);
        cudaThreadExchangeStreamCaptureMode(&cm);
        if (err != cudaSuccess) {
            ss = SideStream();
            return cuda_fail(err, "side stream");
        }
    }
    err = cudaEventRecord(ss.fork, s);
    if (err == cudaSuccess) err = cudaStreamWaitEvent(ss.stream, ss.fork, 0);
    if (err != cudaSuccess) return cuda_fail(err, "fork");
    kernel<<<grid, nt, smem, s>>>(kp, *st, *io, dr, has, nf, fin, phys, repeat);
    if ((rc = check_launch("swarm_step"))) return rc;
    k_raster_follow<<<rgrid, follow_threads, follow_smem, ss.stream>>>(kp, st->x, st->xa, io->grid, io->positions,
                                                                        st->work + 2);
    if ((rc = check_launch("k_raster_follow"))) return rc;
    err = cudaEventRecord(ss.join, ss.stream);
    if (err == cudaSuccess) err = cudaStreamWaitEvent(s, ss.join, 0);
    if (err != cudaSuccess) return cuda_fail(err, "join");
    return check_launch("swarm_step");
}

int swarm_step(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmInjectedDraws* reset_draws,
               swarm_stream_t stream) {
    return step_launch(p, st, io, nullptr, reset_draws, stream);
}

// swarm_step_final with optional per-env physics (phys checked by the caller) and action repeat
static int step_final_launch(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                             const SwarmInjectedDraws* reset_draws, swarm_stream_t stream, const SwarmPhysics* phys,
                             const int repeat = 1) {
    if (!fin) return step_launch(p, st, io, nullptr, reset_draws, stream, phys, repeat);
    if ((fin->grid != nullptr) != (fin->positions != nullptr)) return SWARM_ERR_FLAGS;
    if (fin->grid && (!fin->x || !fin->xa || !grid_aligned(fin->grid))) return SWARM_ERR_FLAGS;
    int rc = step_launch(p, st, io, fin, reset_draws, stream, phys, repeat);
    if (rc || !fin->grid) return rc;
    // The terminal observations: the standalone rasteriser over the done envs, as an ORDINARY launch behind the step (and
    // the follower's join), so it reads fin->x / io->done only once the step grid has completed -- k_step triggers its
    // programmatic dependents early, this kernel is not one.  The next step's PDL launch then depends on this kernel
    // and waits (griddepcontrol.wait) for its completion before touching the state, done or grid.
    return rasterize_launch(p, fin->x, fin->xa, fin->grid, fin->positions, nullptr, io->done, stream);
}

int swarm_step_final(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                     const SwarmInjectedDraws* reset_draws, swarm_stream_t stream) {
    return step_final_launch(p, st, io, fin, reset_draws, stream, nullptr);
}

int swarm_step_physics(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                       const SwarmPhysics* phys, const SwarmInjectedDraws* reset_draws, swarm_stream_t stream) {
    int rc = validate(p);
    if (!rc) rc = check_physics(phys);
    return rc ? rc : step_final_launch(p, st, io, fin, reset_draws, stream, phys);
}

int swarm_step_repeat(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const SwarmStepFinal* fin,
                      const SwarmPhysics* phys, int32_t repeat, const SwarmInjectedDraws* reset_draws, swarm_stream_t stream) {
    int rc = validate(p);
    if (!rc && repeat < 1) rc = SWARM_ERR_SIZE;
    if (!rc && phys) rc = check_physics(phys);
    // repeat 1: the kernels and launches of swarm_step / swarm_step_final / swarm_step_physics
    return rc ? rc : step_final_launch(p, st, io, fin, reset_draws, stream, phys, repeat);
}

void swarm_step_host_clear(void) { host_cache().clear(); }

void swarm_debug_trace(uint64_t* device_words, int64_t n_words) {
    g_trace = reinterpret_cast<unsigned long long*>(device_words);
    g_trace_slots = device_words ? n_words / (2 * TR_PHASES) : 0;
}

int swarm_step_host(const SwarmParams* p, const SwarmState* st, const SwarmStepIO* io, const float* host_actions,
                    float* host_reward, uint8_t* host_done, float* host_grid, uint8_t* host_positions,
                    swarm_stream_t stream) {
    if (!p || !st || !io || !host_actions || !host_reward || !host_done) return SWARM_ERR_NULL;
    if ((io->flags & SWARM_STEP_ACTIONS_F64) || !io->actions_f32) return SWARM_ERR_FLAGS;
    if ((host_grid != nullptr) != (host_positions != nullptr)) return SWARM_ERR_FLAGS;
    if (host_grid && !io->grid) return SWARM_ERR_FLAGS;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t err;
    const size_t grid_bytes = (size_t)p->n_envs * p->grid_size * p->grid_size * 2 * sizeof(float);
    const size_t pos_bytes = (size_t)p->n_envs * p->n_agents * 2;
    // the observation goes back through the copy engine after the step (D2H over PCIe, ordered on the stream)
    auto obs_back = [&](cudaStream_t on) -> int {
        if (!host_grid) return SWARM_OK;
        cudaError_t e = cudaMemcpyAsync(host_grid, io->grid, grid_bytes, cudaMemcpyDeviceToHost, on);
        if (e == cudaSuccess) e = cudaMemcpyAsync(host_positions, io->positions, pos_bytes, cudaMemcpyDeviceToHost, on);
        return e == cudaSuccess ? SWARM_OK : cuda_fail(e, "D2H observation");
    };
    // Zero-copy path: with pinned host buffers the kernel itself pulls each env's 80 bytes of actions over
    // PCIe (its cp.async prefetch runs one env ahead, so the latency hides under the previous env's force
    // phase) and posts reward/done straight into host memory: no staging copies, one launch, one sync.
    float* d_act = mapped_host(const_cast<float*>(host_actions));
    float* d_rew = mapped_host(host_reward);
    uint8_t* d_done = mapped_host(host_done);
    const bool obs_pinned = !host_grid || (mapped_host(host_grid) && mapped_host(host_positions));
    if (d_act && d_rew && d_done && obs_pinned) {
        SwarmStepIO direct = *io;
        direct.actions_f32 = d_act;
        direct.reward = d_rew;
        direct.done = d_done;
        // The same call repeats every step with the same buffers: keep its launches (step kernel, and for large
        // swarms fork -> follower -> join on the side stream, then the observation copies) as ONE instantiated CUDA
        // graph per argument set.  UseNodePriority matters: the follower only runs NEXT TO the step if its kernel node
        // keeps the side stream's higher priority (with equal priorities the step's CTAs are all dispatched first:
        // 0.255 vs 0.189 ms).
        HostStepCache& hc = host_cache();
        HostStepKey key;
        memset(&key, 0, sizeof(key));
        key.p = *p; key.st = *st; key.io = direct; key.host_grid = host_grid; key.host_positions = host_positions;
        if (cudaGetDevice(&key.device) != cudaSuccess) key.device = -1;
        cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(s, &capturing);
        if (capturing == cudaStreamCaptureStatusNone && key.device >= 0) {
            HostStepCache::Entry* hit = nullptr;
            for (int i = 0; i < kHostGraphs; ++i)
                if (hc.entries[i].exec && memcmp(&hc.entries[i].key, &key, sizeof(key)) == 0) hit = &hc.entries[i];
            if (!hit) {
                HostStepCache::Entry& cached = hc.entries[hc.next_victim++ % kHostGraphs];      // round-robin replacement
                if (cached.exec) { cudaGraphExecDestroy(cached.exec); cached.exec = nullptr; }
                // one plain call first: it warms the per-kernel caches (attribute / occupancy queries are not
                // capturable) and is itself this step
                int rc = swarm_step(p, st, &direct, nullptr, stream);
                if (rc == SWARM_OK) rc = obs_back(s);
                if (rc) return rc;
                err = cudaStreamSynchronize(s);
                if (err != cudaSuccess) return cuda_fail(err, "stream sync");
                cudaStream_t cap = nullptr;
                cudaGraph_t graph = nullptr;
                bool ok = false;
                if (cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking) == cudaSuccess) {
                    if (cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                        int rc2 = swarm_step(p, st, &direct, nullptr, (swarm_stream_t)cap);
                        if (rc2 == SWARM_OK) rc2 = obs_back(cap);
                        const cudaError_t e2 = cudaStreamEndCapture(cap, &graph);
                        if (rc2 == SWARM_OK && e2 == cudaSuccess && graph &&
                            cudaGraphInstantiateWithFlags(&cached.exec, graph, cudaGraphInstantiateFlagUseNodePriority) == cudaSuccess) {
                            cached.key = key;
                            ok = true;
                        } else {
                            cached.exec = nullptr;
                        }
                        if (graph) cudaGraphDestroy(graph);
                    }
                    cudaStreamDestroy(cap);
                }
                cudaGetLastError();       // a failed capture must not poison later calls: the plain path still works
                if (!ok && !hc.capture_failure_reported) {
                    hc.capture_failure_reported = true;
                    fprintf(stderr, "libswarm_b200: swarm_step_host could not capture its launches into a CUDA graph; "
                                    "falling back to plain launches (slower, same results)\n");
                }
                return SWARM_OK;
            }
            err = cudaGraphLaunch(hit->exec, s);
            if (err != cudaSuccess) return cuda_fail(err, "cudaGraphLaunch");
            err = cudaStreamSynchronize(s);
            if (err != cudaSuccess) return cuda_fail(err, "stream sync");
            return SWARM_OK;
        }
        int rc = swarm_step(p, st, &direct, nullptr, stream);
        if (rc == SWARM_OK) rc = obs_back(s);
        if (rc) return rc;
        err = cudaStreamSynchronize(s);
        if (err != cudaSuccess) return cuda_fail(err, "stream sync");
        return SWARM_OK;
    }
    // Pageable host memory: staged copies through io->actions_f32 / io->reward / io->done.
    const size_t na = (size_t)p->n_envs * p->n_agents * 2 * sizeof(float);
    err = cudaMemcpyAsync(io->actions_f32, host_actions, na, cudaMemcpyHostToDevice, s);
    if (err != cudaSuccess) return cuda_fail(err, "H2D actions");
    int rc = swarm_step(p, st, io, nullptr, stream);
    if (rc) return rc;
    err = cudaMemcpyAsync(host_reward, io->reward, (size_t)p->n_envs * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (err != cudaSuccess) return cuda_fail(err, "D2H reward");
    err = cudaMemcpyAsync(host_done, io->done, (size_t)p->n_envs, cudaMemcpyDeviceToHost, s);
    if (err != cudaSuccess) return cuda_fail(err, "D2H done");
    if ((rc = obs_back(s))) return rc;
    err = cudaStreamSynchronize(s);
    if (err != cudaSuccess) return cuda_fail(err, "stream sync");
    return SWARM_OK;
}

int swarm_rasterize(const SwarmParams* p, const double* x, const double* xa, float* grid, uint8_t* positions,
                    double* box, swarm_stream_t stream) {
    int rc = validate(p, 0);
    if (rc) return rc;
    if (!x || !grid) return SWARM_ERR_NULL;
    if (p->n_agents > 0 && (!xa || !positions)) return SWARM_ERR_NULL;
    if (!grid_aligned(grid)) return SWARM_ERR_FLAGS;
    return rasterize_launch(p, x, xa, grid, positions, box, nullptr, stream);
}

int swarm_expand_obs(const SwarmParams* p, const float* grid, const uint8_t* positions, float* expanded,
                     swarm_stream_t stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (!grid || !positions || !expanded) return SWARM_ERR_NULL;
    if (!grid_aligned(grid)) return SWARM_ERR_FLAGS;
    const int cells = p->grid_size * p->grid_size;
    dim3 g((cells + 255) / 256, (unsigned)(p->n_envs * p->n_agents));
    if (g.y > 65535u) {
        // split the (e,a) axis over several launches to respect gridDim.y
        const int per = 65535 / p->n_agents;   // envs per launch
        for (int e0 = 0; e0 < p->n_envs; e0 += per) {
            const int ne = (p->n_envs - e0) < per ? (p->n_envs - e0) : per;
            dim3 gg((cells + 255) / 256, (unsigned)(ne * p->n_agents));
            k_expand<<<gg, 256, 0, (cudaStream_t)stream>>>(ne, p->n_agents, p->grid_size,
                reinterpret_cast<const float2*>(grid) + (size_t)e0 * cells, positions + (size_t)e0 * p->n_agents * 2,
                expanded + (size_t)e0 * p->n_agents * cells * 3);
        }
    } else {
        k_expand<<<g, 256, 0, (cudaStream_t)stream>>>(p->n_envs, p->n_agents, p->grid_size,
                                                     reinterpret_cast<const float2*>(grid), positions, expanded);
    }
    return check_launch("swarm_expand_obs");
}

}  // extern "C"

// swarm_forces' launches (PHYS: the k_forces* variants with per-env physics)
template <bool PHYS>
static int forces_launch(const SwarmParams* p, const SwarmPhysics& phys, const double* x, const double* xa, float* v,
                         float* reward, swarm_stream_t stream) {
    int rc = 0;
    if (!x || !xa || (!v && !reward)) return SWARM_ERR_NULL;
    const int mode = force_mode(p->n_locusts);
    const KP kp = make_kp(p, mode);
    cudaStream_t s = (cudaStream_t)stream;
    if (tuning_cluster(p)) {
        ClusterShape sh;
        auto go = [&](auto kernel) {
            int r = cluster_shape(p, kernel, true, &sh);
            return r ? r : launch_cluster(kernel, sh, kp.E, s, "swarm_forces", kp, x, xa, v, reward, sh.nf, phys);
        };
        if (mode == 2) return p->math_mode ? go(k_forces_cluster<2, true, PHYS>) : go(k_forces_cluster<2, false, PHYS>);
        return p->math_mode ? go(k_forces_cluster<4, true, PHYS>) : go(k_forces_cluster<4, false, PHYS>);
    }
    const size_t smem = step_smem(p, 0, 1, mode);
    const int nt = block_threads(kp.N, mode);
    if (nt > kMaxThreads) return SWARM_ERR_SIZE;
    DISPATCH_T(mode,
        if (p->math_mode) {
            if ((rc = prep(k_forces<TT, true, PHYS>, smem))) return rc;
            k_forces<TT, true, PHYS><<<kp.E, nt, smem, s>>>(kp, x, xa, v, reward, phys);
        } else {
            if ((rc = prep(k_forces<TT, false, PHYS>, smem))) return rc;
            k_forces<TT, false, PHYS><<<kp.E, nt, smem, s>>>(kp, x, xa, v, reward, phys);
        })
    return check_launch("swarm_forces");
}

extern "C" {

int swarm_forces(const SwarmParams* p, const double* x, const double* xa, float* v, float* reward,
                 swarm_stream_t stream) {
    const int rc = validate(p);
    return rc ? rc : forces_launch<false>(p, kNoPhysics, x, xa, v, reward, stream);
}

int swarm_forces_physics(const SwarmParams* p, const SwarmPhysics* phys, const double* x, const double* xa, float* v,
                         float* reward, swarm_stream_t stream) {
    int rc = validate(p);
    if (!rc) rc = check_physics(phys);
    return rc ? rc : forces_launch<true>(p, *phys, x, xa, v, reward, stream);
}

int swarm_x_update(double* x, double* v, const double* noise, int64_t n, double dt, swarm_stream_t stream) {
    if (!x || !v || !noise) return SWARM_ERR_NULL;
    if (n <= 0) return n == 0 ? SWARM_OK : SWARM_ERR_SIZE;
    k_x_update<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<double2*>(x), reinterpret_cast<double2*>(v), reinterpret_cast<const double2*>(noise), n, dt, 1);
    return check_launch("swarm_x_update");
}

int swarm_xv_cutoff(double* x, double* v, int64_t n, swarm_stream_t stream) {
    if (!x || !v) return SWARM_ERR_NULL;
    if (n <= 0) return n == 0 ? SWARM_OK : SWARM_ERR_SIZE;
    k_x_update<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<double2*>(x), reinterpret_cast<double2*>(v), nullptr, n, 0.0, 0);
    return check_launch("swarm_xv_cutoff");
}

int swarm_s_potential(const double* r, double* out, int64_t n, double F, double L, swarm_stream_t stream) {
    if (!r || !out) return SWARM_ERR_NULL;
    if (n <= 0) return n == 0 ? SWARM_OK : SWARM_ERR_SIZE;
    k_s_potential<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(r, out, n, F, L);
    return check_launch("swarm_s_potential");
}

int swarm_clip_actions(float* actions, int64_t n_rows, float max_norm, swarm_stream_t stream) {
    if (!actions) return SWARM_ERR_NULL;
    if (n_rows < 0) return SWARM_ERR_SIZE;
    if (n_rows == 0) return SWARM_OK;
    k_clip<<<(unsigned)((n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float2*>(actions), n_rows,
                                                                              max_norm);
    return check_launch("swarm_clip_actions");
}

int swarm_philox_draws(const SwarmParams* p, const SwarmState* st, double* x0, double* xa0, double* burn_actions,
                       double* agent_noise, double* particle_noise, swarm_stream_t stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (!st || !st->episode || !x0 || !xa0 || !burn_actions || !agent_noise || !particle_noise) return SWARM_ERR_NULL;
    const KP kp = make_kp(p);
    k_philox_draws<<<kp.E, 128, 0, (cudaStream_t)stream>>>(kp, *st, reinterpret_cast<double2*>(x0),
        reinterpret_cast<double2*>(xa0), reinterpret_cast<double2*>(burn_actions),
        reinterpret_cast<double2*>(agent_noise), reinterpret_cast<double2*>(particle_noise));
    return check_launch("swarm_philox_draws");
}

int swarm_philox_noise_rows(const SwarmParams* p, const SwarmState* st, int32_t row0, int32_t n_rows, double* agent_noise,
                            double* particle_noise, swarm_stream_t stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (!st || !st->episode || !agent_noise || !particle_noise) return SWARM_ERR_NULL;
    if (row0 < 0 || n_rows <= 0) return SWARM_ERR_SIZE;
    const KP kp = make_kp(p);
    const dim3 grid((unsigned)kp.E, (unsigned)(n_rows < 65535 ? n_rows : 65535));
    k_philox_noise_rows<<<grid, 128, 0, (cudaStream_t)stream>>>(kp, *st, row0, n_rows, reinterpret_cast<double2*>(agent_noise),
                                                               reinterpret_cast<double2*>(particle_noise));
    return check_launch("swarm_philox_noise_rows");
}

int swarm_philox_raw(const uint32_t* ctr, const uint32_t* key, uint32_t* out, int64_t n, swarm_stream_t stream) {
    if (!ctr || !key || !out) return SWARM_ERR_NULL;
    if (n <= 0) return n == 0 ? SWARM_OK : SWARM_ERR_SIZE;
    k_philox_raw<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4*>(ctr), reinterpret_cast<const uint2*>(key), reinterpret_cast<uint4*>(out), n);
    return check_launch("swarm_philox_raw");
}

}  // extern "C"
