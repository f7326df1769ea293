// Block-level device code of the swarm hot path (sm_100a).  A CTA works on one env at a time.  The
// FORCE group (dynamics, reward, auto-reset) and the rasteriser are kept apart so that the
// rasteriser's latency chains and HBM stores run under another env's force phase: either as a
// second warp-specialised thread group of the same persistent CTA (RASTER group, small swarms)
// or as a follower kernel on its own stream (k_raster_follow, large swarms) -- see swarm_b200.cu.
//   * an env's FP64 integrator state, its frozen noise row and its actions are prefetched
//     (cp.async) into one of two shared-memory STAGE buffers while the previous env is being
//     stepped, and stay there for the whole step (step, auto-reset burn-in and rasterise
//     never round-trip through HBM);
//   * the O(N^2) pair forces run in FP32 on an FP32 hi/lo split of the positions staged in
//     shared memory.  For N <= 512 every UNORDERED pair is evaluated once (the pair force is
//     exactly antisymmetric): a warp owns a 32-locust tile, walks the other tiles with a
//     lane rotation, keeps its own forces in registers and hands the reaction forces round
//     the warp with shuffles; reactions are combined through fixed shared-memory slots so
//     the result is bitwise reproducible.  Larger N falls back to an ordered-pair loop with
//     T targets per thread in registers and broadcast LDS.128 sources;
//   * reward is a warp-shuffle + shared-memory reduction in FP64;
//   * the occupancy grid is a shared-memory-privatised histogram with warp-aggregated
//     atomics (match.any), written out as a streaming zero fill + sparse scatter; the
//     counter table is cleaned cell by cell by the threads that scatter, never re-cleared.
//
// Everything here is __forceinline__ on purpose: the shared-memory pointers of `Smem` must
// stay in registers with a known address space (a spilled pointer turns every LDS/STS into
// a generic LD/ST).
//
// Reference semantics restated here: fed_gym/envs/multiagent.py:30-115,
// fed_gym/agents/state_processors.py:25-42 (SURVEY.md Appendix A).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/swarm_b200.h"
#include "swarm_philox.cuh"

namespace swarm {

constexpr int kSymMaxLocusts = 512;     // unordered-pair path (MODE 1) up to here
constexpr unsigned kFull = 0xffffffffu;

// Kernel-side parameter block (derived from SwarmParams on the host).
// Pair geometry is done in coordinates pre-scaled by c = log2(e):  exp(-r) = 2^(-c r), and
// d/(r + eps) is scale free if eps is scaled too, so the scaling costs nothing per pair.
struct KP {
    int E, N, A, G, n_burn, max_steps;
    double sigma, wind, dt, half_w, y_hi, cscale;
    float F, nInvL, U, Gv, eps_s;
    float ri_max;     // 2^-12 / eps_s: pairs with 1/r above it (closer than 4096 eps) take MUFU.RCP for 1/(r + eps), see inv_r_eps
    uint2 key;
    uint32_t env_off;
    int dynamic;      // k_step: draw the third and later envs of a CTA from the work queue (SwarmState::work)
    int n_stage;      // k_step: stage buffers in shared memory (2 = prefetch the CTA's next env, 1 = one env per CTA)
    int publish;      // k_step: raise work[2 + e] once env e's new state is in memory (k_raster_follow waits for it)
    int raster;       // shared-memory layout of the rasteriser: 0 none, 1 a raster GROUP with its own point buffer, 2 the force
                      // group rasterises its own env after the step (points = the stage buffer)
    int filler;       // raster == 2: one extra warp per CTA issues the TMA zero fill of the env's grid and waits for it
    int wind_step;    // 0: the step proper does not add the wind to the actions (SwarmEnv._step(add_wind=False))
    int fresh;        // k_step (SWARM_STEP_FRESH_NOISE): the step proper draws Philox row n_burn + elapsed instead of
                      // reading the frozen row
    unsigned long long* trace;   // debug (swarm_debug_trace): per-CTA phase timestamps, nullptr in production
    long long trace_slots;       // capacity of trace in records of 2 * TR_PHASES words
    // rasteriser constants the host can round exactly like numpy does
    double step_y, inv_y; // (2 HEIGHT - 0) / G and its reciprocal
    double inv_x;         // ~ G / WIDTH: only seeds the bin guess (count_le settles ties against the exact edges)
    double inv_P, inv_G, inv_N;  // correctly rounded 1/(N+A), 1/G, 1/N: exact quotients by one FMA correction (div_by_const)
};

// One STAGE buffer = what is prefetched for the step of one env (the locust noise row follows
// later, straight into Smem::nx):
//   x (N) | xa (A) | noise_a (A) | raw actions (A x 16 B) | misc (16 B: elapsed, episode)
struct Stage {
    double2* xs;            // N   locust positions (FP64 integrator state, updated in place)
    double2* as;            // A   agent positions
    double2* an;            // A   agent noise row
    unsigned char* araw;    // A x 16 B: the env's actions as they sit in HBM (f32 pair or f64 pair)
    int* misc;              // [0] = TimeLimit elapsed steps, [1] = resets so far (fresh noise only)
    double* ph;             // PHYS kernels: the env's physics row (6 doubles, behind the kernel's shared memory, see phys_rows)
};

struct Smem {
    Stage st;         // the stage buffer of the env being stepped
    double2* nx;      // N   locust noise row of the current step (unscaled)
    double2* act;     // A   actions after conversion / clipping
    double* red;      // 32  reduction scratch
    double* box;      // 2   rasteriser: mean x
    // ---- force scratch
    float4* src;      // FP32 sources (hi_x, hi_y, lo_x, lo_y), x = hi + lo to ~2^-48.
                      //   MODE 1/3: nt 32-tiles x 64 (each tile stored twice: wrap-free lane+k reads) + A agents
                      //   MODE 2/4: N locusts + A agents
    float2* slot;     // MODE 1/3: nt x nslots x 32 reaction-force partial sums
    float2* agf;      // MODE 1/3: nt x 32 agent pulls, evaluated by the finishing thread BEFORE the tile passes (off the
                      // critical path after the barrier) and added last
    // ---- rasteriser (present when the kernel rasterises)
    double2* rx;      // N+A: post-step positions handed from the force to the raster group
    int* mail;        // [0] env id handed to the raster group (-1 = no more), [1] next env grabbed from the work queue
    uint32_t* table;  // G*G packed cell counters, 16 bits per cell (two cells per word): locusts in the low
                      // bits, agents above them (kAgentShift); 32 bits per cell (locusts lo16, agents hi16)
                      // when the counts do not fit
    int* cid;         // N+A: cell written out by this point (or -1); before that, the point's y bin count
    float* lut;       // kLutL + kLutA: grid values count / N (locusts) and count / A (agents) of the small counts
    double* rred;     // 2 kMaxWarps + 2: per-warp (sum x, max |x|) of the parallel mean; then the "some point is next to an edge" flag
};

__host__ __device__ inline size_t smem_align(size_t v) { return (v + 15) & ~size_t(15); }
__host__ __device__ inline int n_tiles(int N) { return (N + 31) >> 5; }

__host__ __device__ inline size_t smem_stage_bytes(int N, int A) { return 16 * ((size_t)N + 3 * A + 1); }
__host__ __device__ inline int sym_tiles(int N, int sym);
__host__ __device__ inline size_t smem_src_bytes(int N, int A, int sym) {
    return smem_align(sizeof(float4) * (sym ? (size_t)sym_tiles(N, sym) * 64 + A : (size_t)N + A));
}
__host__ __device__ inline size_t smem_fixed_bytes(int N, int A) {
    return smem_align(sizeof(double2) * N) + smem_align(sizeof(double2) * A) + smem_align(sizeof(double) * 32) +
           smem_align(sizeof(double) * 2) + 16;
}
// 16-bit cell counters hold (locusts | agents << kAgentShift) when N < 2^kAgentShift and A < 2^(16-kAgentShift)
constexpr int kAgentShift = 11;
__host__ __device__ inline bool table_is16(int N, int A) { return N < (1 << kAgentShift) && A < (1 << (16 - kAgentShift)); }
__host__ __device__ inline size_t smem_table_bytes(int N, int A, int G) {
    return table_is16(N, A) ? smem_align(sizeof(uint16_t) * G * G) : smem_align(sizeof(uint32_t) * G * G);
}
// sym: 0 = ordered pairs (MODE 2/4), 1 = unordered, 32-wide tiles (MODE 1), 2 = unordered, 64-wide (MODE 3)
__host__ __device__ inline int sym_tiles(int N, int sym) { return sym == 2 ? 2 * ((N + 63) >> 6) : n_tiles(N); }
__host__ __device__ inline int sym_slots(int N, int sym) {
    return sym == 2 ? 1 + ((N + 63) >> 6) / 2 : 2 * (1 + n_tiles(N) / 2);      // MODE 1: two reaction streams per pass
}
__host__ __device__ inline size_t smem_slot_bytes(int N, int sym) {
    return sym ? smem_align(sizeof(float2) * sym_tiles(N, sym) * sym_slots(N, sym) * 32) : 0;
}
__host__ __device__ inline size_t smem_agf_bytes(int N, int sym) {
    return sym ? smem_align(sizeof(float2) * sym_tiles(N, sym) * 32) : 0;
}
// agf: the agent-pull buffer exists in the latency-bound SELF shape only (raster == 2), see forces_sym*_tiles
__host__ __device__ inline size_t smem_force_bytes(int N, int A, int sym, bool agf) {
    return smem_src_bytes(N, A, sym) + smem_slot_bytes(N, sym) + (agf ? smem_agf_bytes(N, sym) : 0);
}
constexpr int kMaxWarps = 32;             // threads of a rasterising group / 32, at most
constexpr int kLutL = 256, kLutA = 33;     // grid-value look-up: counts below kLutL locusts / kLutA agents per cell
__host__ __device__ inline int lut_locusts(int N) { return N + 1 < kLutL ? N + 1 : kLutL; }
__host__ __device__ inline int lut_agents(int A) { return A + 1 < kLutA ? A + 1 : kLutA; }
// raster: 0 none, 1 raster group with its own point buffer, 2 the force group rasterises (points = stage buffer)
__host__ __device__ inline size_t smem_raster_bytes(int N, int A, int G, int raster) {
    if (!raster) return 0;
    return (raster == 1 ? smem_align(sizeof(double2) * (N + A)) : 0) + smem_table_bytes(N, A, G) +
           smem_align(sizeof(int) * (N + A)) + smem_align(sizeof(float) * (lut_locusts(N) + lut_agents(A))) +
           smem_align(sizeof(double) * (2 * kMaxWarps + 2));
}
// n_stage: stage buffers (2 in the pipelined step kernel, 1 in reset/forces, 0 in the rasteriser)
__host__ __device__ inline size_t smem_bytes(int N, int A, int G, int n_stage, bool force, int raster, int sym) {
    return n_stage * smem_stage_bytes(N, A) + smem_fixed_bytes(N, A) + (force ? smem_force_bytes(N, A, sym, raster == 2) : 0) +
           smem_raster_bytes(N, A, G, raster);
}

__device__ __forceinline__ Stage stage_at(unsigned char* base, int N, int A, int b) {
    unsigned char* p = base + (size_t)b * smem_stage_bytes(N, A);
    Stage s;
    s.xs = reinterpret_cast<double2*>(p);
    s.as = s.xs + N;
    s.an = s.as + A;
    s.araw = reinterpret_cast<unsigned char*>(s.an + A);
    s.misc = reinterpret_cast<int*>(s.araw + 16 * (size_t)A);
    return s;
}

__device__ __forceinline__ Smem carve(unsigned char* base, int N, int A, int G, int n_stage, bool force, int sym,
                                      int raster) {
    Smem s;
    s.st = stage_at(base, N, A, 0);
    size_t o = (size_t)n_stage * smem_stage_bytes(N, A);
    s.nx = reinterpret_cast<double2*>(base + o);  o += smem_align(sizeof(double2) * N);
    s.act = reinterpret_cast<double2*>(base + o); o += smem_align(sizeof(double2) * A);
    s.red = reinterpret_cast<double*>(base + o);  o += smem_align(sizeof(double) * 32);
    s.box = reinterpret_cast<double*>(base + o);  o += smem_align(sizeof(double) * 2);
    s.mail = reinterpret_cast<int*>(base + o);    o += 16;
    s.src = reinterpret_cast<float4*>(base + o);
    s.slot = reinterpret_cast<float2*>(base + o + smem_src_bytes(N, A, sym));
    s.agf = reinterpret_cast<float2*>(base + o + smem_src_bytes(N, A, sym) + smem_slot_bytes(N, sym));
    if (force) o += smem_force_bytes(N, A, sym, raster == 2);
    s.rx = reinterpret_cast<double2*>(base + o);
    if (raster == 1) o += smem_align(sizeof(double2) * (N + A));
    s.table = reinterpret_cast<uint32_t*>(base + o); o += smem_table_bytes(N, A, G);
    s.cid = reinterpret_cast<int*>(base + o);       o += smem_align(sizeof(int) * (N + A));
    s.lut = reinterpret_cast<float*>(base + o);     o += smem_align(sizeof(float) * (lut_locusts(N) + lut_agents(A)));
    s.rred = reinterpret_cast<double*>(base + o);
    return s;
}

// ------------------------------------------------------------------------------------------
// Debug timeline (swarm_debug_trace; only in a library built with -DSWARM_TRACE, see scripts/build_variants.py): record
// `rec` holds, for phase ph < 16, the global timer (ns) in word 2 ph and the SM's cycle counter in word 2 ph + 1.
enum : int { TR_ENTRY = 0, TR_ZFILL = 1, TR_LOADED = 2, TR_STAGED = 3, TR_TILES = 4, TR_FORCES = 5, TR_STEPPED = 6, TR_STORED = 7,
             TR_RASTER = 8, TR_MEAN = 9, TR_BINNED = 10, TR_ZEROS = 11, TR_DONE = 12, TR_PHASES = 16 };
__device__ __forceinline__ void trace_mark(const KP& kp, const long long rec, const int ph) {
#ifndef SWARM_TRACE
    (void)kp; (void)rec; (void)ph;      // compiled out of the production library: the hooks cost 0.5-2.5 % (measured)
#else
    if (kp.trace != nullptr && rec >= 0 && rec < kp.trace_slots) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        kp.trace[rec * 2 * TR_PHASES + 2 * ph] = t;
        kp.trace[rec * 2 * TR_PHASES + 2 * ph + 1] = (unsigned long long)clock64();
    }
#endif
}

// ------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may
// start while its predecessor in the stream is still running; pdl_wait() blocks until every prerequisite grid has
// completed and its memory is visible (a no-op for ordinary launches), pdl_launch_dependents() lets the successor's
// CTAs be scheduled from now on (they then sit in pdl_wait()).  Used by the single-kernel step shapes: the successor's
// launch latency and shared-memory prologue overlap with the predecessor's tail.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// cp.async (LDGSTS): HBM -> shared memory without staging through registers
template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gmem_src) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(d), "l"(gmem_src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// all but the most recently committed group have landed
__device__ __forceinline__ void cp_async_wait_but_one() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// multiagent.py:70-86  x_update = cutoff; x += dt*v + noise; cutoff   (FP64, no FMA contraction
// so that an injected v reproduces the reference's three roundings exactly)
__device__ __forceinline__ void move_particle(double2& p, double2 v, double2 n, double dt, double sigma) {
    if (p.y <= 0.0) {
        p.y = 0.0;
        v.x = 0.0;
        if (v.y <= 0.0) v.y = 0.0;
    }
    p.x = __dadd_rn(p.x, __dadd_rn(__dmul_rn(dt, v.x), __dmul_rn(sigma, n.x)));
    p.y = __dadd_rn(p.y, __dadd_rn(__dmul_rn(dt, v.y), __dmul_rn(sigma, n.y)));
    if (p.y <= 0.0) p.y = 0.0;
}

// ------------------------------------------------------------------------------------------
// Per-env physics (SwarmPhysics; the PHYS kernel instantiations).  A row is {noise, gravity, wind, F, L, dt} in
// SwarmParams' order.  The PHYS kernels keep the row of each stage buffer in kPhysRowBytes behind the kernel's own shared
// memory (so every other offset stays put) and take the env's constants from it with make_kp's roundings: a row equal to
// SwarmParams gives the bits of the launch constants.
constexpr int kPhysCols = 6;
constexpr size_t kPhysRowBytes = sizeof(double) * kPhysCols;     // 48: three 16-byte cp.async pieces

// kp with the constants of row ph (F and -1/L: make_kp's roundings; -1.0 / L == -RN(1 / L) exactly)
__device__ __forceinline__ KP phys_kp(const KP& kp, const double* ph) {
    KP k = kp;
    k.sigma = ph[0];
    k.wind = ph[2];
    k.dt = ph[5];
    k.Gv = (float)ph[1];
    k.U = (float)ph[2];
    k.F = (float)ph[3];
    k.nInvL = (float)(-__drcp_rn(ph[4]));
    return k;
}

// Column c of a SWARM_PHYSICS_RESAMPLE row: lo + (hi - lo) u, u from Philox stream 5 of the reset's DrawCtx.  The bounds
// are picked with constant indices: a thread-dependent index into the kernel parameter would copy lo / hi to local memory.
__device__ __forceinline__ double phys_draw(const DrawCtx& d, const SwarmPhysics& P, const int c) {
    const double2 u = draw_uniform2(d, STREAM_PHYSICS, (uint32_t)(c >> 1));
    double lo = P.lo[0], hi = P.hi[0];
#pragma unroll
    for (int i = 1; i < kPhysCols; ++i) {
        if (c == i) {
            lo = P.lo[i];
            hi = P.hi[i];
        }
    }
    return __dadd_rn(lo, __dmul_rn(__dadd_rn(hi, -lo), (c & 1) ? u.y : u.x));
}

// The row of env e's new episode into row (shared memory), by threads tid < 6: with SWARM_PHYSICS_RESAMPLE drawn (and
// written back to the table when `store`), else the table's.  Visible to the other threads after their next barrier.
__device__ __forceinline__ void phys_reset_row(double* row, const SwarmPhysics& P, const KP& kp, const int e,
                                               const uint32_t episode, const int tid, const bool store) {
    if (tid < kPhysCols) {
        double v;
        if (P.flags & SWARM_PHYSICS_RESAMPLE) {
            DrawCtx d;
            d.key = kp.key;
            d.env = kp.env_off + (uint32_t)e;
            d.episode = episode;
            v = phys_draw(d, P, tid);
            if (store) P.table[(size_t)e * kPhysCols + tid] = v;
        } else {
            v = P.table[(size_t)e * kPhysCols + tid];
        }
        row[tid] = v;
    }
}

// Named barriers (bar.sync id, n) of the warp-specialised step kernel.  0 stays __syncthreads.
enum : int { BAR_FORCE = 1, BAR_RASTER = 2, BAR_FULL = 3, BAR_EMPTY = 4, BAR_ZREAD = 5, BAR_ZDONE = 6 };

template <int ID>
__device__ __forceinline__ void bar_sync(int n) { asm volatile("bar.sync %0, %1;" ::"n"(ID), "r"(n) : "memory"); }
template <int ID>
__device__ __forceinline__ void bar_arrive(int n) { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "r"(n) : "memory"); }

// A group of whole warps that cooperates on one env: tid in [0,n), n a multiple of 32.
template <int BAR>
struct GrpT {
    int tid;
    int n;
    __device__ __forceinline__ void sync() const { bar_sync<BAR>(n); }
};
typedef GrpT<BAR_FORCE> Grp;     // dynamics
typedef GrpT<BAR_RASTER> RGrp;   // rasteriser

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// a / b for a divisor whose correctly rounded reciprocal inv_b = RN(1 / b) the host supplies: q0 = RN(a inv_b) is within
// one ulp, the FMA residual r = a - q0 b is exact and RN(q0 + r inv_b) is the correctly rounded quotient (Markstein
// 1990) -- three FP64 operations instead of the ~40-instruction division routine.  Outside the range where the
// residual is exact (quotients near the subnormals / overflow) the plain division is used.
__device__ __forceinline__ double div_by_const(const double a, const double b, const double inv_b) {
    const double m = fabs(a);
    if (!(m > 1e-280 && m < 1e280)) return a / b;
    const double q0 = __dmul_rn(a, inv_b);
    const double r = __fma_rn(-q0, b, a);
    return __fma_rn(r, inv_b, q0);
}

// ------------------------------------------------------------------------------------------
// Pair weight, multiagent.py:65-68,100-113:  w = s(r)/(r+eps), s(r) = F exp(-r/L) - exp(-r),
// in log2(e)-scaled coordinates:  w = (F 2^(-r/L) - 2^(-r)) / (r + c eps).
// Positions arrive as FP32 hi/lo pairs of the FP64 state, so the difference
//   d = (hi_i - hi_j) + (lo_i - lo_j)
// carries ~2^-24 RELATIVE error of the difference of the two REPRESENTED points however close they
// are (plain FP32 positions lose the direction of close pairs, where s/(r+eps) is steepest).  hi + lo
// itself represents a coordinate only to ~2^-48 |x|, so d is also off by up to ~2^-47 (|x_i| + |x_j|)
// absolutely: nothing near the origin, where TimeLimit episodes stay, but up to ~6e-6 in a close
// pair's force at |x| ~ 1e4 (envelope: DESIGN 3.1).  Coincident points (and the
// self pair of the ordered loop) have d = 0 exactly and contribute exactly 0.
// 1 / (r + eps) from rinv ~ 1/r without a third trip to the XU pipe (the busiest pipe of the pair loop):
//   1/(r + eps) = rinv / (1 + eps rinv) = rinv - (eps rinv) rinv + O((eps/r)^2),
// one FMUL + one FFMA.  The dropped term is below 2^-24 -- the rounding of the result -- when eps rinv <= 2^-12, i.e. for
// every pair further apart than 4096 eps (0.004 in the reference's units); closer pairs (a dense swarm of 256 holds 5-25
// of them at any time) take MUFU.RCP as before.  Which of the two a pair gets depends on the pair alone, so every tiling
// and launch shape still produces the same bits.  Used by the unordered-pair modes (MODE 3: k_forces 144 -> 124 us at
// 4096 x 256; MODE 1: 1-2 %); the ordered modes (N > 512) keep the MUFU.
#ifndef SWARM_RCP_SERIES
#define SWARM_RCP_SERIES 1
#endif
template <bool SERIES>
__device__ __forceinline__ float inv_r_eps(const float r, const float rinv, const float eps_s, const float ri_max) {
    float inv;
    if constexpr (SERIES && SWARM_RCP_SERIES) {
        inv = fmaf(-eps_s * rinv, rinv, rinv);
        if (rinv > ri_max) asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(r + eps_s));
    } else {
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(r + eps_s));
    }
    return inv;
}

template <bool PRECISE, bool SERIES = false>
__device__ __forceinline__ float pair_weight(const float dx, const float dy, const KP& kp) {
    if (PRECISE) {
        const float r = __fsqrt_rn(__fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
        const float s = __fmaf_rn(kp.F, exp2f(__fmul_rn(r, kp.nInvL)), -exp2f(-r));
        return __fdiv_rn(s, __fadd_rn(r, kp.eps_s));
    } else {
        // r2 >= 1e-30 keeps rsqrt finite for coincident points (their dx,dy are 0 anyway)
        const float r2 = fmaf(dx, dx, fmaf(dy, dy, 1e-30f));
        float rinv, e1, e2, inv;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rinv) : "f"(r2));
        const float r = r2 * rinv;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-r));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2) : "f"(r * kp.nInvL));
        const float s = fmaf(kp.F, e2, -e1);
        inv = inv_r_eps<SERIES>(r, rinv, kp.eps_s, kp.ri_max);
        return s * inv;
    }
}

// ordered pair: force of source q on target tg
template <bool PRECISE>
__device__ __forceinline__ void pair_ordered(const float4 q, const float4 tg, const KP& kp, float& ax, float& ay) {
    const float dx = (q.x - tg.x) + (q.z - tg.z);
    const float dy = (q.y - tg.y) + (q.w - tg.w);
    const float w = pair_weight<PRECISE>(dx, dy, kp);
    ax = fmaf(w, dx, ax);
    ay = fmaf(w, dy, ay);
}

__device__ __forceinline__ float4 split_hilo(const double2 p, const double c) {
    const double sx = p.x * c, sy = p.y * c;
    const float hx = (float)sx, hy = (float)sy;
    return make_float4(hx, hy, (float)(sx - (double)hx), (float)(sy - (double)hy));
}

// MODE: 1 = unordered pairs, a warp owns a 32-locust tile, 1 target per lane
//       3 = unordered pairs, a warp owns a 64-locust super-tile, 2 targets per lane (half the
//           shared-memory loads and shuffles per pair; used when N pads to 64 as well as to 32)
//       2/4 = ordered pairs, 2/4 targets per thread (N > 512)
template <int MODE>
struct ModeT {
    static constexpr int T = MODE == 1 ? 1 : (MODE == 3 ? 2 : MODE);
    static constexpr int SYM = MODE == 1 ? 1 : (MODE == 3 ? 2 : 0);
};

// locust owned by thread g.tid as its t-th target
template <int MODE>
__device__ __forceinline__ int target_index(const Grp& g, int t, const KP&) {
    return MODE == 3 ? ((g.tid >> 5) * 64 + t * 32 + (g.tid & 31)) : g.tid + t * g.n;
}

template <int MODE>
__device__ __forceinline__ float4* agent_sources(const Smem& sm, const KP& kp) {
    return sm.src + (ModeT<MODE>::SYM ? sym_tiles(kp.N, ModeT<MODE>::SYM) * 64 : kp.N);
}

// Stage the scaled FP32 hi/lo sources of the locusts.  Thread j stages element j.
template <int MODE>
__device__ __forceinline__ void stage_locusts(const Smem& sm, const KP& kp, const Grp& g) {
    const int N = kp.N;
    if (ModeT<MODE>::SYM) {
        const int nt = sym_tiles(N, ModeT<MODE>::SYM);
        // pad lanes sit far away: as sources they contribute exactly 0 (both exponentials underflow)
        // (and 1e12 from one another: a pad-pad pair must not look like a close pair to inv_r_eps)
        for (int j = g.tid; j < nt * 32; j += g.n) {
            const float4 q = j < N ? split_hilo(sm.st.xs[j], kp.cscale) : make_float4(1e15f + 1e12f * (float)(j - N), 0.f, 0.f, 0.f);
            float4* t = sm.src + (j >> 5) * 64 + (j & 31);
            t[0] = q;
            t[32] = q;
        }
    } else {
        for (int i = g.tid; i < N; i += g.n) sm.src[i] = split_hilo(sm.st.xs[i], kp.cscale);
    }
}

#ifndef SWARM_TILE_UNROLL
#define SWARM_TILE_UNROLL 4
#endif
constexpr int kTileUnroll = SWARM_TILE_UNROLL;   // rotation steps unrolled together (x targets per lane = pair chains in flight)

// one unordered pair: force of source q on target tg, and (REACT) its reaction on the source
template <bool REACT, bool PRECISE, bool SERIES = false>
__device__ __forceinline__ void pair_sym(const float4 q, const float4 tg, const KP& kp, float& ax, float& ay,
                                         float& bx, float& by) {
    const float dx = (q.x - tg.x) + (q.z - tg.z);
    const float dy = (q.y - tg.y) + (q.w - tg.w);
    const float w = pair_weight<PRECISE, SERIES>(dx, dy, kp);
    ax = fmaf(w, dx, ax);
    ay = fmaf(w, dy, ay);
    if (REACT) {
        bx = fmaf(-w, dx, bx);
        by = fmaf(-w, dy, by);
    }
}


// ---- packed FP32 pairs (sm_100 FADD2 / FMUL2 / FFMA2): one issue slot, two FP32 results ------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

struct PairConst2 {
    f32x2 nInvL2, nF2, neps2;
    float ri_max;
};
__device__ __forceinline__ PairConst2 make_pair_const2(const KP& kp) {
    PairConst2 c;
    c.nInvL2 = pk2(kp.nInvL, kp.nInvL);
    c.nF2 = pk2(-kp.F, -kp.F);
    c.neps2 = pk2(-kp.eps_s, -kp.eps_s);
    c.ri_max = kp.ri_max;
    return c;
}

// inv_r_eps for two pairs at once: the same roundings, packed; the close-pair test is one FMNMX + FSETP for both.
template <bool SERIES>
__device__ __forceinline__ f32x2 inv_r_eps2(const f32x2 r, const float riA, const float riB, const PairConst2& c) {
  if constexpr (SERIES && SWARM_RCP_SERIES) {
    const f32x2 ri = pk2(riA, riB);
    f32x2 inv = fma2(mul2(c.neps2, ri), ri, ri);
    // (warp-uniform test: a plain branch, no reconvergence point in the pair loop -- 2 % faster than the divergent form;
    // every caller runs with all 32 lanes)
    if (__any_sync(kFull, fmaxf(riA, riB) > c.ri_max)) {
        float rA, rB, iA, iB, ne, ne_;
        upk2(r, rA, rB);
        upk2(inv, iA, iB);
        upk2(c.neps2, ne, ne_);
        if (riA > c.ri_max) asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iA) : "f"(rA - ne));
        if (riB > c.ri_max) asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iB) : "f"(rB - ne));
        inv = pk2(iA, iB);
    }
    return inv;
  } else {
    float pA, pB, iA, iB, ne, ne_;
    upk2(r, pA, pB);
    upk2(c.neps2, ne, ne_);
    pA -= ne; pB -= ne;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iA) : "f"(pA));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iB) : "f"(pB));
    return pk2(iA, iB);
  }
}


// n2 rotation steps of one tile pass with TWO sources per step: the lane meets tl1[k] (stream 1) and tl2[k] (stream 2;
// the same doubled tile, 8 or 16 elements further on, so tl[k] never needs wrap logic).  The own force accumulates in
// (ax,ay) -- stream 1 first, then stream 2; (b1, b2) are the reactions on the two met elements and move one lane down
// BEFORE every step (also before the first one: they then carry zeros, or the caller's partial sum), so that each follows
// its element.  On return lane l holds the reactions for the two elements met last.  Fast math packs the two pairs into
// FADD2 / FMUL2 / FFMA2 (geometry by component, the r -> w chain across the two sources); MUFU stays scalar.
template <bool PRECISE>
__device__ __forceinline__ void tile_sym_dual(const float4* __restrict__ tl1, const float4* __restrict__ tl2, const int n2,
                                              const float4 tg, const KP& kp, const int nxt, float& ax, float& ay,
                                              float& b1x, float& b1y, float& b2x, float& b2y) {
    if constexpr (PRECISE) {
#pragma unroll 2
        for (int k = 0; k < n2; ++k) {
            b1x = __shfl_sync(kFull, b1x, nxt); b1y = __shfl_sync(kFull, b1y, nxt);
            b2x = __shfl_sync(kFull, b2x, nxt); b2y = __shfl_sync(kFull, b2y, nxt);
            const float4 q1 = tl1[k], q2 = tl2[k];
            {
                const float dx = (q1.x - tg.x) + (q1.z - tg.z), dy = (q1.y - tg.y) + (q1.w - tg.w);
                const float w = pair_weight<PRECISE>(dx, dy, kp);
                ax = fmaf(w, dx, ax); ay = fmaf(w, dy, ay);
                b1x = fmaf(-w, dx, b1x); b1y = fmaf(-w, dy, b1y);
            }
            {
                const float dx = (q2.x - tg.x) + (q2.z - tg.z), dy = (q2.y - tg.y) + (q2.w - tg.w);
                const float w = pair_weight<PRECISE>(dx, dy, kp);
                ax = fmaf(w, dx, ax); ay = fmaf(w, dy, ay);
                b2x = fmaf(-w, dx, b2x); b2y = fmaf(-w, dy, b2y);
            }
        }
    } else {
        const f32x2 nh = pk2(-tg.x, -tg.y), nl = pk2(-tg.z, -tg.w);
        const PairConst2 c = make_pair_const2(kp);
        f32x2 na = pk2(-ax, -ay);
#pragma unroll kTileUnroll
        for (int k = 0; k < n2; ++k) {
            b1x = __shfl_sync(kFull, b1x, nxt); b1y = __shfl_sync(kFull, b1y, nxt);
            b2x = __shfl_sync(kFull, b2x, nxt); b2y = __shfl_sync(kFull, b2y, nxt);
            const float4 q1 = tl1[k], q2 = tl2[k];
            const f32x2 d1 = add2(add2(pk2(q1.x, q1.y), nh), add2(pk2(q1.z, q1.w), nl));
            const f32x2 d2 = add2(add2(pk2(q2.x, q2.y), nh), add2(pk2(q2.z, q2.w), nl));
            float d1x, d1y, d2x, d2y;
            upk2(d1, d1x, d1y);
            upk2(d2, d2x, d2y);
            // r2 >= 1e-30 keeps rsqrt finite for coincident points (their d is 0 anyway)
            const float r2a = fmaf(d1x, d1x, fmaf(d1y, d1y, 1e-30f));
            const float r2b = fmaf(d2x, d2x, fmaf(d2y, d2y, 1e-30f));
            float ria, rib;
            asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(ria) : "f"(r2a));
            asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rib) : "f"(r2b));
            const f32x2 r = mul2(pk2(r2a, r2b), pk2(ria, rib));
            const f32x2 arg = mul2(r, c.nInvL2);
            float ra, rb, ga, gb;
            upk2(r, ra, rb);
            upk2(arg, ga, gb);
            float e1a, e1b, e2a, e2b;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1a) : "f"(-ra));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1b) : "f"(-rb));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2a) : "f"(ga));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2b) : "f"(gb));
            const f32x2 ns = fma2(c.nF2, pk2(e2a, e2b), pk2(e1a, e1b));    // -(F e2 - e1)
            const f32x2 nw = mul2(ns, inv_r_eps2<true>(r, ria, rib, c));   // (-w_1, -w_2)
            float nwa, nwb;
            upk2(nw, nwa, nwb);
            const f32x2 nwa2 = pk2(nwa, nwa), nwb2 = pk2(nwb, nwb);
            na = fma2(nwa2, d1, na);
            na = fma2(nwb2, d2, na);
            f32x2 b1 = fma2(nwa2, d1, pk2(b1x, b1y)), b2 = fma2(nwb2, d2, pk2(b2x, b2y));
            upk2(b1, b1x, b1y);
            upk2(b2, b2x, b2y);
        }
        upk2(na, ax, ay);
        ax = -ax; ay = -ay;
    }
}

// MODE 1, part 1: all locust-locust pairs once.  Thread = locust j (tile I = warp, lane).  Tile I
// meets itself (lane offsets 1..15 with reaction, offset 16 one way: each such pair appears in two
// lanes, offset 0 = self), tiles I+1..I+floor((nt-1)/2) fully and tile I+nt/2 (nt even) half each
// way.  Every pass walks its offsets as TWO streams, half a pass apart (tile_sym_dual): 16 + 16 offsets of a full
// tile, 8 + 8 of a half tile, and in the own tile 1..7 next to 9..15 with offset 8 taken first by stream 2 alone.
// One loop over the passes, so the pair code exists once.  The two reaction sums of a pass land in sm.slot; the
// caller must barrier before forces_sym_finish.
template <bool PRECISE, bool AGF>
__device__ __forceinline__ void forces_sym_tiles(const Smem& sm, const KP& kp, const Grp& g, float& ax, float& ay) {
    const int lane = g.tid & 31, I = g.tid >> 5;
    const int nt = n_tiles(kp.N), nslots = 1 + nt / 2;
    const int nxt = (lane + 1) & 31;
    const int nfull = (nt - 1) >> 1;
    const float4* S = sm.src;
    const float4 tg = S[I * 64 + lane];
    if constexpr (AGF) {   // the agents' pull on this lane's locust (multiagent.py:108-113), summed from 0, added last in the finish
        const float4* ag = S + nt * 64;
        float gx = 0.f, gy = 0.f;
#pragma unroll 2
        for (int k = 0; k < kp.A; ++k) pair_ordered<PRECISE>(ag[k], tg, kp, gx, gy);
        sm.agf[I * 32 + lane] = make_float2(gx, gy);
    }
    ax = 0.f;
    ay = 0.f;
    pair_ordered<PRECISE>(S[I * 64 + lane + 16], tg, kp, ax, ay);
#pragma unroll 1
    for (int o = 0; o < nslots; ++o) {
        int B = I, first = 1, n2 = 7, gap = 8;           // own tile: offsets 1..7 | 9..15 (8 below)
        if (o > 0) {
            if (o <= nfull) {                            // a full tile pair: offsets 0..15 | 16..31
                B = I + o;
                if (B >= nt) B -= nt;
                first = 0;
                n2 = 16;
                gap = 16;
            } else {   // lane offsets 0..15 from the lower tile, 16..31 (= 1..16 seen from the partner) from the upper
                B = I < o ? I + o : I - o;
                first = I < o ? 0 : 1;
                n2 = 8;
                gap = 8;
            }
        }
        const float4* tl = S + B * 64 + lane + first;
        float b1x = 0.f, b1y = 0.f, b2x = 0.f, b2y = 0.f;
        if (o == 0) {     // own tile, offset 8: stream 2's first element (lanes are whole here: b2 is still zero everywhere)
            pair_sym<true, PRECISE>(tl[7], tg, kp, ax, ay, b2x, b2y);
        }
        tile_sym_dual<PRECISE>(tl, tl + gap, n2, tg, kp, nxt, ax, ay, b1x, b1y, b2x, b2y);
        float2* sl = sm.slot + (size_t)((B * nslots + o) * 2) * 32;
        sl[(lane + first + n2 - 1) & 31] = make_float2(b1x, b1y);
        sl[32 + ((lane + first + gap + n2 - 1) & 31)] = make_float2(b2x, b2y);
    }
}

// MODE 1, part 2: add the reactions (fixed order: bitwise reproducible) and the agents' pull.
template <bool PRECISE, bool AGF>
__device__ __forceinline__ void forces_sym_finish(const Smem& sm, const KP& kp, const Grp& g, float& ax, float& ay) {
    const int lane = g.tid & 31, I = g.tid >> 5;
    const int nt = n_tiles(kp.N), nslots = 1 + nt / 2;
    for (int o = 0; o < nslots; ++o) {
        const float2* sl = sm.slot + (size_t)((I * nslots + o) * 2) * 32;
        const float2 r1 = sl[lane], r2 = sl[32 + lane];
        ax += r1.x;
        ay += r1.y;
        ax += r2.x;
        ay += r2.y;
    }
    // the agents' pull, summed from 0 and added last: either evaluated before the tile passes (AGF: the latency-bound
    // shape, where this keeps it off the critical path behind the barrier) or here -- the same bits either way
    if constexpr (AGF) {
        const float2 a = sm.agf[I * 32 + lane];     // written by this very thread in forces_sym_tiles
        ax += a.x;
        ay += a.y;
    } else {
        const float4 tg = sm.src[I * 64 + lane];
        const float4* ag = sm.src + nt * 64;
        float gx = 0.f, gy = 0.f;
#pragma unroll 2
        for (int k = 0; k < kp.A; ++k) pair_ordered<PRECISE>(ag[k], tg, kp, gx, gy);
        ax += gx;
        ay += gy;
    }
}

// ---- MODE 3: 64-wide super-tiles, two targets (A: first half, B: second half) per lane -------
// Two targets of one lane, negated and split like the sources: d = (q.hi + nh) + (q.lo + nl).
struct Targets2 {
    f32x2 nhA, nlA, nhB, nlB;
};
__device__ __forceinline__ Targets2 make_targets2(const float4 tgA, const float4 tgB) {
    Targets2 t;
    t.nhA = pk2(-tgA.x, -tgA.y); t.nlA = pk2(-tgA.z, -tgA.w);
    t.nhB = pk2(-tgB.x, -tgB.y); t.nlB = pk2(-tgB.z, -tgB.w);
    return t;
}
// One source q against both targets of the lane, fast math.  The geometry is packed by component
// (x,y), the scalar chain r -> w by target (A,B); MUFU stays scalar.  Accumulates the NEGATED
// forces: naX += -w_X d_X (X = A, B) and, with REACT, the reaction b += -(w_A d_A + w_B d_B).
// Operation for operation the same roundings as pair_sym<.., false> (negation is exact).
template <bool REACT>
__device__ __forceinline__ void pair2_fast(const float4 q, const Targets2& t, const PairConst2& c, f32x2& naA, f32x2& naB,
                                           f32x2& b) {
    const f32x2 qh = pk2(q.x, q.y), ql = pk2(q.z, q.w);
    const f32x2 dA = add2(add2(qh, t.nhA), add2(ql, t.nlA));
    const f32x2 dB = add2(add2(qh, t.nhB), add2(ql, t.nlB));
    float dAx, dAy, dBx, dBy;
    upk2(dA, dAx, dAy);
    upk2(dB, dBx, dBy);
    // r2 >= 1e-30 keeps rsqrt finite for coincident points (their d is 0 anyway)
    const float r2A = fmaf(dAx, dAx, fmaf(dAy, dAy, 1e-30f));
    const float r2B = fmaf(dBx, dBx, fmaf(dBy, dBy, 1e-30f));
    float riA, riB;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(riA) : "f"(r2A));
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(riB) : "f"(r2B));
    const f32x2 r = mul2(pk2(r2A, r2B), pk2(riA, riB));
    const f32x2 arg = mul2(r, c.nInvL2);
    float rA, rB, gA, gB;
    upk2(r, rA, rB);
    upk2(arg, gA, gB);
    float e1A, e1B, e2A, e2B;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1A) : "f"(-rA));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1B) : "f"(-rB));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2A) : "f"(gA));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2B) : "f"(gB));
    const f32x2 ns = fma2(c.nF2, pk2(e2A, e2B), pk2(e1A, e1B));      // -(F e2 - e1)
    const f32x2 nw = mul2(ns, inv_r_eps2<true>(r, riA, riB, c));     // (-w_A, -w_B)
    float nwA, nwB;
    upk2(nw, nwA, nwB);
    const f32x2 nwA2 = pk2(nwA, nwA), nwB2 = pk2(nwB, nwB);
    naA = fma2(nwA2, dA, naA);
    naB = fma2(nwB2, dB, naB);
    if (REACT) {
        b = fma2(nwA2, dA, b);
        b = fma2(nwB2, dB, b);
    }
}

// n rotation steps of one half-tile pass with both targets (see tile_sym for the conventions).
template <bool PRECISE>
__device__ __forceinline__ void tile_sym2(const float4* __restrict__ tl, const int n, const float4 tgA, const float4 tgB,
                                          const KP& kp, const int nxt, float& aAx, float& aAy, float& aBx, float& aBy,
                                          float& bx, float& by) {
    if constexpr (PRECISE) {
#pragma unroll kTileUnroll
        for (int k = 0; k < n; ++k) {
            bx = __shfl_sync(kFull, bx, nxt);
            by = __shfl_sync(kFull, by, nxt);
            const float4 q = tl[k];
            pair_sym<true, PRECISE>(q, tgA, kp, aAx, aAy, bx, by);
            pair_sym<true, PRECISE>(q, tgB, kp, aBx, aBy, bx, by);
        }
    } else {
        const Targets2 t = make_targets2(tgA, tgB);
        const PairConst2 c = make_pair_const2(kp);
        f32x2 naA = pk2(-aAx, -aAy), naB = pk2(-aBx, -aBy);
#pragma unroll kTileUnroll
        for (int k = 0; k < n; ++k) {
            bx = __shfl_sync(kFull, bx, nxt);
            by = __shfl_sync(kFull, by, nxt);
            f32x2 b = pk2(bx, by);
            pair2_fast<true>(tl[k], t, c, naA, naB, b);
            upk2(b, bx, by);
        }
        upk2(naA, aAx, aAy);
        upk2(naB, aBx, aBy);
        aAx = -aAx; aAy = -aAy; aBx = -aBx; aBy = -aBy;
    }
}

// MODE 3, part 1.  Warp I owns super-tile I = half-tiles 2I (A targets) and 2I+1 (B targets).
// Passes (one loop, so the pair code exists once):
//   p = 0  own A half as sources: offset 0 (B target only: the A x B block is split by offset, (B target,
//          A source) takes 0..15), offsets 1..15 both targets, offset 16 A target one way;
//   p = 1  own B half as sources: offsets 1..15 both targets, offset 16 A target ((A target, B source)
//          takes 1..16) with reaction + B target one way;
//   then   super-tiles I+1 .. I+floor((nt2-1)/2): both halves, all 32 offsets;
//          super-tile I+nt2/2 (nt2 even): both halves, half the offsets each way.
// AGF: the agents' pull on the lane's two targets is evaluated first and parked in sm.agf (see forces_sym64_finish).
template <bool PRECISE, bool AGF>
__device__ __forceinline__ void forces_sym64_tiles(const Smem& sm, const KP& kp, const Grp& g, float (&vx)[2],
                                                   float (&vy)[2]) {
    const int lane = g.tid & 31, I = g.tid >> 5;
    const int nt2 = (kp.N + 63) >> 6, nslots = 1 + nt2 / 2;
    const int nxt = (lane + 1) & 31;
    const int nfull = (nt2 - 1) >> 1;
    const int npass = 2 * nslots;
    const float4* S = sm.src;
    const float4 tgA = S[(2 * I) * 64 + lane], tgB = S[(2 * I + 1) * 64 + lane];
    if constexpr (AGF) {
        const float4* ag = S + nt2 * 128;
        float gAx = 0.f, gAy = 0.f, gBx = 0.f, gBy = 0.f;
        if constexpr (PRECISE) {
            for (int k = 0; k < kp.A; ++k) {
                const float4 q = ag[k];
                pair_ordered<PRECISE>(q, tgA, kp, gAx, gAy);
                pair_ordered<PRECISE>(q, tgB, kp, gBx, gBy);
            }
        } else {
            const Targets2 t = make_targets2(tgA, tgB);
            const PairConst2 c = make_pair_const2(kp);
            f32x2 naA = 0, naB = 0, b = 0;
#pragma unroll 2
            for (int k = 0; k < kp.A; ++k) pair2_fast<false>(ag[k], t, c, naA, naB, b);
            upk2(naA, gAx, gAy);
            upk2(naB, gBx, gBy);
            gAx = -gAx; gAy = -gAy; gBx = -gBx; gBy = -gBy;
        }
        sm.agf[(2 * I) * 32 + lane] = make_float2(gAx, gAy);
        sm.agf[(2 * I + 1) * 32 + lane] = make_float2(gBx, gBy);
    }
    float aAx = 0.f, aAy = 0.f, aBx = 0.f, aBy = 0.f;
#pragma unroll 1
    for (int p = 0; p < npass; ++p) {
        const int o = p >> 1, h = p & 1;
        int J = I, first = 1, n = 15;
        if (o > 0) {
            if (o <= nfull) {
                J = I + o;
                if (J >= nt2) J -= nt2;
                first = 0;
                n = 32;
            } else {
                J = I < o ? I + o : I - o;
                first = I < o ? 0 : 1;
                n = 16;
            }
        }
        const int H = 2 * J + h;
        const float4* tl = S + H * 64 + lane;
        float bx = 0.f, by = 0.f;
        if (p == 0) pair_sym<true, PRECISE, true>(tl[0], tgB, kp, aBx, aBy, bx, by);
        tile_sym2<PRECISE>(tl + first, n, tgA, tgB, kp, nxt, aAx, aAy, aBx, aBy, bx, by);
        int last = first + n - 1;                        // offset of the element whose reaction this lane holds
        if (p == 0) {
            float ux, uy;
            pair_sym<false, PRECISE, true>(tl[16], tgA, kp, aAx, aAy, ux, uy);
        } else if (p == 1) {
            bx = __shfl_sync(kFull, bx, nxt);
            by = __shfl_sync(kFull, by, nxt);
            const float4 q = tl[16];
            float ux, uy;
            pair_sym<true, PRECISE, true>(q, tgA, kp, aAx, aAy, bx, by);
            pair_sym<false, PRECISE, true>(q, tgB, kp, aBx, aBy, ux, uy);
            last = 16;
        }
        sm.slot[(H * nslots + o) * 32 + ((lane + last) & 31)] = make_float2(bx, by);
    }
    vx[0] = aAx; vy[0] = aAy; vx[1] = aBx; vy[1] = aBy;
}

// MODE 3, part 2: reactions (fixed order: bitwise reproducible), then the agents' pull summed from 0 and added last --
// evaluated before the tile passes in the latency-bound SELF shape (AGF: off the critical path behind the barrier) or
// here (the throughput-bound shapes: no buffer); the same bits either way.
template <bool PRECISE, bool AGF>
__device__ __forceinline__ void forces_sym64_finish(const Smem& sm, const KP& kp, const Grp& g, float (&vx)[2],
                                                    float (&vy)[2]) {
    const int lane = g.tid & 31, I = g.tid >> 5;
    const int nt2 = (kp.N + 63) >> 6, nslots = 1 + nt2 / 2;
    for (int o = 0; o < nslots; ++o) {
        const float2 ra = sm.slot[((2 * I) * nslots + o) * 32 + lane];
        const float2 rb = sm.slot[((2 * I + 1) * nslots + o) * 32 + lane];
        vx[0] += ra.x; vy[0] += ra.y;
        vx[1] += rb.x; vy[1] += rb.y;
    }
    float gAx = 0.f, gAy = 0.f, gBx = 0.f, gBy = 0.f;
    if constexpr (AGF) {
        const float2 a = sm.agf[(2 * I) * 32 + lane], b = sm.agf[(2 * I + 1) * 32 + lane];   // this thread's own writes
        gAx = a.x; gAy = a.y; gBx = b.x; gBy = b.y;
    } else {
        const float4 tgA = sm.src[(2 * I) * 64 + lane], tgB = sm.src[(2 * I + 1) * 64 + lane];
        const float4* ag = sm.src + nt2 * 128;      // agents act on locusts only (multiagent.py:108-113)
        if constexpr (PRECISE) {
            for (int k = 0; k < kp.A; ++k) {
                const float4 q = ag[k];
                pair_ordered<PRECISE>(q, tgA, kp, gAx, gAy);
                pair_ordered<PRECISE>(q, tgB, kp, gBx, gBy);
            }
        } else {
            const Targets2 t = make_targets2(tgA, tgB);
            const PairConst2 c = make_pair_const2(kp);
            f32x2 naA = 0, naB = 0, b = 0;
#pragma unroll 2
            for (int k = 0; k < kp.A; ++k) pair2_fast<false>(ag[k], t, c, naA, naB, b);
            upk2(naA, gAx, gAy);
            upk2(naB, gBx, gBy);
            gAx = -gAx; gAy = -gAy; gBx = -gBx; gBy = -gBy;
        }
    }
    vx[0] += gAx; vy[0] += gAy;
    vx[1] += gBx; vy[1] += gBy;
}

// MODE 2/4: ordered pairs, T targets per thread (j = tid + t*n), broadcast LDS.128 sources.
template <int T, bool PRECISE>
__device__ __forceinline__ void forces_ordered(const Smem& sm, const KP& kp, const Grp& g, float (&vx)[T], float (&vy)[T]) {
    const int N = kp.N, S = kp.N + kp.A;
    float4 tg[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
        const int j = g.tid + t * g.n;
        tg[t] = sm.src[j < N ? j : N - 1];
        vx[t] = 0.f;
        vy[t] = 0.f;
    }
#pragma unroll 4
    for (int i = 0; i < S; ++i) {
        const float4 q = sm.src[i];
#pragma unroll
        for (int t = 0; t < T; ++t) pair_ordered<PRECISE>(q, tg[t], kp, vx[t], vy[t]);
    }
}

// SwarmEnv.v_calculate (multiagent.py:88-115) on staged sources: v of this thread's targets (wind
// and gravity added, before any cutoff).  Needs the staged sources visible (a barrier since stage_*);
// contains one group barrier in the unordered-pair modes.
template <int MODE, bool PRECISE, bool AGF = false>
__device__ __forceinline__ void pair_forces(const Smem& sm, const KP& kp, const Grp& g, float (&vx)[ModeT<MODE>::T],
                                            float (&vy)[ModeT<MODE>::T], const long long trace_rec = -1) {
    constexpr int T = ModeT<MODE>::T;
    if (g.tid == 0) trace_mark(kp, trace_rec, TR_STAGED);
    if constexpr (MODE == 1) {
        forces_sym_tiles<PRECISE, AGF>(sm, kp, g, vx[0], vy[0]);
        if (g.tid == 0) trace_mark(kp, trace_rec, TR_TILES);
        g.sync();
        forces_sym_finish<PRECISE, AGF>(sm, kp, g, vx[0], vy[0]);
    } else if constexpr (MODE == 3) {
        forces_sym64_tiles<PRECISE, AGF>(sm, kp, g, vx, vy);
        if (g.tid == 0) trace_mark(kp, trace_rec, TR_TILES);
        g.sync();
        forces_sym64_finish<PRECISE, AGF>(sm, kp, g, vx, vy);
    } else {
        forces_ordered<T, PRECISE>(sm, kp, g, vx, vy);
    }
#pragma unroll
    for (int t = 0; t < T; ++t) {
        vx[t] += kp.U;
        vy[t] += kp.Gv;
    }
}

// reward = -mean_j |v_j|^2 (multiagent.py:114-115, v before any cutoff): a warp-shuffle sum per 32-locust tile
// into one slot per tile, then the slots in order.
// The caller barriers between energy_put and energy_get.
template <int MODE>
__device__ __forceinline__ int energy_slots(const KP&, const Grp& g) { return g.n >> 5; }
template <int MODE>
__device__ __forceinline__ void energy_put(const Smem& sm, const KP& kp, const Grp& g, const float (&vx)[ModeT<MODE>::T],
                                           const float (&vy)[ModeT<MODE>::T]) {
    constexpr int T = ModeT<MODE>::T;
    double e = 0.0;
#pragma unroll
    for (int t = 0; t < T; ++t)
        if (target_index<MODE>(g, t, kp) < kp.N) e += (double)vx[t] * (double)vx[t] + (double)vy[t] * (double)vy[t];
    e = warp_sum(e);
    if ((g.tid & 31) == 0) sm.red[g.tid >> 5] = e;
}
template <int MODE>
__device__ __forceinline__ double energy_get(const Smem& sm, const KP& kp, const Grp& g) {
    double tot = 0.0;
    const int nw = energy_slots<MODE>(kp, g);
    for (int w = 0; w < nw; ++w) tot += sm.red[w];   // same order in every thread
    return -div_by_const(tot, (double)kp.N, kp.inv_N);
}

// SwarmEnv._step on the stage buffer sm.st.  Preconditions: st.xs/as/an, sm.nx and sm.act filled, each
// element written by the thread that owns it here (element i <-> thread i mod n) or visible through
// a barrier.  Postcondition: state updated and visible to the whole group; returns the reward.
// PHYS: the physics constants come from the row sm.st.ph (visible to the group), read where they are used.
template <int MODE, bool PRECISE, bool AGF = false, bool PHYS = false>
__device__ __forceinline__ double env_step(const Smem& sm, const KP& kp, const Grp& g, float* v_out, const double wind_a,
                                           const long long trace_rec = -1) {
    constexpr int T = ModeT<MODE>::T;
    // multiagent.py:33-38  agents move first: v_action (+wind on x unless add_wind=False) through x_update; the
    // mover stages the agent's NEW position as a force source (multiagent.py:39: old x, new xa)
    float4* ag = agent_sources<MODE>(sm, kp);
    for (int k = g.tid; k < kp.A; k += g.n) {
        double2 a = sm.st.as[k];
        double2 w = sm.act[k];
        w.x = __dadd_rn(w.x, wind_a);
        if constexpr (PHYS) move_particle(a, w, sm.st.an[k], sm.st.ph[5], sm.st.ph[0]);
        else move_particle(a, w, sm.st.an[k], kp.dt, kp.sigma);
        sm.st.as[k] = a;
        ag[k] = split_hilo(a, kp.cscale);
    }
    stage_locusts<MODE>(sm, kp, g);
    g.sync();
    float vx[T], vy[T];
    if constexpr (PHYS) pair_forces<MODE, PRECISE, AGF>(sm, phys_kp(kp, sm.st.ph), g, vx, vy, trace_rec);
    else pair_forces<MODE, PRECISE, AGF>(sm, kp, g, vx, vy, trace_rec);
    if (g.tid == 0) trace_mark(kp, trace_rec, TR_FORCES);
    energy_put<MODE>(sm, kp, g, vx, vy);
    cp_async_wait_but_one();   // this thread's own noise rows have landed in sm.nx (no-op outside k_step)
    // multiagent.py:40  locusts move with the pre-cutoff v just computed
#pragma unroll
    for (int t = 0; t < T; ++t) {
        const int j = target_index<MODE>(g, t, kp);
        if (j < kp.N) {
            if (v_out) reinterpret_cast<float2*>(v_out)[j] = make_float2(vx[t], vy[t]);
            double2 p = sm.st.xs[j];
            if constexpr (PHYS) move_particle(p, make_double2((double)vx[t], (double)vy[t]), sm.nx[j], sm.st.ph[5], sm.st.ph[0]);
            else move_particle(p, make_double2((double)vx[t], (double)vy[t]), sm.nx[j], kp.dt, kp.sigma);
            sm.st.xs[j] = p;
        }
    }
    g.sync();
    return energy_get<MODE>(sm, kp, g);
}

// SwarmEnv._reset (multiagent.py:46-63) for env e on the stage buffer, in two pieces so that the
// burn-in steps can share the ONE env_step call site of the calling kernel:
//   reset_begin      the initial positions (injected or Philox draws)
//   reset_row(r)     noise row r and burn-in action r into the stage buffer; for r == n_burn the row is
//                    the frozen one: it is stored to HBM for all later steps (SURVEY Q1) and the
//                    function returns true (no step follows).
// Sequence: reset_begin; for (r = 0; !reset_row(r); ++r) env_step.
struct ResetCtx {
    DrawCtx draw;
    int e;
    bool inj;
};

__device__ __forceinline__ ResetCtx reset_begin(const Smem& sm, const KP& kp, const Grp& g, int e, uint32_t episode,
                                                const bool inj, const SwarmInjectedDraws& dr) {
    const int N = kp.N, A = kp.A;
    ResetCtx rc;
    rc.draw.key = kp.key;
    rc.draw.env = kp.env_off + (uint32_t)e;
    rc.draw.episode = episode;
    rc.e = e;
    rc.inj = inj;
    g.sync();      // the previous step's readers of red / src / xs are done
    for (int i = g.tid; i < N; i += g.n)
        sm.st.xs[i] = inj ? reinterpret_cast<const double2*>(dr.x0)[(size_t)e * N + i]
                          : draw_uniform2(rc.draw, STREAM_X0, i);
    for (int k = g.tid; k < A; k += g.n)
        sm.st.as[k] = inj ? reinterpret_cast<const double2*>(dr.xa0)[(size_t)e * A + k]
                          : draw_uniform2(rc.draw, STREAM_XA0, k);
    return rc;
}

__device__ __forceinline__ bool reset_row(const Smem& sm, const KP& kp, const Grp& g, const ResetCtx& rc, const int r,
                                          const SwarmInjectedDraws& dr, const SwarmState& st) {
    const int N = kp.N, A = kp.A, e = rc.e, rows = kp.n_burn + 1;
    const bool last = r >= kp.n_burn;
    for (int j = g.tid; j < N; j += g.n) {
        const double2 z = rc.inj ? reinterpret_cast<const double2*>(dr.particle_noise)[((size_t)e * rows + r) * N + j]
                                 : draw_normal2(rc.draw, STREAM_NOISE_X, r, j);
        sm.nx[j] = z;
        if (last) reinterpret_cast<double2*>(st.noise_x)[(size_t)e * N + j] = z;
    }
    for (int k = g.tid; k < A; k += g.n) {
        const double2 z = rc.inj ? reinterpret_cast<const double2*>(dr.agent_noise)[((size_t)e * rows + r) * A + k]
                                 : draw_normal2(rc.draw, STREAM_NOISE_A, r, k);
        sm.st.an[k] = z;
        if (last) {
            reinterpret_cast<double2*>(st.noise_a)[(size_t)e * A + k] = z;
        } else {
            sm.act[k] = rc.inj ? reinterpret_cast<const double2*>(dr.burn_actions)[((size_t)e * kp.n_burn + r) * A + k]
                               : draw_normal2(rc.draw, STREAM_BURN, r, k);
        }
    }
    if (last) g.sync();
    return last;
}

// ------------------------------------------------------------------------------------------
// np.searchsorted(edges, p, side='right') for edges = linspace(lo, hi, G+1) as numpy builds
// them: e[i] = fl(fl(i*step) + lo) for i < G, e[G] = hi  (numpy/_core/function_base.py).
__device__ __forceinline__ double edge_at(int i, double lo, double hi, double step, int G) {
    return i >= G ? hi : __dadd_rn(__dmul_rn((double)i, step), lo);
}

// The bin is guessed with a reciprocal multiply.  Each of numpy's edges is within an ulp of max(|lo|, |hi|) of
// lo + i*step (the rounding of fl(i*step) + lo), and the subtraction and the multiply of the guess
// q = (p - lo) / step add a few ulp of the bin width, so q is within slack = 1e-9 + 16 max(|lo|, |hi|) 2^-52 / step
// bins of the real position of p between numpy's edges: a guess whose fractional part is further than that from
// 0 and 1 is certain.  Anything else -- points on or next to an edge, outside [lo, hi) -- is settled against the
// exact edges.  (The magnitude term matters far from the origin: at |lo| ~ 1e6 one ulp is already ~3e-9 bins.)
__device__ __forceinline__ int count_le(double p, double lo, double hi, double step, double inv_step, int G) {
    if (p == lo) return 1;                       // e[0] = lo exactly (the grounded locusts' y = 0 lands here)
    const double q = (p - lo) * inv_step;
    const double fl = floor(q);
    const double fr = q - fl;
    const double slack = 1e-9 + 16.0 * fmax(fabs(lo), fabs(hi)) * 2.220446049250313e-16 * inv_step;
    if (q > 0.0 && q < (double)G && fr > slack && fr < 1.0 - slack) return (int)fl + 1;
    if (!(p == p)) return G + 1;                 // NaN sorts last
    int g = q < -1.0 ? -1 : (q > (double)G ? G : (int)fl);
    while (g < G && edge_at(g + 1, lo, hi, step, G) <= p) ++g;
    while (g >= 0 && edge_at(g, lo, hi, step, G) > p) --g;
    return g + 1;                                // #{i in [0,G] : e[i] <= p}
}

// Streaming zero fill of one env's (G,G,2) f32 grid by n threads (evict-first stores): 16-byte stores where the grid
// is 16-byte aligned, 8-byte ones otherwise (a grid only needs 8-byte alignment, e.g. a slot of a caller's buffer).
__device__ __forceinline__ void raster_zero_fill(float* __restrict__ grid_e, int cells, int tid, int n) {
    if ((cells & 1) == 0 && (reinterpret_cast<uintptr_t>(grid_e) & 15) == 0) {
        float4* g4 = reinterpret_cast<float4*>(grid_e);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = tid; i < cells / 2; i += n) __stcs(g4 + i, z);
    } else {
        float2* g2 = reinterpret_cast<float2*>(grid_e);
        for (int i = tid; i < cells; i += n) __stcs(g2 + i, make_float2(0.f, 0.f));
    }
}

// The same zero fill by the TMA engine (cp.async.bulk shared -> global): the source of the zeros is
// the rasteriser's own counter table, which is all zero between two envs (env_raster cleans it),
// so a whole 56 KB observation costs ONE thread a handful of instructions and no LSU traffic.
// Usable when the table size is a multiple of 16 bytes (cells % 4 == 0) and grid_e is 16-byte
// aligned.  Protocol (one thread issues, see k_step):
//   tma_zero_fill_issue    after a barrier that follows the table clean-up
//   tma_zero_fill_wait_read  before the first atomic on the table (the engine has read its zeros)
//   tma_zero_fill_wait_done  before the first ordinary store to grid_e (the zeros have landed)
__device__ __forceinline__ bool tma_zero_fill_ok(const void* grid, int cells) {
    return (cells & 7) == 0 && (reinterpret_cast<uintptr_t>(grid) & 15) == 0;
}
// table_bytes: size of the (all-zero) counter table, a multiple of 16 that divides the grid's 8*cells bytes
__device__ __forceinline__ void tma_zero_fill_issue(float* __restrict__ grid_e, const uint32_t* table, int cells,
                                                    uint32_t table_bytes) {
    // make the generic-proxy zeros of the table visible to the async proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const uint32_t src = (uint32_t)__cvta_generic_to_shared(table);
    unsigned char* dst = reinterpret_cast<unsigned char*>(grid_e);
    const uint32_t total = (uint32_t)cells * 8u;
    for (uint32_t off = 0; off < total; off += table_bytes)
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + off), "r"(src),
                     "r"(table_bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_zero_fill_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_zero_fill_wait_done() {
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    asm volatile("fence.proxy.async;" ::: "memory");         // async-proxy writes before the generic stores that follow
}

// One-time clear of the counter table (afterwards env_raster leaves it clean).
template <typename Group>
__device__ __forceinline__ void raster_table_clear(const Smem& sm, int words, const Group& g) {
    uint4* t4 = reinterpret_cast<uint4*>(sm.table);      // (smem_table_bytes is a multiple of 16, the table 16-byte aligned)
    for (int i = g.tid; i < (words >> 2); i += g.n) t4[i] = make_uint4(0u, 0u, 0u, 0u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the TMA zero fill reads these zeros
}

// grid values of the small counts, once per CTA: lut[c] = c / N (c < lut_locusts), lut[lut_locusts + a] = a / A, rounded
// like the scatter's own division
__device__ __forceinline__ void raster_lut_fill(const Smem& sm, const KP& kp, const int tid, const int n) {
    const float fN = (float)kp.N, fA = (float)(kp.A > 0 ? kp.A : 1);
    const int nl = lut_locusts(kp.N), na = lut_agents(kp.A);
    for (int c = tid; c < nl; c += n) sm.lut[c] = __fdiv_rn((float)c, fN);
    for (int c = tid; c < na; c += n) sm.lut[nl + c] = __fdiv_rn((float)c, fA);
}

// How env_raster waits for the zero fill of its grid (besides being a group barrier at both points):
//   ZeroOwn     a thread of the group issued the TMA fill (tma_tid) or the group stored the zeros itself
//   ZeroSelf    k_step's SELF shape: a filler warp outside the group issued it and arrives on BAR_ZREAD / BAR_ZDONE, or
//               (no filler) the group stored the zeros itself
struct ZeroOwn {
    bool tma;
    int tma_tid;
    template <typename Group>
    __device__ __forceinline__ void before_table(const Group& g) const {
        if (tma && g.tid == tma_tid) tma_zero_fill_wait_read();      // the table may be written from here on
        g.sync();
    }
    template <typename Group>
    __device__ __forceinline__ void before_scatter(const Group& g) const {
        if (tma && g.tid == tma_tid) tma_zero_fill_wait_done();      // the zeros are in place before anyone scatters over them
        g.sync();
    }
};
struct ZeroSelf {            // filler: the warp outside the group; else the group stored the zeros itself
    bool filler;
    int n_all;
    template <typename Group>
    __device__ __forceinline__ void before_table(const Group& g) const {
        if (filler) bar_sync<BAR_ZREAD>(n_all); else g.sync();
    }
    template <typename Group>
    __device__ __forceinline__ void before_scatter(const Group& g) const {
        if (filler) bar_sync<BAR_ZDONE>(n_all); else g.sync();
    }
};

// SwarmStateProcessor.process_state (state_processors.py:25-42) of the points pts = [N locusts; A
// agents] in shared memory, by the thread group g.  grid_e: (G,G,2) f32, pos_e: (A,2) u8 of this env.
// Preconditions: grid_e zero-filled or being zero-filled (see ZeroOwn / ZeroFiller), sm.table all zero, sm.lut filled
// (raster_lut_fill) and pts visible (a barrier since).  Postcondition: sm.table all zero again, after a group barrier.
// overlap_fn(tid, n) is the caller's work that only needs pts (e.g. the write-back of the state); early_release_fn() is
// called by every thread once it has read its last point from pts (the step kernel hands the buffer back to the force
// group there).
//
// The window's centre is np.mean(vstack([x, xa]), axis=0)[0]: a plain left-to-right FP64 sum, i.e. a chain of N+A dependent
// DADDs on ONE thread (23 cycles each: 3 us at N = 256, the longest single piece of an env's rasterisation).  The chain is
// only needed when some point sits so close to a bin edge that the last bits of the mean decide its bin.  So every
// thread first bins its points against a PARALLEL mean (tree sum; it differs from numpy's sequential one by at most
// (N+A) 2^-52 max|x|) and checks that each point is further from the nearest edge than everything that could separate
// the two computations (tol below, a rigorous bound with slack).  If all points pass, the bins -- hence the whole
// observation -- are provably the ones numpy's edges give, and the chain is never walked; if any point fails (or EXACT:
// the standalone rasteriser, which also reports the box) thread 0 walks the chain and the x bins are taken again against
// numpy's exact edges.
struct NoRelease { __device__ __forceinline__ void operator()() const {} };
struct NoOverlap { __device__ __forceinline__ void operator()(int, int) const {} };

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

#ifndef SWARM_SPEC_MEAN
#define SWARM_SPEC_MEAN 1
#endif
template <bool EXACT, typename Group, typename Zero, typename Release, typename Overlap>
__device__ __forceinline__ void env_raster(const Smem& sm, const double2* __restrict__ pts, const KP& kp, const Group& g,
                                           float* __restrict__ grid_e, uint8_t* __restrict__ pos_e, const bool tma,
                                           const Zero zero, const Release early_release_fn, const Overlap overlap_fn,
                                           const long long trace_rec = -1) {
    const int N = kp.N, A = kp.A, G = kp.G, P = N + A;
    float2* g2 = reinterpret_cast<float2*>(grid_e);
    const bool t16 = table_is16(N, A);
    if (g.tid == 0) trace_mark(kp, trace_rec, TR_RASTER);
    const double lo_y = 0.0, hi_y = kp.y_hi;
    const double step_y = kp.step_y, inv_y = kp.inv_y;
    constexpr bool SPEC = !EXACT && SWARM_SPEC_MEAN;
    int* const unsure = reinterpret_cast<int*>(sm.rred + 2 * kMaxWarps);
    overlap_fn(g.tid, g.n);
    if constexpr (SPEC) {
        // phase 0: the parallel mean and the largest |x| (for the error bound)
        double part = 0.0, amax = 0.0;
        for (int p = g.tid; p < P; p += g.n) {
            const double v = pts[p].x;
            part += v;
            amax = fmax(amax, fabs(v));
        }
        part = warp_sum(part);
        amax = warp_max(amax);
        if ((g.tid & 31) == 0) {
            sm.rred[2 * (g.tid >> 5)] = part;
            sm.rred[2 * (g.tid >> 5) + 1] = amax;
        }
        if (g.tid == 0) *unsure = 0;
        g.sync();
        double tot = 0.0, xmax = 0.0;
        for (int w = 0; w < (g.n >> 5); ++w) {
            tot += sm.rred[2 * w];
            xmax = fmax(xmax, sm.rred[2 * w + 1]);
        }
        if (g.tid == 0) trace_mark(kp, trace_rec, TR_MEAN);
        // Distance, in bins, that the guess q~ = (x - lo~) G/W can be from the point's position between numpy's edges
        // e[i] = fl(fl(i step) + lo):  the two means differ by <= (P + 1) 2^-52 xmax (both sums carry <= (P-1) 2^-53 sum|x|,
        // quotient / reciprocal-multiply roundings), lo, hi, step and each edge add a few ulp of (xmax + W), the guess's
        // own subtraction and multiply another few ulp.  (P + 16) xmax + 16 W covers all of it; twice that, plus 1e-9.
        const double lo_s = tot * kp.inv_P - kp.half_w;
        const double tol = 1e-9 + 2.0 * ((double)(P + 16) * xmax + 32.0 * kp.half_w) * 2.220446049250313e-16 * kp.inv_x;
        bool bad = !(tol < 0.25);       // (absurd magnitudes, NaN)
        for (int p = g.tid; p < P; p += g.n) {
            const double2 q = pts[p];
            const int cy = count_le(q.y, lo_y, hi_y, step_y, inv_y, G);
            const double qs = (q.x - lo_s) * kp.inv_x;
            const double fl = floor(qs);
            const double fr = qs - fl;
            bad |= !(fr > tol && fr < 1.0 - tol);          // next to an edge (q.x == hi_x included), or NaN
            const int cx = (int)fmin(fmax(fl, -1.0), (double)G) + 1;    // #{edges <= x}: 0 left of the box, G + 1 right of it
            if (p >= N) {   // np.digitize -> bin+1, clamped to G-1 (state_processors.py:35-40)
                pos_e[2 * (p - N) + 0] = (uint8_t)(cx < G - 1 ? cx : G - 1);
                pos_e[2 * (p - N) + 1] = (uint8_t)(cy < G - 1 ? cy : G - 1);
            }
            const int by = (q.y == hi_y) ? cy - 2 : cy - 1;             // histogramdd right-edge fix-up
            sm.cid[p] = cx | ((by + 1) << 16);                          // bin + 1 in both halves
        }
        if (bad) *unsure = 1;
    }
    zero.before_table(g);
    if (!SPEC || *unsure) {
        if (g.tid == 0) {
            double s = 0.0;
#pragma unroll 8
            for (int i = 0; i < P; ++i) s = __dadd_rn(s, pts[i].x);
            sm.box[0] = div_by_const(s, (double)P, kp.inv_P);
        }
        g.sync();
        // bin every point's x in FP64 against numpy's edges
        const double m = sm.box[0];
        const double lo_x = m - kp.half_w, hi_x = m + kp.half_w;
        const double step_x = div_by_const(hi_x - lo_x, (double)G, kp.inv_G);
        // 1 / step_x seeds the bin guess: two Newton steps from the host's G / WIDTH (step_x differs from WIDTH / G by
        // the rounding of mean +- WIDTH/2 only), a real division when the window sits absurdly far out
        double inv_x = kp.inv_x;
        const double dev = __fma_rn(-step_x, inv_x, 1.0);
        if (fabs(dev) < 1e-4) {
            inv_x = __fma_rn(inv_x, dev, inv_x);
            inv_x = __fma_rn(inv_x, __fma_rn(-step_x, inv_x, 1.0), inv_x);
        } else {
            inv_x = 1.0 / step_x;
        }
        for (int p = g.tid; p < P; p += g.n) {
            const double2 q = pts[p];
            const int cx = count_le(q.x, lo_x, hi_x, step_x, inv_x, G);
            const int cy = count_le(q.y, lo_y, hi_y, step_y, inv_y, G);
            if (p >= N) {
                pos_e[2 * (p - N) + 0] = (uint8_t)(cx < G - 1 ? cx : G - 1);
                pos_e[2 * (p - N) + 1] = (uint8_t)(cy < G - 1 ? cy : G - 1);
            }
            const int bx = (q.x == hi_x) ? cx - 2 : cx - 1;
            const int by = (q.y == hi_y) ? cy - 2 : cy - 1;
            sm.cid[p] = (bx + 1) | ((by + 1) << 16);
        }
    }
    early_release_fn();
    // phase 1: count with warp-aggregated atomics
    for (int base = 0; base < P; base += g.n) {
        const int p = base + g.tid;
        uint32_t key = 0xffffffffu;
        int cell = 0;
        if (p < P) {
            const int packed = sm.cid[p];
            const int bx = (packed & 0xffff) - 1, by = (packed >> 16) - 1;
            if (bx >= 0 && bx < G && by >= 0 && by < G) {
                cell = bx * G + by;
                key = ((uint32_t)cell << 1) | (p >= N ? 1u : 0u);
            }
        }
        const uint32_t peers = __match_any_sync(kFull, key);
        int mine = -1;
        if (key != 0xffffffffu && (__ffs(peers) - 1) == (g.tid & 31)) {
            const uint32_t cnt = (uint32_t)__popc(peers);
            if (t16) {   // 16 bits per cell, two cells per word
                const int sh = (cell & 1) << 4;
                const uint32_t old = atomicAdd(&sm.table[cell >> 1], (cnt << ((key & 1u) ? kAgentShift : 0)) << sh);
                if (((old >> sh) & 0xffffu) == 0u) mine = cell;   // first arrival writes the cell out
            } else {
                const uint32_t old = atomicAdd(&sm.table[cell], cnt << ((key & 1u) ? 16 : 0));
                if (old == 0u) mine = cell;
            }
        }
        if (p < P) sm.cid[p] = mine;
    }
    if (g.tid == 0) trace_mark(kp, trace_rec, TR_BINNED);
    zero.before_scatter(g);
    if (g.tid == 0) trace_mark(kp, trace_rec, TR_ZEROS);
    // phase 2: sparse scatter of the non-zero cells over the zeros; the writer cleans its counter
    for (int p = g.tid; p < P; p += g.n) {
        const int c = sm.cid[p];
        if (c >= 0) {
            uint32_t nl, na;
            if (t16) {
                const int sh = (c & 1) << 4;
                const uint32_t w = (atomicAnd(&sm.table[c >> 1], ~(0xffffu << sh)) >> sh) & 0xffffu;
                nl = w & ((1u << kAgentShift) - 1u);
                na = w >> kAgentShift;
            } else {
                const uint32_t w = sm.table[c];
                sm.table[c] = 0u;
                nl = w & 0xffffu;
                na = w >> 16;
            }
            const uint32_t ll = (uint32_t)lut_locusts(N);
            const float vl = nl < ll ? sm.lut[nl] : __fdiv_rn((float)nl, (float)N);
            const float va = A > 0 ? (na < (uint32_t)lut_agents(A) ? sm.lut[ll + na] : __fdiv_rn((float)na, (float)A)) : 0.f;
            g2[c] = make_float2(vl, va);
        }
    }
    if (tma) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // cleaned counters -> next TMA zero fill
    g.sync();
    if (g.tid == 0) trace_mark(kp, trace_rec, TR_DONE);
}

}  // namespace swarm
