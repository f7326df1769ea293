// Device code of the CLUSTER layout (SwarmParams::tuning bits 8-12): one env spread over the K CTAs of a thread-block
// cluster, for 512 < N <= 8192 (DESIGN 3.4).  The arithmetic is that of the one-CTA ordered-pair modes (MODE 2/4), so
// every output is bitwise the one-CTA kernels' for N <= 2048 and the same for every K:
//   * the env keeps the one-CTA kernel's VIRTUAL thread mapping: nf = block_threads(N, MODE) threads, thread v owning
//     targets v + t nf (t < T).  Its nf / 32 warps are split into K contiguous ranges, one per CTA, so pair_forces and
//     energy_put run unchanged with the virtual tid;
//   * every CTA builds all N + A FP32 hi/lo sources itself from the FP64 state in global memory (L2): O(N) against
//     the O(N^2 / K) pair work.  Every CTA moves all A agents (same bits); rank 0 alone writes them back;
//   * the per-warp FP64 energy slots are gathered over DSMEM and summed in virtual-warp order by every CTA, so every
//     CTA holds the same reward and takes the same done / auto-reset decision;
//   * the new locust positions go straight to global memory, after a cluster barrier that follows every CTA's reads
//     of the old ones;
//   * the observation is rasterised by the cluster itself: counters in x-bin bands across the CTAs (DSMEM atomics).
#pragma once
#include "swarm_kernels.cuh"

namespace swarm {

constexpr int kClusterMinLocusts = kSymMaxLocusts + 1;   // below: the one-CTA kernels use unordered pairs (other bits)
constexpr int kClusterMaxLocusts = 8192;                 // the CTA's copy of all sources must fit shared memory
constexpr int kClusterMaxK = 16;                         // non-portable cluster size of sm_100
constexpr int kClusterVWarps = 64;                       // virtual warps at N = 8192 (T = 4)

// ---- cluster primitives -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_ctas() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
// every thread of every CTA of the cluster; release / acquire at cluster scope (shared AND global memory)
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}
// the shared::cluster address of *p in the shared memory of CTA `rank`
__device__ __forceinline__ uint32_t dsmem(const void* p, uint32_t rank) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ double dsmem_ld_f64(uint32_t a) {
    double v;
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t dsmem_ld_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t dsmem_add_u32(uint32_t a, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared::cluster.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
    return old;
}

// ---- layout ---------------------------------------------------------------------------------------------------------
// first virtual warp of CTA r when nw warps are split over K CTAs
__host__ __device__ inline int cl_warp0(int r, int nw, int K) { return (int)(((long long)r * nw) / K); }
// threads per CTA: the largest warp range
__host__ __device__ inline int cl_threads(int nw, int K) { return ((nw + K - 1) / K) * 32; }
// rows of the grid's x bins whose counters CTA r holds: [r band, (r + 1) band)
__host__ __device__ inline int cl_band(int G, int K) { return (G + K - 1) / K; }

struct CSmem {
    float4* src;       // N + A FP32 hi/lo sources (step / forces); the rasteriser's counter band overlaps them
    uint32_t* table;   // band x G 32-bit cell counters (locusts lo16, agents hi16) of this CTA's x bins
    double2* as;       // A   agent positions (every CTA keeps all of them)
    double2* an;       // A   agent noise row
    double2* act;      // A   actions after conversion / clipping
    double* red;       // kClusterVWarps: this CTA's per-warp energy slots (by local warp)
    double* slots;     // kClusterVWarps: every virtual warp's slot, gathered in order
    double* rred;      // 2 kMaxWarps: per-warp (sum x, max |x|); then 2 (this CTA's); 2 kClusterMaxK (all CTAs'); 2 (box)
    int* flag;         // 4 ints
    float* lut;        // grid values of the small counts (raster_lut_fill)
};

__host__ __device__ inline size_t cl_src_bytes(int N, int A, int G, int K, bool force) {
    const size_t s = force ? sizeof(float4) * ((size_t)N + A) : 0, t = sizeof(uint32_t) * (size_t)cl_band(G, K) * G;
    return smem_align(s > t ? s : t);
}
__host__ __device__ inline size_t cl_smem_bytes(int N, int A, int G, int K, bool force) {
    return cl_src_bytes(N, A, G, K, force) + 3 * smem_align(sizeof(double2) * A) + 2 * smem_align(sizeof(double) * kClusterVWarps) +
           smem_align(sizeof(double) * (2 * kMaxWarps + 2 + 2 * kClusterMaxK + 2)) + 16 +
           smem_align(sizeof(float) * (lut_locusts(N) + lut_agents(A)));
}
__device__ __forceinline__ CSmem cl_carve(unsigned char* base, int N, int A, int G, int K, bool force) {
    CSmem s;
    size_t o = 0;
    s.src = reinterpret_cast<float4*>(base);
    s.table = reinterpret_cast<uint32_t*>(base);
    o += cl_src_bytes(N, A, G, K, force);
    s.as = reinterpret_cast<double2*>(base + o);  o += smem_align(sizeof(double2) * A);
    s.an = reinterpret_cast<double2*>(base + o);  o += smem_align(sizeof(double2) * A);
    s.act = reinterpret_cast<double2*>(base + o); o += smem_align(sizeof(double2) * A);
    s.red = reinterpret_cast<double*>(base + o);  o += smem_align(sizeof(double) * kClusterVWarps);
    s.slots = reinterpret_cast<double*>(base + o); o += smem_align(sizeof(double) * kClusterVWarps);
    s.rred = reinterpret_cast<double*>(base + o); o += smem_align(sizeof(double) * (2 * kMaxWarps + 2 + 2 * kClusterMaxK + 2));
    s.flag = reinterpret_cast<int*>(base + o);    o += 16;
    s.lut = reinterpret_cast<float*>(base + o);
    return s;
}

// This CTA's share of the env's virtual thread mapping.
struct CMap {
    int rank, K;       // cluster rank and size
    int nf, nw;        // virtual threads / warps of the env
    int w0, nwl;       // first virtual warp of this CTA, and how many it runs
    int vtid;          // virtual tid of this thread
    bool active;       // this thread runs a virtual thread (whole warps)
};
__device__ __forceinline__ CMap cl_map(const int nf) {
    CMap m;
    m.rank = (int)cluster_rank();
    m.K = (int)cluster_ctas();
    m.nf = nf;
    m.nw = nf >> 5;
    m.w0 = cl_warp0(m.rank, m.nw, m.K);
    m.nwl = cl_warp0(m.rank + 1, m.nw, m.K) - m.w0;
    m.vtid = m.w0 * 32 + (int)threadIdx.x;
    m.active = (int)threadIdx.x < m.nwl * 32;
    return m;
}

// Sources of one step: agents (moved first when MOVE, multiagent.py:33-39) and locusts, split like stage_locusts
// (FP64 state from global memory, L2).  Ends with a CTA barrier.
template <bool MOVE>
__device__ __forceinline__ void cl_stage(const CSmem& sm, const KP& kp, const double2* __restrict__ xe,
                                         const double2* __restrict__ xae, const double wind_a) {
    const int N = kp.N, A = kp.A, tid = (int)threadIdx.x, n = (int)blockDim.x;
    float4* ag = sm.src + N;
    if (tid < A) {
        double2 a;
        if (MOVE) {
            a = sm.as[tid];
            double2 w = sm.act[tid];
            w.x = __dadd_rn(w.x, wind_a);
            move_particle(a, w, sm.an[tid], kp.dt, kp.sigma);
            sm.as[tid] = a;
        } else {
            a = xae[tid];
        }
        ag[tid] = split_hilo(a, kp.cscale);
    }
    for (int i = tid; i < N; i += n) sm.src[i] = split_hilo(__ldcg(xe + i), kp.cscale);
    __syncthreads();
}

// pair forces + wind / gravity of this thread's virtual targets and its warp's energy slot (= pair_forces + energy_put
// of the one-CTA kernel with the virtual tid)
template <int MODE, bool PRECISE>
__device__ __forceinline__ void cl_forces(const CSmem& sm, const KP& kp, const CMap& m, float (&vx)[ModeT<MODE>::T],
                                          float (&vy)[ModeT<MODE>::T]) {
    Smem s;
    s.src = sm.src;
    s.red = sm.red - m.w0;          // energy_put writes slot (virtual warp); this CTA keeps its own warps' slots
    const Grp vg = {m.vtid, m.nf};
    pair_forces<MODE, PRECISE>(s, kp, vg, vx, vy);
    energy_put<MODE>(s, kp, vg, vx, vy);
}

// reward after the cluster barrier that follows every cl_forces: every CTA sums all virtual warps' slots in order
// (energy_get).  Contains a CTA barrier.
__device__ __forceinline__ double cl_reward(const CSmem& sm, const KP& kp, const CMap& m) {
    const int w = (int)threadIdx.x;
    if (w < m.nw) {
        const int r = ((w + 1) * m.K - 1) / m.nw;              // owner: cl_warp0(r) <= w < cl_warp0(r + 1)
        sm.slots[w] = dsmem_ld_f64(dsmem(sm.red + (w - cl_warp0(r, m.nw, m.K)), (uint32_t)r));
    }
    __syncthreads();
    double tot = 0.0;
    for (int i = 0; i < m.nw; ++i) tot += sm.slots[i];
    return -div_by_const(tot, (double)kp.N, kp.inv_N);
}

// ---- rasteriser ------------------------------------------------------------------------------------------------------
// process_state of the cluster's env (env_raster's algorithm, DESIGN 3.4): CTA r bins the points of its own virtual
// threads' targets (+ rank 0: the agents), counts them into the owner CTA's band of counters over DSMEM, and
// scatters the cells it wrote first over the zeros.  Points come from global memory: xe / xae must hold the final
// state, written by this very thread (own targets, rank 0's agents) or before a cluster barrier.  Every thread of the
// cluster calls it; it ends after the scatter: the caller's cluster barrier must follow before any CTA exits.
// EXACT: the window's centre is always numpy's sequential sum (the box is reported by rank 0).
template <int T, bool EXACT>
__device__ __forceinline__ void cl_raster(const CSmem& sm, const KP& kp, const CMap& m, const double2* __restrict__ xe,
                                          const double2* __restrict__ xae, float* __restrict__ grid_e,
                                          uint8_t* __restrict__ pos_e, double* __restrict__ box_e) {
    const int N = kp.N, A = kp.A, G = kp.G, P = N + A, cells = G * G;
    const int tid = (int)threadIdx.x, n = (int)blockDim.x;
    const int band = cl_band(G, m.K);
    const bool agent = m.rank == 0 && tid < A;          // this thread also owns agent point `tid`
    const double lo_y = 0.0, hi_y = kp.y_hi;
    // this CTA's counters and zeros; the grid values of the small counts
    for (int i = tid; i < band * G; i += n) sm.table[i] = 0u;
    {
        float2* g2 = reinterpret_cast<float2*>(grid_e);
        const int c0 = (int)(((long long)m.rank * cells) / m.K), c1 = (int)(((long long)(m.rank + 1) * cells) / m.K);
        for (int i = c0 + tid; i < c1; i += n) __stcs(g2 + i, make_float2(0.f, 0.f));
        Smem s;
        s.lut = sm.lut;
        raster_lut_fill(s, kp, tid, n);
    }
    double2 q[T + 1];
#pragma unroll
    for (int t = 0; t < T; ++t) {
        const int j = m.vtid + t * m.nf;
        q[t] = (m.active && j < N) ? __ldcg(xe + j) : make_double2(0.0, 0.0);
    }
    q[T] = agent ? __ldcg(xae + tid) : make_double2(0.0, 0.0);
    auto owns = [&](const int t) { return t < T ? (m.active && m.vtid + t * m.nf < N) : agent; };
    constexpr bool SPEC = !EXACT && SWARM_SPEC_MEAN;
    double tot = 0.0, xmax = 0.0;
    if constexpr (SPEC) {   // this CTA's partial (sum x, max |x|)
        double part = 0.0, amax = 0.0;
#pragma unroll
        for (int t = 0; t <= T; ++t)
            if (owns(t)) {
                part += q[t].x;
                amax = fmax(amax, fabs(q[t].x));
            }
        part = warp_sum(part);
        amax = warp_max(amax);
        if ((tid & 31) == 0) {
            sm.rred[2 * (tid >> 5)] = part;
            sm.rred[2 * (tid >> 5) + 1] = amax;
        }
        __syncthreads();
        if (tid == 0) {
            double s = 0.0, mx = 0.0;
            for (int w = 0; w < (n >> 5); ++w) {
                s += sm.rred[2 * w];
                mx = fmax(mx, sm.rred[2 * w + 1]);
            }
            sm.rred[2 * kMaxWarps] = s;
            sm.rred[2 * kMaxWarps + 1] = mx;
        }
    }
    cluster_sync();     // counters clear, zeros stored, partials and (the caller's) state writes visible cluster-wide
    double* const allp = sm.rred + 2 * kMaxWarps + 2;
    int cid[T + 1];
    bool unsure = !SPEC;
    if constexpr (SPEC) {
        if (tid < m.K) {
            allp[2 * tid] = dsmem_ld_f64(dsmem(sm.rred + 2 * kMaxWarps, (uint32_t)tid));
            allp[2 * tid + 1] = dsmem_ld_f64(dsmem(sm.rred + 2 * kMaxWarps + 1, (uint32_t)tid));
        }
        __syncthreads();
        for (int r = 0; r < m.K; ++r) {     // rank order (the bound below does not depend on it)
            tot += allp[2 * r];
            xmax = fmax(xmax, allp[2 * r + 1]);
        }
        const double lo_s = tot * kp.inv_P - kp.half_w;
        const double tol = 1e-9 + 2.0 * ((double)(P + 16) * xmax + 32.0 * kp.half_w) * 2.220446049250313e-16 * kp.inv_x;
        bool bad = !(tol < 0.25);
#pragma unroll
        for (int t = 0; t <= T; ++t) {
            cid[t] = 0;
            if (!owns(t)) continue;
            const double2 p = q[t];
            const int cy = count_le(p.y, lo_y, hi_y, kp.step_y, kp.inv_y, G);
            const double qs = (p.x - lo_s) * kp.inv_x;
            const double fl = floor(qs);
            const double fr = qs - fl;
            bad |= !(fr > tol && fr < 1.0 - tol);
            const int cx = (int)fmin(fmax(fl, -1.0), (double)G) + 1;
            if (t == T) {
                pos_e[2 * tid + 0] = (uint8_t)(cx < G - 1 ? cx : G - 1);
                pos_e[2 * tid + 1] = (uint8_t)(cy < G - 1 ? cy : G - 1);
            }
            const int by = (p.y == hi_y) ? cy - 2 : cy - 1;
            cid[t] = cx | ((by + 1) << 16);
        }
        // a point far enough from every edge has numpy's bins whatever the other points do: the fall-back is per CTA
        unsure = __syncthreads_or(bad) != 0;
    }
    if (unsure) {
        // numpy's sequential mean, walked from global memory (every point is final and visible since the barrier)
        if (tid == 0) {
            double s = 0.0;
#pragma unroll 8
            for (int i = 0; i < N; ++i) s = __dadd_rn(s, __ldcg(&xe[i].x));
            for (int k = 0; k < A; ++k) s = __dadd_rn(s, __ldcg(&xae[k].x));
            sm.rred[2 * kMaxWarps + 2 + 2 * kClusterMaxK] = div_by_const(s, (double)P, kp.inv_P);
        }
        __syncthreads();
        const double mean = sm.rred[2 * kMaxWarps + 2 + 2 * kClusterMaxK];
        const double lo_x = mean - kp.half_w, hi_x = mean + kp.half_w;
        const double step_x = div_by_const(hi_x - lo_x, (double)G, kp.inv_G);
        double inv_x = kp.inv_x;
        const double dev = __fma_rn(-step_x, inv_x, 1.0);
        if (fabs(dev) < 1e-4) {
            inv_x = __fma_rn(inv_x, dev, inv_x);
            inv_x = __fma_rn(inv_x, __fma_rn(-step_x, inv_x, 1.0), inv_x);
        } else {
            inv_x = 1.0 / step_x;
        }
#pragma unroll
        for (int t = 0; t <= T; ++t) {
            cid[t] = 0;
            if (!owns(t)) continue;
            const double2 p = q[t];
            const int cx = count_le(p.x, lo_x, hi_x, step_x, inv_x, G);
            const int cy = count_le(p.y, lo_y, hi_y, kp.step_y, kp.inv_y, G);
            if (t == T) {
                pos_e[2 * tid + 0] = (uint8_t)(cx < G - 1 ? cx : G - 1);
                pos_e[2 * tid + 1] = (uint8_t)(cy < G - 1 ? cy : G - 1);
            }
            const int bx = (p.x == hi_x) ? cx - 2 : cx - 1;
            const int by = (p.y == hi_y) ? cy - 2 : cy - 1;
            cid[t] = (bx + 1) | ((by + 1) << 16);
        }
        if (EXACT && box_e && m.rank == 0 && tid == 0) {
            box_e[0] = lo_x;
            box_e[1] = hi_x;
            box_e[2] = 0.0;
            box_e[3] = kp.y_hi;
        }
    }
    // count: warp-aggregated DSMEM atomics into the owner CTA's band; the first arrival at a cell writes it out
    const bool warp_live = m.active || (m.rank == 0 && tid < 32 && A > 0);     // warp-uniform
    uint32_t addr[T + 1];
#pragma unroll
    for (int t = 0; t <= T; ++t) {
        addr[t] = 0xffffffffu;
        if (!warp_live || (t == T && !(m.rank == 0 && tid < 32))) continue;    // (warp-uniform)
        uint32_t key = 0xffffffffu;
        int cell = 0;
        if (owns(t)) {
            const int bx = (cid[t] & 0xffff) - 1, by = (cid[t] >> 16) - 1;
            if (bx >= 0 && bx < G && by >= 0 && by < G) {
                cell = bx * G + by;
                key = ((uint32_t)cell << 1) | (t == T ? 1u : 0u);
            }
        }
        const uint32_t peers = __match_any_sync(kFull, key);
        if (key != 0xffffffffu && (__ffs(peers) - 1) == (tid & 31)) {
            const int bx = cell / G, owner = bx / band;
            const uint32_t a = dsmem(sm.table + (bx - owner * band) * G + (cell - bx * G), (uint32_t)owner);
            const uint32_t old = dsmem_add_u32(a, (uint32_t)__popc(peers) << ((key & 1u) ? 16 : 0));
            if (old == 0u) addr[t] = a;
            cid[t] = cell;
        }
    }
    cluster_sync();     // every count is in
    float2* g2 = reinterpret_cast<float2*>(grid_e);
    const uint32_t ll = (uint32_t)lut_locusts(N);
#pragma unroll
    for (int t = 0; t <= T; ++t) {
        if (addr[t] == 0xffffffffu) continue;
        const uint32_t w = dsmem_ld_u32(addr[t]);
        const uint32_t nl = w & 0xffffu, na = w >> 16;
        const float vl = nl < ll ? sm.lut[nl] : __fdiv_rn((float)nl, (float)N);
        const float va = A > 0 ? (na < (uint32_t)lut_agents(A) ? sm.lut[ll + na] : __fdiv_rn((float)na, (float)A)) : 0.f;
        g2[cid[t]] = make_float2(vl, va);
    }
}

}  // namespace swarm
