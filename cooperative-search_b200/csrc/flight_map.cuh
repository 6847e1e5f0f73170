// Belief map of the flight variant: _update_prob_map + _percent_in_agent_viewrange (env/flight_env.py:275-303).
//
// The map of an env is stored as 4x4-cell TILES of 64 bytes (FlightParams::tiles per side; flight_common.cuh: tile_off):
// HBM moves 64-byte atoms, and an agent's disc (R = 7) covers ~11 tiles where it straddles ~17 atoms of a row-major
// map with 200-byte rows.  The reference classifies the 4 corners of every cell against every agent
// (2500 x 4 x n fp64 tests).  Here, per env and per sensing call ("job" = agent positions + cells of the targets that
// call found):
//  (1) corner classification by ROW INTERVALS: for agent a and integer corner row cx, the corner columns cy with
//      fl(fl((cx-ax)^2) + fl((cy-ay)^2)) < R^2 form an interval (the expression is monotone in |cy-ay|).  Its ends
//      come from one fp32 sqrt; only when an end lies within 1e-3 of an integer is the reference's exact fp64
//      predicate evaluated there.  One lane per (agent, corner row): <= 2R*n tasks.  The interval is OR-ed as a bit
//      mask into R[cx] (bit cy), the union over agents ("any agent", the `break` of :299-302).
//  (2) percent of cell (i,j) = popc of bits j,j+1 of R[i] and R[i+1]; touched <=> any of them set.  One lane per tile
//      row ORs its five corner rows and lists the touched tiles of that row (prefix sum over the env's lanes).
//  (3) sweep: the env's lanes walk the tile list, four lanes per tile, one float4 (4 cells of one map row) per lane
//      and four tiles in flight per lane; the 10 corner bits of a float4 index a 1024-entry table (32 KB, L1
//      resident) that yields the four weights corners/4 and the four "untouched" flags, and the update runs as
//      packed fp32 pairs (FMUL2 / FADD2 / FFMA2 + MUFU.RCP).  Untouched float4s are neither read nor written.
//  (4) the cells of targets found by THIS call become 1 where percent > 0 (:288-289), after the sweep.
// The fused form runs inside the thread-per-env step kernel (flight_tpe.cu): the env's 8 lanes just computed the
// positions, so the job never leaves shared memory.  Needs map_size <= 63 (one 64-bit mask per corner row) and
// n_agents <= 8; everything else takes flight_map_generic_kernel (per-cell corner tests, bit-identical results).
#pragma once
#include "flight_common.cuh"

#ifndef CS_MAP_U
#define CS_MAP_U 2             // measured on the c4 workload (tools/exp_c4.py): 2 loads in flight per lane at 12 CTAs per SM beat 4 at 10 / 12 / 14
#endif

namespace csf {

// ---- packed fp32 pairs (sm_100: FADD2 / FMUL2 / FFMA2) ----------------------------------------------------------
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 f2_sub(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tsub.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 f2_add(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\tfma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float f_max3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// two cells of belief_cell() at once
__device__ __forceinline__ float2 belief_pair(float2 pv, float2 w, float2 u, float qf, float ql) {
    const float2 qp = f2_fma(make_float2(qf, qf), pv, f2_mul(make_float2(ql, ql), pv));
    const float2 num = f2_mul(w, qp), keep = f2_mul(u, pv);
    const float2 den = f2_add(qp, f2_sub(make_float2(1.0f, 1.0f), pv));
    return f2_fma(num, make_float2(rcp_approx(den.x), rcp_approx(den.y)), keep);
}

// corners in view of cell k (0..3) of a float4 whose corner bits are idx = x0 | x1 << 5 (x0: corner row i, x1: row i+1)
__device__ __forceinline__ int f4_corners(unsigned idx, int k) { return __popc(idx & (0x63u << k)); }

// One float4 of cells: old values v, corner bits idx (!= 0).  Exact cases: a cell at exactly 1 -> exactly percent; with
// detect_prob = 1 (qf = 0: 0/0 = nan, like the reference) the untouched cells of the float4 keep their bits.
__device__ __forceinline__ float4 belief_f4(const FlightParams& p, float4 v, unsigned idx, float qf, float ql) {
    const float4 c = __ldg(p.lut_cells + 2 * idx), u = __ldg(p.lut_cells + 2 * idx + 1);
    const float2 lo = belief_pair(make_float2(v.x, v.y), make_float2(c.x, c.y), make_float2(u.x, u.y), qf, ql);
    const float2 hi = belief_pair(make_float2(v.z, v.w), make_float2(c.z, c.w), make_float2(u.z, u.w), qf, ql);
    float4 r = make_float4(lo.x, lo.y, hi.x, hi.y);
    if (qf == 0.0f) {
        r.x = (u.x != 0.0f) ? v.x : r.x; r.y = (u.y != 0.0f) ? v.y : r.y;
        r.z = (u.z != 0.0f) ? v.z : r.z; r.w = (u.w != 0.0f) ? v.w : r.w;
    } else if (fmaxf(f_max3(v.x, v.y, v.z), v.w) == 1.0f) {
        if (v.x == 1.0f && u.x == 0.0f) r.x = 0.25f * (float)f4_corners(idx, 0);
        if (v.y == 1.0f && u.y == 0.0f) r.y = 0.25f * (float)f4_corners(idx, 1);
        if (v.z == 1.0f && u.z == 0.0f) r.z = 0.25f * (float)f4_corners(idx, 2);
        if (v.w == 1.0f && u.w == 0.0f) r.w = 0.25f * (float)f4_corners(idx, 3);
    }
    return r;
}

// (1) of the header comment for task t = (agent, corner row) of one env: OR the agent's corner-column interval of that
// corner row into R.  xy: the job's agent positions, clo[a]: first corner row of agent a.
__device__ __forceinline__ void corner_interval_task(const FlightParams& p, int t, const double* xy, const int* clo,
                                                     unsigned long long* R) {
    const int M = p.M;
    const int a = t >> p.span_shift, r = t & (p.span_cap - 1);
    const double axa = xy[2 * a], aya = xy[2 * a + 1];
    const int cx = clo[a] + r;
    const double dx = (double)cx - axa;
    const double A = dx * dx;
    if (!(A < p.R2) || cx < 0 || cx > M) return;                     // past the last corner row of this agent
    // candidate ends in fp32 (ay <= map_size: absolute error ~4e-6, far inside the 1e-3 guard band)
    float wf;                                                        // approximate sqrt (2 ulp): far inside the guard band
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(wf) : "f"(fmaxf((float)(p.R2 - A), 0.0f)));
    const float ayf = (float)aya;
    const float yh = ayf + wf, yl = ayf - wf;
    float fh = floorf(yh), cl = ceilf(yl);
    if (yh - fh < 1e-3f || yh - fh > 1.0f - 1e-3f) {                 // end within 1e-3 of an integer: decide exactly
        const double Y = (double)rintf(yh);
        fh = (float)(corner_pred(A, Y, aya, p.R2) ? Y : Y - 1.0);
    }
    if (cl - yl < 1e-3f || cl - yl > 1.0f - 1e-3f) {
        const double Y = (double)rintf(yl);
        cl = (float)(corner_pred(A, Y, aya, p.R2) ? Y : Y + 1.0);
    }
    const int yhi = min((int)fh, M), ylo = max((int)cl, 0);
    if (ylo <= yhi) {
        const unsigned long long mk = ((2ull << yhi) - 1ull) & ~((1ull << ylo) - 1ull);
        unsigned* w = reinterpret_cast<unsigned*>(&R[cx]);
        if ((unsigned)mk) atomicOr(w, (unsigned)mk);
        if ((unsigned)(mk >> 32)) atomicOr(w + 1, (unsigned)(mk >> 32));
    }
}

// ------------------------------------------------------------------------------------------------
// Fused form: the GL lanes that own env e (consecutive lanes of one warp, kk = index inside the group) update its map
// for the `njobs` (0..2) sensing calls the step / reset code just stashed in the env's scratch S:
//   S + 0        R[M+2]        corner-row masks (u64)
//   S + fm_list  list[]        touched tiles (u16: tile row << 12 | tile col << 8 | linear tile index)
//   S + fm_clo   clo[n]        first corner row of each agent
//   S + fm_job   job[2]        { double xy[2n]; int nh; int hit[m]; } padded to fm_jobsz
// Every lane of the warp calls this (groups without a job idle through the warp barriers).
// ------------------------------------------------------------------------------------------------
template <int GL>
__device__ __forceinline__ void fused_map_phase(const FlightParams& p, int e, int kk, unsigned char* S, int njobs) {
    static_assert(GL == 4 || GL == 8 || GL == 16, "GL");
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int QP = GL / 4;                                       // tiles the group's lanes cover per float4 slot
    constexpr int U = CS_MAP_U;                                      // float4 loads in flight per lane
    const int n = p.n, M = p.M, TC = p.tiles;
    unsigned long long* R = reinterpret_cast<unsigned long long*>(S);
    unsigned short* list = reinterpret_cast<unsigned short*>(S + p.fm_list);
    int* clo = reinterpret_cast<int*>(S + p.fm_clo);
    float* map = p.prob_map + (size_t)e * p.map_stride;
    const float qf = (float)p.q_miss, ql = (float)(p.q_miss - (double)qf);      // q = 1-d as an fp32 pair
    const unsigned long long cellmask = (1ull << M) - 1ull;          // M <= 63
    const int r4 = kk & 3, quad = kk >> 2;
    unsigned touched = 0;

    for (int job = 0; job < 2; ++job) {
        const bool run = job < njobs;
        if (!__any_sync(FULL, run)) break;
        const double* xy = reinterpret_cast<const double*>(S + p.fm_job + job * p.fm_jobsz);
        const int* hit = reinterpret_cast<const int*>(xy + 2 * n);   // hit[0] = count, hit[1..] = cells
        __syncwarp();                                                // the job (written by the group's first lane) is visible; the previous job is done with R
        if (run) {
            for (int r = kk; r <= M + 1; r += GL) R[r] = 0ull;
            for (int a = kk; a < n; a += GL) {
                int lo, hi;
                corner_span(xy[2 * a], p.R, p.R2, &lo, &hi);
                clo[a] = lo;
            }
        }
        __syncwarp();
        // (1) corner-row intervals
        if (run)
            for (int t = kk; t < (n << p.span_shift); t += GL) corner_interval_task(p, t, xy, clo, R);
        __syncwarp();
        // (2) touched tiles: lane <-> tile row (GL lanes cover TC <= 16 rows in at most 4 rounds)
        int Nt = 0;
        for (int tr0 = 0; tr0 < TC; tr0 += GL) {                     // warp-uniform trip count
            const int tr = tr0 + kk;
            unsigned long long G = 0ull;
            if (run && tr < TC) {
                const int i0 = 4 * tr, ihi = min(i0 + 4, M);         // cell rows i0..i0+3 (< M) use corner rows i0..ihi
                unsigned long long Uo = 0ull;
                for (int c = i0; c <= ihi; ++c) Uo |= R[c];
                const unsigned long long Tm = (Uo | (Uo >> 1)) & cellmask;       // cells of these rows with percent > 0
                G = (Tm | (Tm >> 1) | (Tm >> 2) | (Tm >> 3)) & 0x1111111111111111ull;   // bit 4*tc: tile column tc is touched
            }
            const int cnt = __popcll(G);
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < GL; o <<= 1) {
                const int v = __shfl_up_sync(FULL, incl, o, GL);
                if (kk >= o) incl += v;
            }
            int pos = Nt + incl - cnt;
            for (; G; G &= G - 1ull) {
                const int tc = (__ffsll((long long)G) - 1) >> 2;
                list[pos++] = (unsigned short)((tr << 12) | (tc << 8) | (tr * TC + tc));
            }
            Nt += __shfl_sync(FULL, incl, GL - 1, GL);
        }
        __syncwarp();
        // (3) sweep: slot s of the list <-> tile s, lane r4 of a quad <-> map row 4*tr + r4 of that tile
        if (run) {
            for (int t0 = 0; t0 < Nt; t0 += QP * U) {
                float4 v[U];
                unsigned idx[U];
                int off[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int ti = t0 + u * QP + quad;
                    idx[u] = 0u;
                    off[u] = 0;
                    if (ti < Nt) {
                        const unsigned ent = list[ti];
                        const int i = 4 * (int)(ent >> 12) + r4, j0 = 4 * (int)((ent >> 8) & 15u);
                        if (i < M) {
                            const unsigned x0 = (unsigned)(R[i] >> j0) & 0x1Fu, x1 = (unsigned)(R[i + 1] >> j0) & 0x1Fu;
                            idx[u] = x0 | (x1 << 5);                 // 0: no cell of this float4 has a corner in view (:285-286)
                            off[u] = (int)(ent & 255u) * 16 + r4 * 4;
                        }
                    }
                    if (idx[u]) v[u] = __ldcg(reinterpret_cast<const float4*>(map + off[u]));
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (idx[u]) __stcg(reinterpret_cast<float4*>(map + off[u]), belief_f4(p, v[u], idx[u], qf, ql));
            }
        }
        __syncwarp();                                                // sweep stores before the stores below (same cells)
        // (4) targets found by THIS call -> 1 where the cell has a corner in view (:288-289)
        if (run) {
            const int nh = hit[0];
            for (int h = kk; h < nh; h += GL) {
                const int cell = hit[1 + h];
                if (cell < 0) continue;
                const int ci = cell / M, cj = cell - ci * M;
                if (((unsigned)(R[ci] >> cj) | (unsigned)(R[ci + 1] >> cj)) & 3u) map[tile_off(TC, ci, cj)] = 1.0f;
            }
            if (p.count_touched)
                for (int i = kk; i < M; i += GL) {
                    const unsigned long long a = R[i], b = R[i + 1];
                    touched += __popcll((a | (a >> 1) | b | (b >> 1)) & cellmask);
                }
        }
    }
    if (p.count_touched) {
        const unsigned tot = __reduce_add_sync(FULL, touched);
        if ((threadIdx.x & 31) == 0 && tot) atomicAdd(p.stats + CS_STAT_TOUCHED, (double)tot);
    }
}

// ------------------------------------------------------------------------------------------------
// Two-kernel form: flight_map_tile_kernel runs after the thread-per-env step / reset kernel (flight_tpe.cu), which
// left one job record per env in FlightParams::jobs (header {jobs, fill flag}, up to two job slots).  GL = 16 lanes own
// one env: they copy the record into the env's shared-memory scratch and run fused_map_phase on it.  On its own the
// map update needs no fp64 state and no Philox: few registers, many resident warps, which is what covers the
// latency of the scattered 64-byte tile accesses.  With cs_flight_cfg.map_overlap the kernel runs on the handle's own
// stream, concurrently with the step kernel of the NEXT call (flight_host.cu).
// ------------------------------------------------------------------------------------------------
#ifdef CS_MAP_KERNELS           // instantiated by flight_mapk.cu only
constexpr int kMapThreads = 128;
#ifndef CS_TILE_LANES
#define CS_TILE_LANES 16
#endif
constexpr int kTileLanes = CS_TILE_LANES;
#ifndef CS_MAP_MIN_CTAS
#define CS_MAP_MIN_CTAS 12
#endif

static __global__ void __launch_bounds__(kMapThreads, CS_MAP_MIN_CTAS) flight_map_tile_kernel(const __grid_constant__ FlightParams p) {
    constexpr int GL = kTileLanes;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char tsm[];
    const int grp = threadIdx.x / GL, kk = threadIdx.x % GL;
    const int e_raw = blockIdx.x * (kMapThreads / GL) + grp;
    const int e = min(e_raw, p.E - 1);
    const unsigned char* rec = p.jobs + (size_t)e * p.job_stride;
    const int2 hdr = *reinterpret_cast<const int2*>(rec);
    const int njobs = e_raw < p.E ? hdr.x : 0;
    const bool fill = e_raw < p.E && hdr.y != 0;
    if (!__any_sync(FULL, njobs != 0 || fill)) return;
    unsigned char* S = tsm + (size_t)grp * p.fm_env;
    if (fill) {                                                      // reset(init=True): prob_map <- 0.5 (flight_env.py:84-86), tiles incl. padding
        float4* m4 = reinterpret_cast<float4*>(p.prob_map + (size_t)e * p.map_stride);
        for (int c = kk; c < p.map_stride / 4; c += GL) m4[c] = make_float4(0.5f, 0.5f, 0.5f, 0.5f);
    }
    {
        const uint4* src = reinterpret_cast<const uint4*>(rec + 16);
        uint4* dst = reinterpret_cast<uint4*>(S + p.fm_job);
        for (int c = kk; c < njobs * (p.fm_jobsz / 16); c += GL) dst[c] = src[c];
    }
    fused_map_phase<GL>(p, e, kk, S, njobs);                         // its first __syncwarp orders the fill and the copy
}

// ------------------------------------------------------------------------------------------------
// Generic form (any map_size, any n_agents): its own kernel after the lane-per-agent step / reset kernel, one warp
// per env, per-cell corner tests in fp64 like the reference.  The step kernel leaves a job for every env it sensed: a
// non-zero meta word CS_META_SENSE (cleared again by the next call that does not sense the env), the agent positions
// in the state record, the targets found by that call in CS_META_NEWFOUND; an env that was auto-reset inside the call
// was sensed twice (flight_env.py:266 runs inside reset() too) and its first job -- positions and hit cells before
// the reset -- sits in the `pre` side buffer.  Same cell arithmetic as the fused form: bit-identical maps.
// ------------------------------------------------------------------------------------------------
// Loads job `job` of env e into the warp's scratch: agent positions -> xy[2n], hit cells -> hit[]; returns the number
// of hit cells.  job 0 = the sensing before an in-call auto-reset (side buffer), job 1 = the state record as the step
// / reset kernel left it.
template <int GL>
__device__ __forceinline__ int map_job_load(const FlightParams& p, int e, int job, int lane, uint32_t newf, double* xy, int* hit) {
    const int n = p.n, m = p.m;
    int nh;
    if (job == 0) {
        const double* pj = p.pre + (size_t)e * p.pre_stride;
        for (int a = lane; a < n; a += GL) {
            const double2 v = reinterpret_cast<const double2*>(pj)[a];
            xy[2 * a] = v.x; xy[2 * a + 1] = v.y;
        }
        const int* ph = reinterpret_cast<const int*>(pj + 2 * n);
        nh = ph[0];
        for (int k = lane; k < nh; k += GL) hit[k] = ph[1 + k];
    } else {
        for (int a = lane; a < n; a += GL) {
            const double2 v = xy_ld(p, a, e);
            xy[2 * a] = v.x; xy[2 * a + 1] = v.y;
        }
        nh = __popc(newf);
        for (int j = lane; j < m; j += GL)
            if ((newf >> j) & 1u) {
                const double2 t = tgt_ld(p, j, e);
                hit[__popc(newf & ((1u << j) - 1u))] = hit_cell(p, t.x, t.y);
            }
    }
    return nh;
}

static __global__ void __launch_bounds__(kMapThreads) flight_map_generic_kernel(const __grid_constant__ FlightParams p, uint32_t seq) {
    extern __shared__ __align__(16) unsigned long long msm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * (kMapThreads / 32) + warp;
    if (e >= p.E) return;
    const int n = p.n, M = p.M;
    uint4 m0, m1;
    meta_ld(p, e, &m0, &m1);
    if ((m1.w >> 1) != seq) return;
    unsigned long long* S = msm + (size_t)warp * p.ms_warp;
    int4* box = reinterpret_cast<int4*>(S + p.ms_box);
    double* xy = reinterpret_cast<double*>(S + p.ms_xy);
    int* hit = reinterpret_cast<int*>(S + p.ms_hit);
    float* map = p.prob_map + (size_t)e * p.map_stride;
    const float qf = (float)p.q_miss, ql = (float)(p.q_miss - (double)qf);
    const int colk = lane & 15, half = lane >> 4;
    unsigned touched = 0;
    for (int job = (m1.w & 1u) ? 0 : 1; job < 2; ++job) {
        const int nh = map_job_load<32>(p, e, job, lane, m0.y, xy, hit);
        __syncwarp();
        if (lane < n) {
            int lo, hi;
            corner_span(xy[2 * lane], p.R, p.R2, &lo, &hi);
            const int i0 = max(0, lo - 1), i1 = min(M - 1, hi);
            corner_span(xy[2 * lane + 1], p.R, p.R2, &lo, &hi);
            box[lane] = make_int4(i0, i1, max(0, lo - 1), min(M - 1, hi));
        }
        __syncwarp();
        for (int a = 0; a < n; ++a) {
            const int4 bx = box[a];
            for (int jc = bx.z; jc <= bx.w; jc += 16) {
                const int j = jc + colk;
                if (j > bx.w) continue;
                const double y0 = (double)j, y1 = (double)(j + 1);
                for (int i = bx.x + half; i <= bx.y; i += 2) {
                    bool mine = true;
                    for (int b = 0; b < a; ++b) {
                        const int4 bb = box[b];
                        mine &= !(i >= bb.x && i <= bb.y && j >= bb.z && j <= bb.w);
                    }
                    if (!mine) continue;
                    const double x0 = (double)i, x1 = (double)(i + 1);
                    uint32_t bits = 0;
                    for (int q = 0; q < n; ++q) {
                        const double qx = xy[2 * q], qy = xy[2 * q + 1];
                        const double dx0 = x0 - qx, dx1 = x1 - qx, dy0 = y0 - qy, dy1 = y1 - qy;
                        const double sx0 = dx0 * dx0, sx1 = dx1 * dx1, sy0 = dy0 * dy0, sy1 = dy1 * dy1;
                        bits |= (sx0 + sy0 < p.R2) ? 1u : 0u;
                        bits |= (sx1 + sy0 < p.R2) ? 2u : 0u;
                        bits |= (sx0 + sy1 < p.R2) ? 4u : 0u;
                        bits |= (sx1 + sy1 < p.R2) ? 8u : 0u;
                    }
                    if (!bits) continue;                                      // percent == 0 -> untouched (:285-286)
                    ++touched;
                    const int cnt = __popc(bits);
                    float* cellp = map + tile_off(p.tiles, i, j);
                    const float pv = *cellp;
                    float v = belief_cell(pv, 0.25f * (float)cnt, 0.0f, qf, ql);
                    if (pv == 1.0f && qf != 0.0f) v = 0.25f * (float)cnt;    // see belief_cell: the exact case
                    for (int k = 0; k < nh; ++k)
                        if (hit[k] == i * M + j) v = 1.0f;                    // found by THIS call (:288-289)
                    *cellp = v;
                }
            }
        }
        __syncwarp();
    }
    if (p.count_touched) {
        const unsigned tot = __reduce_add_sync(0xffffffffu, touched);
        if (lane == 0 && tot) atomicAdd(p.stats + CS_STAT_TOUCHED, (double)tot);
    }
}

#endif  // CS_MAP_KERNELS

}  // namespace csf
