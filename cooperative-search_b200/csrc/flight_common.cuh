// Shared device code of the flight_easy / flight kernels (B200, sm_100a): parameter block, state accessors,
// heading trig table, wall handling, reset-time target placement, belief-cell arithmetic, tiled map addressing.
//
// What is restated in the flight_*.cu files (reference: WZN1ng/Cooperative-Search, pure Python):
//   _agent_step + _potential_energy_force   env/flight_env_easy.py:255-301, env/flight_env.py:305-355
//   _update_obs (detection, reward, win)    env/flight_env_easy.py:223-253, env/flight_env.py:232-266
//   _update_prob_map / _percent_in_...      env/flight_env.py:275-303
//   step / reset / get_obs / get_state      env/flight_env_easy.py:79-221,303-314
//
// Files (DESIGN.md section 4 has the full account):
//   flight_tpe.cu   thread-per-env step / reset kernels (n_agents <= 8; the default), the grouped step of many handles,
//                   and the FUSED step + belief-map kernel of the flight variant (8 lanes per env)
//   flight_lpa.cu   lane-per-agent step / reset kernel (n_agents > 8 or lanes_per_env >= 16)
//   flight_map.cuh  belief-map update: the fused phase (row-interval corner masks, touched 4x4 tiles, float4 sweep) and
//                   the generic per-cell kernel
//   flight_aux.cu   map observation (de-tiling, TMA bulk stores), map export / import, episode-batch writer, statistics
//   flight_host.cu  cs_flight handle, C ABI
// Positions / headings / targets are fp64 so that the in-range test and the wall test take the same branch as the
// reference's Python floats; everything is compiled with -fmad=false so a*b+c keeps the reference's two roundings.
// Detection draws are keyed Philox words (cs_philox.cuh), order independent.
#pragma once
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include "cs_common.cuh"
#include "cs_philox.cuh"

namespace csf {

constexpr int kThreads = 128;          // lane-per-agent kernel
struct FlightParams {
    int E, n, m, M, T;
    int variant, auto_reset, agent_mode, target_mode, count_touched;
    // per-env record geometry (doubles)
    int rec, yaw_off, meta_off, state_len;
    long long dyn_rs, dyn_es, tgt_rs, tgt_es;   // strides (in doubles) of a row / an env in dyn and tgt
    int state_stride;            // floats per state row in HBM (state_len rounded up to a multiple of 4)
    int s_lut, s_warp;           // lane-per-agent kernel: per-warp shared-memory scratch (doubles) for the heading-table index
    int span_cap, span_shift;    // power of two >= 2R: corner rows per agent in the interval pass (and its log2)
    // belief map, stored as 4x4-cell tiles of 64 bytes: cell (i, j) of env e lives at
    // prob_map[e*map_stride + ((i>>2)*tiles + (j>>2))*16 + (i&3)*4 + (j&3)], tiles = ceil(M/4) per side
    int tiles, map_stride;
    // tiled map update (fused kernel / flight_map_tile_kernel): per-env shared-memory scratch, offsets / sizes in bytes
    int fm_list, fm_clo, fm_job, fm_jobsz, fm_env;
    // two-kernel form: belief-map job records the step / reset kernel leaves for flight_map_tile_kernel, one per env:
    // int2 {jobs (0..2), fill flag} at +0, job slots of fm_jobsz bytes from +16.  Double buffered by the host (the step
    // kernel of call t+1 may run while the map kernel of call t still reads): `jobs` is the buffer of THIS launch.
    unsigned char* jobs;
    int job_stride;
    // generic map kernel: per-warp scratch offsets / size in 8-byte words
    int ms_box, ms_xy, ms_hit, ms_warp;
    int pre_stride;              // doubles per env in `pre`
    double* pre;                 // [E][pre_stride]: agent xy (2n) | int nh, hit cells -- the sensing before an in-call auto-reset (generic map path)
    double Md, half_M, inv_half, R, R2, v, fk, fd2, near2, q_miss;
    double turn, pi, two_pi, three_pi, half_pi;
    long long thr;
    uint32_t seed, env_id_base;
    double* dyn;
    double* tgt;
    float* obs;
    float* state;
    float* reward;
    uint8_t* terminated;
    uint8_t* win;
    int32_t* target_find;
    float* prob_map;
    double* stats;
    const double* tmpl;   // [m][5]: x, y, sx, sy, random   (already scaled by a = M/10)
    const float4* lut_cells;     // [1024][2]: corner bits of a float4 of cells -> (corners-in-view * (1-d)/4) x4, (untouched ? 1 : 0) x4
    // heading-lattice trig table (see HeadingLut in flight_host.cu)
    const longlong2* lut_meta;   // [37]: x = bit pattern of the cluster centre, y = base | (half << 32)
    const double2* lut;          // (sin, cos) of every bit pattern in every cluster window, from the HOST libm
    double inv_turn;             // 18/pi
    double cos0, sin0;           // cos/sin of the start heading of agent_mode, from the host libm
    double lin[CS_MAX_AGENTS];   // i*map_size/(n-1) (map_size/2 for n == 1), flight_env_easy.py:140-143
};

enum { MODE_STEP = 0, MODE_RESET = 1 };

// ------------------------------------------------------------------------------------------------
// State layout, chosen per handle (cs_flight_create): element (row r, env e) of dyn lives at dyn[r*dyn_rs + e*dyn_es],
// of tgt at tgt[r*tgt_rs + e*tgt_es].  Rows of dyn: 0..2n-1 = x0, y0, x1, y1, ..., 2n..3n-1 the headings,
// meta_off..meta_off+3 the 8 uint32 meta words (two per row); rows of tgt: 2j = x of target j, 2j+1 = y.
//   * structure of arrays (rs = E, es = 1), from 32768 envs per handle (= one thread per env, flight_tpe_kernel<N, 1>): with one thread per env every load and store
//     of a warp is one contiguous 256-byte run (the record layout cost the thread-per-env kernel ~1100 L1 wavefronts
//     per warp and bounded it: 1M envs 5.05e9 -> 5.5e9, 65536 envs 2.67e9 -> 2.9e9 env-steps/s);
//   * record per env (rs = 1, es = rows), below: a launch of a few thousand envs is latency-bound and 12 % faster
//     when a warp's state is a handful of consecutive lines instead of 43 rows 32 KB apart.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double* dyn_at(const FlightParams& p, int row, int e) {
    return p.dyn + (size_t)row * p.dyn_rs + (size_t)e * p.dyn_es;
}
// record layout (row stride 1): pairs of rows are adjacent and 16-byte aligned -> one 16-byte access
__device__ __forceinline__ double2 xy_ld(const FlightParams& p, int a, int e) {
    const double* q = dyn_at(p, 2 * a, e);
    if (p.dyn_rs == 1) return *reinterpret_cast<const double2*>(q);
    return make_double2(q[0], q[p.dyn_rs]);
}
__device__ __forceinline__ void xy_st(const FlightParams& p, int a, int e, double x, double y) {
    double* q = dyn_at(p, 2 * a, e);
    if (p.dyn_rs == 1) { *reinterpret_cast<double2*>(q) = make_double2(x, y); return; }
    q[0] = x;
    q[p.dyn_rs] = y;
}
__device__ __forceinline__ double2 tgt_ld(const FlightParams& p, int j, int e) {
    const double* t = p.tgt + (size_t)(2 * j) * p.tgt_rs + (size_t)e * p.tgt_es;
    if (p.tgt_rs == 1) return *reinterpret_cast<const double2*>(t);
    return make_double2(t[0], t[p.tgt_rs]);
}
__device__ __forceinline__ void tgt_st(const FlightParams& p, int j, int e, double2 v) {
    double* t = p.tgt + (size_t)(2 * j) * p.tgt_rs + (size_t)e * p.tgt_es;
    if (p.tgt_rs == 1) { *reinterpret_cast<double2*>(t) = v; return; }
    t[0] = v.x;
    t[p.tgt_rs] = v.y;
}
__device__ __forceinline__ uint2* meta_at(const FlightParams& p, int pair, int e) {       // words 2*pair, 2*pair+1
    return reinterpret_cast<uint2*>(dyn_at(p, p.meta_off + pair, e));
}
__device__ __forceinline__ void meta_ld(const FlightParams& p, int e, uint4* m0, uint4* m1) {
    if (p.dyn_rs == 1) {
        const uint4* mp = reinterpret_cast<const uint4*>(dyn_at(p, p.meta_off, e));
        *m0 = mp[0]; *m1 = mp[1];
        return;
    }
    const uint2 a = *meta_at(p, 0, e), b = *meta_at(p, 1, e), c = *meta_at(p, 2, e), d = *meta_at(p, 3, e);
    *m0 = make_uint4(a.x, a.y, b.x, b.y);
    *m1 = make_uint4(c.x, c.y, d.x, d.y);
}
__device__ __forceinline__ void meta_st(const FlightParams& p, int e, uint4 m0, uint4 m1) {
    if (p.dyn_rs == 1) {
        uint4* mp = reinterpret_cast<uint4*>(dyn_at(p, p.meta_off, e));
        mp[0] = m0; mp[1] = m1;
        return;
    }
    *meta_at(p, 0, e) = make_uint2(m0.x, m0.y);
    *meta_at(p, 1, e) = make_uint2(m0.z, m0.w);
    *meta_at(p, 2, e) = make_uint2(m1.x, m1.y);
    *meta_at(p, 3, e) = make_uint2(m1.z, m1.w);
}

// ------------------------------------------------------------------------------------------------
// cos/sin of a heading.
//
// Headings only ever take the values reachable from {0, pi/2, pi} under +-pi/18 turns, the 2*pi wrap and
// the wall reflection (flight_env_easy.py:259-266,281-284): 37 clusters of fp64 values, each a few hundred
// ulps wide after 200 steps (rounding drift ~1.7e-16 per step).  Whether an agent that comes back to a
// wall ends at y = 0.0 or y = -5e-17 -- and therefore its out-of-map flag, its reward and its reflected
// heading -- depends on the LAST BIT of sin/cos, and the reference's bits are those of the host libm
// (numpy -> glibc), which is not correctly rounded (measured: 2 of 652 evaluations).  So the handle tabulates
// the host libm's sin/cos for every bit pattern in every cluster window at create time and the kernel looks
// the pair up (one 16-byte load) -- bit-identical to the reference and cheaper than evaluating sincos().
// Off-lattice headings (user-injected state) fall back to CUDA's sincos (<= 2 ulp).
// ------------------------------------------------------------------------------------------------
// (returns by value: results handed back through pointers would live in local memory for every lookup)
static __device__ __noinline__ double2 offlattice_sincos(double h) {
    double sn, c;
    sincos(h, &sn, &c);
    return make_double2(sn, c);
}

// (sin, cos) of heading h
__device__ __forceinline__ double2 heading_sincos(const FlightParams& p, const longlong2* lutm, double h) {
    const int k = __double2int_rn(h * p.inv_turn);
    if (k == 0 && fabs(h) < 7.450580596923828e-09) return make_double2(h, 1.0);   // |h| < 2^-27: libm returns sin = h, cos = 1
    if (k >= 1 && k <= 36) {
#ifdef CS_LUTM_STAGED
        const longlong2 mt = lutm[k];                      // cluster index staged in shared memory by the CTA
#else
        // the 37-entry cluster index straight from L1 (every warp of the SM reads the same 592 bytes).  Staging it in shared
        // memory per CTA costs 37 loads and a block barrier before the first state load: measured +2..3 % on the grouped
        // c2 launch and on c3 without it, -1 % on the 1M-env launch.
        const longlong2 mt = __ldg(p.lut_meta + k);
#endif
        const long long off = __double_as_longlong(h) - mt.x;
        const long long half = mt.y >> 32;
        if (off >= -half && off <= half) return __ldg(p.lut + ((mt.y & 0xffffffffLL) + half + off));
    }
    return offlattice_sincos(h);
}

// ------------------------------------------------------------------------------------------------
// wall handling of one agent: env/flight_env_easy.py:278-290 ('>' test), env/flight_env.py:328 ('>=')
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool wall_reg(const FlightParams& p, double& x, double& y, double& h, double& c) {
    const double Md = p.Md;
    const bool outside = p.variant ? (x < 0.0 || x >= Md || y < 0.0 || y >= Md)
                                   : (x < 0.0 || x > Md || y < 0.0 || y > Md);
    if (outside) {
        x = fmin(fmax(x, 0.0), Md);
        y = fmin(fmax(y, 0.0), Md);
        h = (h <= p.pi) ? (p.pi - h) : (p.three_pi - h);
        c = -c;   // cos(pi - h) = cos(3pi - h) = -cos(h); sin unchanged (only the fp32 outputs use them)
    }
    return outside;
}

// Reset-time target placement (env/flight_env_easy.py:95-127) from the keyed stream; cold, out of line.
static __device__ __noinline__ double2 draw_target(const FlightParams& p, const double* tmpl, uint32_t seed, uint32_t env_id, uint32_t episode, int j) {
    const cs_u4 w = cs_philox4x32_10(env_id, (episode & 0xFFFFu) << 16, (uint32_t)j, 0u, seed, cs_stream_key(CS_STREAM_TARGET, episode));
    const double u1 = cs_u53(w.x, w.y), u2 = cs_u53(w.z, w.w);
    double x, y;
    if (p.target_mode == 0) {
        const double* row = tmpl + 5 * j;
        x = row[0];
        y = row[1];
        if (row[4] != 0.0) {                      // deter == 'f' (:106-110)
            const double rad = sqrt(-2.0 * log(u1));
            double sn, c;
            sincos(2.0 * p.pi * u2, &sn, &c);
            x += row[2] * 2.0 * (rad * c - 0.5);
            y += row[3] * 2.0 * (rad * sn - 0.5);
        }
    } else {                                      // target_mode 1 (:122-127)
        x = p.Md * u1;
        y = p.Md * u2;
    }
    return make_double2(x, y);
}

// Integer corner coordinates c with fl((c - a)^2) < R^2 -- a necessary condition for a corner in that
// row/column to be inside the agent's disc, evaluated with the SAME floating-point expression as the corner test
// (an agent at x = 1.0000000000000004 has corner x = 4 inside although fl(x + 3) = 4.0; bounds derived from
// floor/ceil of a +- R alone lose such corners).  Returns [lo, hi], at most 2R wide.
__device__ __forceinline__ void corner_span(double a, double R, double R2, int* lo, int* hi) {
    int c = (int)floor(a - R);
    double d = (double)c - a;
    *lo = (d * d < R2) ? c : c + 1;
    c = (int)ceil(a + R);
    d = (double)c - a;
    *hi = (d * d < R2) ? c : c - 1;
}

__device__ __forceinline__ bool corner_pred(double A, double cy, double ay, double R2) {
    const double dy = cy - ay;
    return A + dy * dy < R2;                                   // strict '<' (:300)
}

// cell of a target found by the sensing call: [min(int(x), M-1), min(int(y), M-1)], Python int() truncates toward
// zero (flight_env.py:279); negative indices never match a swept cell
__device__ __forceinline__ int hit_cell(const FlightParams& p, double tx, double ty) {
    const int ci = min((int)fmin(tx, p.Md), p.M - 1), cj = min((int)fmin(ty, p.Md), p.M - 1);
    return (ci < 0 || cj < 0) ? -1 : ci * p.M + cj;
}

// float offset of cell (i, j) inside an env's tiled map
__host__ __device__ __forceinline__ int tile_off(int tiles, int i, int j) {
    return (((i >> 2) * tiles + (j >> 2)) << 4) + ((i & 3) << 2) + (j & 3);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// One cell of the belief update (flight_env.py:291-292), p' = percent*(1-d)*p / ((1-d)*p + (1-p)), fp32 and branch
// free: w = corners-in-view / 4 (exact; 0 for an untouched cell), u = 1 for an untouched cell else 0, so that
// r = (w*qp) * rcp(den) + u*p is the update for a touched cell and p itself for an untouched one.  q = 1-d enters as
// the pair qf + ql (qf = fl32(q), ql = fl32(q - qf)), so that qp is q*p to fp32 accuracy: q rounded to fp32 alone
// would shift every update by |fl32(q) - q| / q in the same direction (1.5e-8 at d = 0.9, 1.3e-8 at d = 0.05), and
// a cell collects that once per call for as long as it stays in view (DESIGN section 4.4).  The reference's own
// grouping (1-d)*p + (1-p) matters: 1-p is exact near p = 1.  A cell at exactly 1 (a found target) must map to
// exactly percent -- in particular stay exactly 1 while all four corners are in view -- because the map's derivative
// there is 1/q and any seed error would grow by that factor per step; the callers take that case exactly
// (values never approach 1 from below: p' <= p).  The fused kernel evaluates the same operations two cells at a time
// (FMUL2 / FADD2 / FFMA2), bit for bit the same results.
__device__ __forceinline__ float belief_cell(float pv, float w, float u, float qf, float ql) {
    const float qp = fmaf(qf, pv, ql * pv);                     // (1-d)*p
    const float num = w * qp;                                   // percent*(1-d)*p
    const float keep = u * pv;
    const float den = qp + (1.0f - pv);                         // (1-d)*p + (1-p)
    return fmaf(num, rcp_approx(den), keep);
}

}  // namespace csf
