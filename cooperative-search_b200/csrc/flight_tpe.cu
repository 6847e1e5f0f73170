// Thread-per-env step / reset kernels of flight_easy / flight (n_agents <= 8), the grouped step of many handles, and
// the fused step + belief-map kernel of the flight variant.  See flight_common.cuh for the file map.
// Compiled once per CS_TPE_PART (0..3): part P instantiates n_agents = 2P+1 and 2P+2 (parallel builds).
#include "flight_internal.h"
#include "flight_map.cuh"

#ifndef CS_TPE_PART
#error "compile with -DCS_TPE_PART=0..3"
#endif

namespace csf {
namespace {

// ------------------------------------------------------------------------------------------------
// The step / reset kernel, THREAD-PER-ENV form (n_agents <= kTpeMaxAgents; the default).
//
// flight_kernel above spends ~380 warp instructions per env-step with most lanes idle in the agent phases and every
// reduction a shuffle or a ballot: on B200 that is issue-bound at 14 % of the HBM roofline.  Here one THREAD owns one
// env: agent state lives in registers (arrays indexed by compile-time constants), the targets stream through from
// global memory, the agents x targets test and the reward are plain loops, and nothing is exchanged between lanes --
// a warp advances 32 envs per instruction.  K > 1 splits the long part, the loop over the targets, over K threads
// that each repeat the (short) agent phase: the same latency as flight_kernel with 32/K envs per warp, for launches too
// small to fill the GPU with one thread per env.  Only the rare heavy pieces are warp-cooperative: the Box-Muller target
// redraw of a reset env (one lane per target) and the 0.5 fill of a belief map.
// Same arithmetic, same operation order, same Philox counters as flight_kernel: the two are interchangeable bit for
// bit (tests/test_gpu_flight_easy.py compares them).
//   pass 0 (STEP): _agent_step -> _update_obs -> step bookkeeping            (flight_env_easy.py:255-314)
//   pass 1       : reset (selected envs in RESET mode; just-terminated envs under auto_reset) -> _update_obs (:79-182)
// MAP (the flight variant, K = 8): every sensing call also stashes a belief-map job (agent positions, cells of the
// targets it found) in the env's shared-memory scratch; the fused kernel runs fused_map_phase on them afterwards.
// ------------------------------------------------------------------------------------------------
#ifndef CS_TPE_TU
#define CS_TPE_TU 5            // targets a thread loads together in the sensing loop
#endif
#ifndef CS_TPE_MIN_CTAS
#define CS_TPE_MIN_CTAS 8      // resident CTAs per SM the thread-per-env kernel is compiled for (register budget 65536/(64*N))
#endif
// One thread per env with the targets staged in shared memory (StagedView): up to three agents fit 10 CTAs per SM (102
// registers) without spills when the sensing loop takes one target at a time -- measured on B200 with variant libraries
// (tools/build_variant.sh): 1M envs 5.5e9 -> 6.2e9 env-steps/s, the grouped c2 launch 4.79e9 -> 4.83e9; with five agents
// the same setting spills (65536 envs: 3.15e9 -> 2.78e9), so larger teams keep 8 CTAs and blocks of CS_TPE_TU targets.
#ifndef CS_TPE_SMALL_CTAS
#define CS_TPE_SMALL_CTAS 10
#endif
constexpr int tpe_min_ctas(int N, int K, int mode) { return (K == 1 && mode == 0 && N <= 3) ? CS_TPE_SMALL_CTAS : CS_TPE_MIN_CTAS; }

// Where a thread finds its env's state.  GlobalView: straight from HBM, layout known at compile time (structure of arrays with
// one thread per env, record per env otherwise).  StagedView (below): the same, with the target rows staged in shared memory.
// What differs between the handles of a grouped launch comes from `g` (kernel parameter space), the rest from `p`.
template <bool SOA>
struct GlobalView {
    static constexpr bool kStaged = false;
    struct Ctx {};
    const FlightParams& p; const GroupEntry& g; int e;
    __device__ __forceinline__ GlobalView(const FlightParams& p_, const GroupEntry& g_, int e_, Ctx) : p(p_), g(g_), e(e_) {}
    __device__ __forceinline__ double* dynp(int row) const { return SOA ? g.dyn + (size_t)row * g.E + e : g.dyn + (size_t)e * p.rec + row; }
    __device__ __forceinline__ double2 xy_ld(int a) const {
        if (SOA) { const double* q = dynp(2 * a); return make_double2(q[0], q[g.E]); }
        return *reinterpret_cast<const double2*>(dynp(2 * a));
    }
    __device__ __forceinline__ void xy_st(int a, double x, double y) const {
        if (SOA) { double* q = dynp(2 * a); q[0] = x; q[g.E] = y; return; }
        *reinterpret_cast<double2*>(dynp(2 * a)) = make_double2(x, y);
    }
    __device__ __forceinline__ double yaw_ld(int a) const { return *dynp(p.yaw_off + a); }
    __device__ __forceinline__ void yaw_st(int a, double v) const { *dynp(p.yaw_off + a) = v; }
    __device__ __forceinline__ double2 tgt_ld(int j) const {
        if (SOA) { const double* t = g.tgt + (size_t)(2 * j) * g.E + e; return make_double2(t[0], t[g.E]); }
        return *reinterpret_cast<const double2*>(g.tgt + ((size_t)e * p.m + j) * 2);
    }
    // reset: target j of env `es` (owned by lane `src` of this warp), written by the lane that drew it
    __device__ __forceinline__ void tgt_publish(int j, int es, int /*src*/, double2 v) const {
        if (SOA) { double* t = g.tgt + (size_t)(2 * j) * g.E + es; t[0] = v.x; t[g.E] = v.y; return; }
        *reinterpret_cast<double2*>(g.tgt + ((size_t)es * p.m + j) * 2) = v;
    }
    __device__ __forceinline__ void meta_ld(uint4* m0, uint4* m1) const {
        if (SOA) {
            const uint2* q = reinterpret_cast<const uint2*>(dynp(p.meta_off));
            const uint2 a = q[0], b = q[g.E], c = q[2 * (size_t)g.E], d = q[3 * (size_t)g.E];
            *m0 = make_uint4(a.x, a.y, b.x, b.y);
            *m1 = make_uint4(c.x, c.y, d.x, d.y);
            return;
        }
        const uint4* mp = reinterpret_cast<const uint4*>(dynp(p.meta_off));
        *m0 = mp[0]; *m1 = mp[1];
    }
    __device__ __forceinline__ void meta_st(uint4 m0, uint4 m1) const {
        if (SOA) {
            uint2* q = reinterpret_cast<uint2*>(dynp(p.meta_off));
            q[0] = make_uint2(m0.x, m0.y); q[g.E] = make_uint2(m0.z, m0.w);
            q[2 * (size_t)g.E] = make_uint2(m1.x, m1.y); q[3 * (size_t)g.E] = make_uint2(m1.z, m1.w);
            return;
        }
        uint4* mp = reinterpret_cast<uint4*>(dynp(p.meta_off));
        mp[0] = m0; mp[1] = m1;
    }
    // the targets are needed after the agent phase: start pulling this warp's target rows into L1 together with the
    // state loads, so that the sensing loop pays no further HBM round trip
    template <int K>
    __device__ __forceinline__ void prefetch_targets(int kk) const {
        const int m = p.m;
        if (SOA) {
            const double* tp = g.tgt + e;
            for (int r = 0; r < 2 * m; ++r) asm volatile("prefetch.global.L1 [%0];" ::"l"(tp + (size_t)r * g.E));
        } else {
            const char* tb = reinterpret_cast<const char*>(g.tgt + (size_t)e * m * 2);
            for (int off = 128 * kk; off < m * 16; off += 128 * K) asm volatile("prefetch.global.L1 [%0];" ::"l"(tb + off));
            if (kk == K - 1) asm volatile("prefetch.global.L1 [%0];" ::"l"(tb + m * 16 - 1));
        }
    }
    __device__ __forceinline__ void targets_ready() const {}
};

// Structure-of-arrays state with the env's 2m target rows STAGED in shared memory: every thread copies its own column
// with 8-byte cp.async (LDGSTS) at kernel entry -- all 2m loads of a warp in flight at once, no registers held, one HBM
// round trip that overlaps the state loads and the agent phase -- and reads it back before the sensing loop.  (The L1
// prefetch of GlobalView does not do that job: with and without it the kernel takes the same time, and the sensing loop
// pays a round trip per block of targets.)
template <int TE>
struct StagedView : GlobalView<true> {
    static constexpr bool kStaged = true;
    struct Ctx { double* col; };                 // this thread's column of the CTA's staging area: row r at col[r * TE]
    double* col;
    __device__ __forceinline__ StagedView(const FlightParams& p_, const GroupEntry& g_, int e_, Ctx c) : GlobalView<true>(p_, g_, e_, GlobalView<true>::Ctx{}), col(c.col) {}
    __device__ __forceinline__ double2 tgt_ld(int j) const { return make_double2(col[(2 * j) * TE], col[(2 * j + 1) * TE]); }
    __device__ __forceinline__ void tgt_publish(int j, int es, int src, double2 v) const {
        double* t = this->g.tgt + (size_t)(2 * j) * this->g.E + es;
        t[0] = v.x; t[this->g.E] = v.y;
        double* w = col - (int)(threadIdx.x & 31) + src + (2 * j) * TE;                // the owner reads it back from its column
        w[0] = v.x; w[TE] = v.y;
    }
    template <int K>
    __device__ __forceinline__ void prefetch_targets(int) const {
        const double* tp = this->g.tgt + this->e;
        const size_t E = (size_t)this->g.E;
        uint32_t d = smem_u32(col);
#pragma unroll 6
        for (int r = 0; r < 2 * this->p.m; ++r, d += TE * 8, tp += E)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(tp) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    // every lane's own copies have landed; the warp barrier orders them before tgt_publish writes of OTHER lanes into this
    // lane's column (auto-reset, later in the kernel)
    __device__ __forceinline__ void targets_ready() const { asm volatile("cp.async.wait_all;" ::: "memory"); __syncwarp(); }
};

__device__ __forceinline__ GroupEntry entry_of(const FlightParams& p) {
    GroupEntry g;
    g.E = p.E; g.env_id_base = p.env_id_base; g.seed = p.seed; g.pad = 0;
    g.dyn_rs = p.dyn_rs; g.dyn_es = p.dyn_es; g.tgt_rs = p.tgt_rs; g.tgt_es = p.tgt_es;
    g.dyn = p.dyn; g.tgt = p.tgt; g.obs = p.obs; g.state = p.state; g.reward = p.reward; g.terminated = p.terminated;
    g.win = p.win; g.target_find = p.target_find; g.stats = p.stats; g.tmpl = p.tmpl;
    return g;
}

// e_raw: the env of this thread (>= g.E: none); t_first: e_raw * K + kk of lane 0 of this warp.
template <int N, int K, int MODE, bool MAP, bool FUSED, class V>
__device__ __forceinline__ int flight_tpe_body(const FlightParams& p, const GroupEntry& g, typename V::Ctx ctx,
                                               const int e_raw, const int t_first, const uint8_t* __restrict__ actions,
                                               const uint8_t* __restrict__ mask, uint32_t rflags, unsigned char* jobslots) {
    constexpr unsigned FULL = 0xffffffffu;
    static_assert(K == 1 || K == 4 || K == 8, "K");
    constexpr uint32_t MINE = 0xFFFFFFFFu / ((1u << K) - 1u);          // targets j with j % K == 0
    const int lane32 = threadIdx.x & 31, kk = threadIdx.x % K;          // kk: which of the env's K threads this is
    const bool active = e_raw < g.E;
    const int e = active ? e_raw : g.E - 1;
    const int m = p.m;
    const uint32_t env_id = g.env_id_base + (uint32_t)e;
    const V L(p, g, e, ctx);

    // ---- state of this env ---------------------------------------------------------------------------------
    if (MODE == MODE_STEP) L.template prefetch_targets<K>(kk);
    double ax[N], ay[N], yaw[N], c_h[N], s_h[N];
#pragma unroll
    for (int a = 0; a < N; ++a) {
        const double2 v = L.xy_ld(a);
        ax[a] = v.x; ay[a] = v.y;
        yaw[a] = L.yaw_ld(a);
        c_h[a] = 0.0; s_h[a] = 0.0;
    }
    uint4 m0, m1;
    L.meta_ld(&m0, &m1);
    uint32_t found = m0.x, newf_last = m0.y, outmask = m0.z, time_step = m0.w;
    uint32_t episode = m1.x, flags = m1.y;
    float ep_reward = __uint_as_float(m1.z);
    int njobs = 0;                              // belief-map jobs written to `jobslots` (MAP)

    bool done = (flags & CS_FLAG_DONE) != 0;
    bool do_sense = false, emit = false, state_full = false, have_result = false;
    float res_reward = 0.f;
    uint32_t res_term = 0, res_win = 0, res_found = 0, t_key = 0;   // what step()/reset() report for this env
    float st_eps = 0.f, st_rew = 0.f, st_found = 0.f, st_wins = 0.f, st_len = 0.f;

    // ---- _agent_step -------------------------------------------------------------------------------------------
    if (MODE == MODE_STEP) {
        const bool stepping = active && !done;
        if (stepping) {
            cs_u4 pw = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int a = 0; a < N; ++a) {
                int act;
                if (actions != nullptr) {
                    act = (int)actions[(size_t)e * N + a];
                } else {
                    // one Philox block serves 4 agents; action = word % 3 (np.random.randint(0, 3), agent.py:36)
                    if ((a & 3) == 0)
                        pw = cs_philox4x32_10(env_id, ((episode & 0xFFFFu) << 16) | ((time_step + 1u) & 0xFFFFu),
                                              (uint32_t)(a >> 2), 0u, g.seed, cs_stream_key(CS_STREAM_POLICY, episode));
                    act = (int)(cs_word(pw, a & 3) % 3u);
                }
                double h = yaw[a] + ((act == 1) ? p.turn : ((act == 2) ? -p.turn : 0.0));   // dyaw = [0, pi/18, -pi/18] (:259-262)
                if (h > p.two_pi) h -= p.two_pi;                                             // strict tests (:263-266)
                else if (h < 0.0) h += p.two_pi;
                const double2 sc = heading_sincos(p, h);
                s_h[a] = sc.x; c_h[a] = sc.y;
                yaw[a] = h;
            }
            // Can any repulsion term be non-zero this step?  (see flight_kernel / DESIGN.md 4.2)
            bool close = false;
#pragma unroll
            for (int a = 0; a < N; ++a)
#pragma unroll
                for (int q = a + 1; q < N; ++q) {
                    const double dx = ax[q] - ax[a], dy = ay[q] - ay[a];
                    close |= (dx * dx + dy * dy < p.near2);
                }
            uint32_t ob = 0;
            if (!close) {
#pragma unroll
                for (int a = 0; a < N; ++a) {
                    ax[a] = ax[a] + p.v * c_h[a];                 // x += v*cos(yaw)   (:267-268)
                    ay[a] = ay[a] + p.v * s_h[a];
                    if (wall_reg(p, ax[a], ay[a], yaw[a], c_h[a])) ob |= 1u << a;
                }
            } else {
                // the reference's sequential, in-place update (:271,:293-301): agent k sees its own OLD position and the
                // already-moved q < k; the terms are added in ascending q
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double x0 = ax[k], y0 = ay[k];
                    double fx = 0.0, fy = 0.0;
#pragma unroll
                    for (int q = 0; q < N; ++q) {
                        if (q == k) continue;
                        const double dxq = ax[q] - x0, dyq = ay[q] - y0;
                        if ((dxq * dxq + dyq * dyq < p.fd2) && (ax[q] != x0 || ay[q] != y0)) {
                            const double ex = x0 - ax[q], ey = y0 - ay[q];
                            const double r2 = ex * ex + ey * ey;
                            fx += p.fk * ex / r2;
                            fy += p.fk * ey / r2;
                        }
                    }
                    double nx = x0 + p.v * c_h[k], ny = y0 + p.v * s_h[k];
                    nx += fx;
                    ny += fy;
                    ax[k] = nx; ay[k] = ny;
                    if (wall_reg(p, ax[k], ay[k], yaw[k], c_h[k])) ob |= 1u << k;
                }
            }
            outmask = ob;
            do_sense = true;
            t_key = time_step + 1u;
        } else if (active) {
            have_result = true;                            // masked no-op on a finished env
            res_reward = 0.f;
            res_term = 1;
            res_win = flags & CS_FLAG_WIN;
            res_found = (uint32_t)__popc(found);
        }
    }

    L.targets_ready();                                  // (staged targets: every lane's own column has landed)
    for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1) {
            const bool do_reset = active && ((MODE == MODE_RESET) ? (mask == nullptr || mask[e] != 0) : (p.auto_reset && done));
            const unsigned rmask = __ballot_sync(FULL, do_reset && kk == 0);
            if (!rmask) break;
            do_sense = do_reset;
            if (do_reset) {                                                   // reset (:79-180)
                episode += (rflags & CS_RESET_KEEP_EPISODE) ? 0u : 1u;
                found = 0; outmask = 0; time_step = 0; flags = 0; ep_reward = 0.f; done = false;
#pragma unroll
                for (int a = 0; a < N; ++a) {
                    const double lin = p.lin[a];                                          // (:140-143)
                    switch (p.agent_mode) {
                        case 0: ax[a] = lin; ay[a] = 0.0; yaw[a] = p.half_pi; break;
                        case 1: ax[a] = lin; ay[a] = p.Md / 2.0; yaw[a] = p.half_pi; break;
                        case 2: ax[a] = 0.0; ay[a] = lin; yaw[a] = 0.0; break;
                        default: ax[a] = p.Md; ay[a] = lin; yaw[a] = p.pi; break;
                    }
                    c_h[a] = p.cos0; s_h[a] = p.sin0;
                }
                t_key = 0;
                emit = true;
                state_full = true;
                if (MODE == MODE_RESET) { have_result = true; res_reward = 0.f; res_term = 0; }
            }
            // warp-cooperative heavy parts of a reset, one resetting env at a time: its targets (one lane per
            // target, :95-127) and, for reset(init=True), its belief map (flight_env.py:84-86)
            if (!(rflags & CS_RESET_KEEP_TARGETS) || (FUSED && (rflags & CS_RESET_INIT))) {
                unsigned left = rmask;
                while (left) {
                    const int src = __ffs(left) - 1;
                    left &= left - 1;
                    const int es = (t_first + src) / K;
                    const uint32_t ep_s = __shfl_sync(FULL, episode, src);
                    if (!(rflags & CS_RESET_KEEP_TARGETS)) {
                        for (int j = lane32; j < m; j += 32) {
                            const double2 t = draw_target(p, g.tmpl, g.seed, g.env_id_base + (uint32_t)es, ep_s, j);
                            L.tgt_publish(j, es, src, t);
                        }
                    }
                    if (FUSED && (rflags & CS_RESET_INIT)) {     // (the map kernel does this fill in the two-kernel form)
                        float4* map = reinterpret_cast<float4*>(p.prob_map + (size_t)es * p.map_stride);
                        for (int c = lane32; c < p.map_stride / 4; c += 32) map[c] = make_float4(0.5f, 0.5f, 0.5f, 0.5f);
                    }
                }
                __syncwarp();                                   // the owners read the new targets back below
            }
        } else if (MODE == MODE_RESET) {
            continue;
        }

        // ---- _update_obs: detection + reward + win (:223-253) ----------------------------------------------
        uint32_t newf = 0;
        if (do_sense) {
            // the env's K threads share the targets; TU of a thread's targets are loaded together so that their
            // latency is paid once per block, not once per target
            constexpr int TU = (K >= 8) ? 2 : ((V::kStaged && N <= 3) ? 1 : CS_TPE_TU);
            uint32_t need = 0;                          // targets in view of some agent and not found yet
            for (int j0 = kk; j0 < m; j0 += K * TU) {
                double2 t[TU];
#pragma unroll
                for (int u = 0; u < TU; ++u) {
                    const int j = min(j0 + u * K, m - 1);
                    t[u] = L.tgt_ld(j);
                }
#pragma unroll
                for (int u = 0; u < TU; ++u) {
                    const int j = j0 + u * K;
                    if (j >= m) break;
                    uint32_t amask = 0;
#pragma unroll
                    for (int a = 0; a < N; ++a) {
                        const double dx = t[u].x - ax[a], dy = t[u].y - ay[a];
                        if (dx * dx + dy * dy <= p.R2) amask |= 1u << a;               // '<=' (:237)
                    }
                    if (amask && !((found >> j) & 1u)) need |= 1u << j;                // draw is irrelevant once found (:239)
                }
            }
            // The detection draws, in a second loop over the targets that need one.  Inside the loop above the warp would
            // run the Philox rounds in every iteration where ANY of its 32 envs has the target in view (about half of the
            // iterations); here it runs them max-over-lanes(number of needed targets) times -- two or three.
            for (uint32_t left = need; left; left &= left - 1u) {
                const int j = __ffs(left) - 1;
                const double2 tj = L.tgt_ld(j);
                uint32_t amask = 0;
#pragma unroll
                for (int a = 0; a < N; ++a) {
                    const double dx = tj.x - ax[a], dy = tj.y - ay[a];
                    if (dx * dx + dy * dy <= p.R2) amask |= 1u << a;
                }
                bool got = false;
#pragma unroll
                for (int blk = 0; 4 * blk < N; ++blk) {
                    const uint32_t bits = (amask >> (4 * blk)) & 0xFu;
                    if (!bits || got) continue;
                    const cs_u4 w = cs_detect_words(g.seed, env_id, episode, t_key, (uint32_t)blk, (uint32_t)j);
                    got = ((bits & 1u) && (long long)w.x <= p.thr) || ((bits & 2u) && (long long)w.y <= p.thr) ||
                          ((bits & 4u) && (long long)w.z <= p.thr) || ((bits & 8u) && (long long)w.w <= p.thr);
                }
                if (got) newf |= 1u << j;
            }
        }
#pragma unroll
        for (int o = K / 2; o > 0; o >>= 1) newf |= __shfl_xor_sync(FULL, newf, o);
        int rew = 0;
        if (do_sense) {
            found |= newf;
            newf_last = newf;
            const int c = __popc(newf);
            rew = -1 + 10 * c;                                                 // MOVE_COST + FIND_ONE_TGT (:228,:241)
            if (c > 0 && __popc(found) == m && !(flags & CS_FLAG_WIN)) {
                rew += 100;                                                    // FIND_ALL_TGT (:244-246)
                flags |= CS_FLAG_WIN;
            }
            rew -= __popc(outmask);                                            // OUT_PUNISH per agent outside (:249-250)
        }
        if (MODE == MODE_RESET && do_sense) {
            res_win = flags & CS_FLAG_WIN;
            res_found = (uint32_t)__popc(found);
        }
        if (pass == 0 && do_sense) {                                           // step bookkeeping (:308-314)
            time_step += 1u;
            ep_reward += (float)rew;
            const int nfound = __popc(found);
            const bool term = (nfound >= m) || ((int)time_step >= p.T);
            if (term) flags |= CS_FLAG_DONE;
            done = term;
            emit = true;
            have_result = true;
            res_reward = (float)rew;
            res_term = term ? 1u : 0u;
            res_win = flags & CS_FLAG_WIN;          // of the episode this step belongs to, also when auto_reset follows
            res_found = (uint32_t)nfound;
            if (term && kk == 0) {
                st_eps = 1.f; st_rew = ep_reward; st_found = (float)nfound; st_wins = (flags & CS_FLAG_WIN) ? 1.f : 0.f;
                st_len = (float)time_step;
            }
        }
        // ---- belief map (flight_env.py:266,:275-303): a job for fused_map_phase -- the positions this sensing call
        //      saw and the cells of the targets it found.  An env that is reset inside this call leaves two jobs.
        if (MAP && do_sense) {
            if (kk == 0) {
                double* jx = reinterpret_cast<double*>(jobslots + njobs * p.fm_jobsz);
                int* jh = reinterpret_cast<int*>(jx + 2 * N);
#pragma unroll
                for (int a = 0; a < N; ++a) *reinterpret_cast<double2*>(jx + 2 * a) = make_double2(ax[a], ay[a]);
                int k = 0;
                for (uint32_t left = newf; left; left &= left - 1) {
                    const int j = __ffs(left) - 1;
                    const double2 t = L.tgt_ld(j);
                    jh[1 + k++] = hit_cell(p, t.x, t.y);
                }
                jh[0] = k;
            }
            ++njobs;
        }
    }

    // ---- outputs ---------------------------------------------------------------------------------------------
    if (active && emit) {
        float* srow = g.state + (size_t)e * p.state_stride;
#pragma unroll
        for (int a = 0; a < N; ++a) {
            if (a % K != kk) continue;                                  // the env's K threads share the rows
            L.xy_st(a, ax[a], ay[a]);
            L.yaw_st(a, yaw[a]);
            // get_obs row = agent part of get_state (flight_env_easy.py:218-221, :192-193)
            const float4 o = make_float4((float)((ax[a] - p.half_M) * p.inv_half), (float)((ay[a] - p.half_M) * p.inv_half),
                                         (float)c_h[a], (float)s_h[a]);
            reinterpret_cast<float4*>(g.obs)[(size_t)e * N + a] = o;
            reinterpret_cast<float4*>(srow)[a] = o;
        }
        if (kk == 0) {
            L.meta_st(make_uint4(found, newf_last, outmask, time_step), make_uint4(episode, flags, __float_as_uint(ep_reward), 0u));
        }
        // target part of the state row (:201-211): rewritten in full after a reset, otherwise only the 'find' entry of
        // a target found by this call
        if (state_full) {
            for (int j = kk; j < m; j += K) {
                const double2 t = L.tgt_ld(j);
                float* s3 = srow + 4 * N + 3 * j;
                const float nx = (float)((t.x - p.half_M) * p.inv_half), ny = (float)((t.y - p.half_M) * p.inv_half);
                const float fj = ((found >> j) & 1u) ? 1.0f : 0.0f;
                s3[0] = nx; s3[1] = ny; s3[2] = fj;
            }
        } else {
            for (uint32_t left = newf_last & (MINE << kk); left; left &= left - 1) srow[4 * N + 3 * (__ffs(left) - 1) + 2] = 1.0f;
        }
    }
    if (active && have_result && kk == 0) {
        g.reward[e] = res_reward;
        g.terminated[e] = (uint8_t)res_term;
        g.win[e] = res_win ? 1 : 0;
        g.target_find[e] = (int32_t)res_found;
    }
    // ---- statistics of episodes that ended in this call: warp reduction, then one atomic per statistic per warp
    if (MODE == MODE_STEP) {
        if (__any_sync(FULL, st_eps != 0.f)) {
            for (int o = 16; o > 0; o >>= 1) {
                st_eps += __shfl_xor_sync(FULL, st_eps, o);
                st_rew += __shfl_xor_sync(FULL, st_rew, o);
                st_found += __shfl_xor_sync(FULL, st_found, o);
                st_wins += __shfl_xor_sync(FULL, st_wins, o);
                st_len += __shfl_xor_sync(FULL, st_len, o);
            }
            if (lane32 == 0) {
                atomicAdd(g.stats + CS_STAT_EPISODES, (double)st_eps);
                atomicAdd(g.stats + CS_STAT_EP_REWARD, (double)st_rew);
                atomicAdd(g.stats + CS_STAT_TARGETS_FOUND, (double)st_found);
                atomicAdd(g.stats + CS_STAT_WINS, (double)st_wins);
                atomicAdd(g.stats + CS_STAT_EP_LEN, (double)st_len);
            }
        }
    }
    return active ? njobs : 0;
}

template <int N, int K, int MODE, bool MAP>
__global__ void __launch_bounds__(kTpeThreads, tpe_min_ctas(N, K, MAP ? 1 : MODE)) flight_tpe_kernel(const __grid_constant__ FlightParams p, const uint8_t* __restrict__ actions,
                                                                 const uint8_t* __restrict__ mask, uint32_t rflags) {
    const GroupEntry g = entry_of(p);
    const int t0 = (int)blockIdx.x * kTpeThreads + (int)threadIdx.x;
    const int e_raw = t0 / K, t_first = t0 & ~31;
    if (K == 1 && MODE == MODE_STEP && !MAP) {                          // one thread per env: targets staged in shared memory
        extern __shared__ __align__(16) double tstage[];
        using S = StagedView<kTpeThreads>;
        typename S::Ctx ctx;
        ctx.col = tstage + threadIdx.x;
        flight_tpe_body<N, K, MODE, false, false, S>(p, g, ctx, e_raw, t_first, actions, mask, rflags, nullptr);
        return;
    }
    using V = GlobalView<K == 1>;                                       // one thread per env <-> structure of arrays (cs_flight_create)
    if (!MAP) {
        flight_tpe_body<N, K, MODE, false, false, V>(p, g, typename V::Ctx{}, e_raw, t_first, actions, mask, rflags, nullptr);
        return;
    }
    // flight variant, two-kernel form: this env's belief-map job record for flight_map_tile_kernel, which runs next
    // (on the same stream, or on the handle's map stream): header {jobs, fill flag} + up to two job slots
    const int e = e_raw < p.E ? e_raw : p.E - 1;
    unsigned char* rec = p.jobs + (size_t)e * p.job_stride;
    const int njobs = flight_tpe_body<N, K, MODE, true, false, V>(p, g, typename V::Ctx{}, e_raw, t_first, actions, mask, rflags, rec + 16);
    if (e_raw < p.E && threadIdx.x % K == 0) {
        const int fill = (MODE == MODE_RESET && (rflags & CS_RESET_INIT) && (mask == nullptr || mask[e] != 0)) ? 1 : 0;   // reset(init=True): map <- 0.5 (flight_env.py:84-86)
        *reinterpret_cast<int2*>(rec) = make_int2(njobs, fill);
    }
}

// The flight variant: step / reset and the belief-map update of the same envs in ONE kernel (flight_map.cuh).  8 lanes
// own one env through both phases: they share the target loop of the step (K = 8), the first of them stashes the
// belief-map job(s) in the env's shared-memory scratch, and the same 8 lanes then sweep the env's map tiles.  16384 envs
// are 1024 CTAs of 128 threads: one wave at 7 CTAs per SM.
constexpr int kFusedThreads = 128;
constexpr int kFusedLanes = 8;
#ifndef CS_FUSED_MIN_CTAS
#define CS_FUSED_MIN_CTAS 7
#endif

template <int N, int MODE>
__global__ void __launch_bounds__(kFusedThreads, CS_FUSED_MIN_CTAS) flight_fused_kernel(const __grid_constant__ FlightParams p, const uint8_t* __restrict__ actions,
                                                                                       const uint8_t* __restrict__ mask, uint32_t rflags) {
    extern __shared__ __align__(16) unsigned char fsm[];
    using V = GlobalView<false>;
    const GroupEntry g = entry_of(p);
    unsigned char* S = fsm + (size_t)(threadIdx.x / kFusedLanes) * p.fm_env;
    const int t0 = (int)blockIdx.x * kFusedThreads + (int)threadIdx.x;
    const int njobs = flight_tpe_body<N, kFusedLanes, MODE, true, true, V>(p, g, typename V::Ctx{}, t0 / kFusedLanes, t0 & ~31, actions, mask,
                                                                            rflags, S + p.fm_job);
    const int e = min(t0 / kFusedLanes, p.E - 1);
    fused_map_phase<kFusedLanes>(p, e, (int)(threadIdx.x % kFusedLanes), S, njobs);
}

// Grouped step of several handles (independent env batches of the same shape: rollout workers) in ONE launch:
// blockIdx.y picks the handle.  A launch of a few thousand envs is bound by the launch path (2.2 us per 4096-env launch
// inside a 64-node graph, DESIGN.md section 8); grouped, the same batches fill the GPU like one large handle.  Everything
// arrives through the kernel parameter space (constant bank): the configuration the group's handles share (`common`), what
// differs per handle (GroupTable: sizes, global ids, buffers) and the action pointers.  flight_easy variant only.
template <int N, int K>
__global__ void __launch_bounds__(kTpeThreads, tpe_min_ctas(N, K, 0)) flight_tpe_group_kernel(const __grid_constant__ FlightParams common,
                                                                                       const __grid_constant__ GroupTable tab,
                                                                                       const __grid_constant__ GroupActions acts) {
    const GroupEntry& g = tab.h[blockIdx.y];
    if ((long long)blockIdx.x * kTpeThreads >= (long long)g.E * K) return;          // handles may differ in num_envs
    const int t0 = (int)blockIdx.x * kTpeThreads + (int)threadIdx.x;
    if (K == 1) {
        extern __shared__ __align__(16) double tstage[];
        using S = StagedView<kTpeThreads>;
        typename S::Ctx ctx;
        ctx.col = tstage + threadIdx.x;
        flight_tpe_body<N, K, MODE_STEP, false, false, S>(common, g, ctx, t0, t0 & ~31, acts.a[blockIdx.y], nullptr, 0u, nullptr);
        return;
    }
    using V = GlobalView<false>;
    flight_tpe_body<N, K, MODE_STEP, false, false, V>(common, g, typename V::Ctx{}, t0 / K, t0 & ~31, acts.a[blockIdx.y], nullptr, 0u, nullptr);
}

// shared-memory staging area of the targets in the one-thread-per-env step kernels: 2m rows of kTpeThreads doubles
inline size_t tstage_bytes(int m) { return (size_t)2 * m * kTpeThreads * sizeof(double); }

template <int N, int K>
cudaError_t launch_tpe_k(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    const long long threads = (long long)h->p.E * K;
    const int grid = (int)((threads + kTpeThreads - 1) / kTpeThreads);
    if (h->p.variant) {
        if (mode == MODE_STEP)
            flight_tpe_kernel<N, K, MODE_STEP, true><<<grid, kTpeThreads, 0, st>>>(h->p, actions, mask, rflags);
        else
            flight_tpe_kernel<N, K, MODE_RESET, true><<<grid, kTpeThreads, 0, st>>>(h->p, actions, mask, rflags);
    } else {
        if (mode == MODE_STEP)
            flight_tpe_kernel<N, K, MODE_STEP, false><<<grid, kTpeThreads, K == 1 ? tstage_bytes(h->p.m) : 0, st>>>(h->p, actions, mask, rflags);
        else
            flight_tpe_kernel<N, K, MODE_RESET, false><<<grid, kTpeThreads, 0, st>>>(h->p, actions, mask, rflags);
    }
    cs_count_launch(1);
    return cudaGetLastError();
}

template <int N>
cudaError_t launch_fused(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    const long long threads = (long long)h->p.E * kFusedLanes;
    const int grid = (int)((threads + kFusedThreads - 1) / kFusedThreads);
    const size_t smem = (size_t)(kFusedThreads / kFusedLanes) * h->p.fm_env;
    if (mode == MODE_STEP)
        flight_fused_kernel<N, MODE_STEP><<<grid, kFusedThreads, smem, st>>>(h->p, actions, mask, rflags);
    else
        flight_fused_kernel<N, MODE_RESET><<<grid, kFusedThreads, smem, st>>>(h->p, actions, mask, rflags);
    cs_count_launch(1);
    return cudaGetLastError();
}

template <int N>
cudaError_t launch_tpe_n(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    if (h->fused) return launch_fused<N>(h, mode, actions, mask, rflags, st);
    switch (h->tpe_k) {
        case 1: return launch_tpe_k<N, 1>(h, mode, actions, mask, rflags, st);
        default: return launch_tpe_k<N, 4>(h, mode, actions, mask, rflags, st);
    }
}

template <int N>
cudaError_t launch_group_n(const cs_flight_group* g, const GroupActions& acts, cudaStream_t st) {
    const dim3 grid((unsigned)g->grid_x, (unsigned)g->count);
    if (g->k == 1) flight_tpe_group_kernel<N, 1><<<grid, kTpeThreads, tstage_bytes(g->envs[0]->p.m), st>>>(g->envs[0]->p, g->table, acts);
    else flight_tpe_group_kernel<N, 4><<<grid, kTpeThreads, 0, st>>>(g->envs[0]->p, g->table, acts);
    cs_count_launch(1);
    return cudaGetLastError();
}

constexpr int kNLo = 2 * CS_TPE_PART + 1, kNHi = kNLo + 1;

}  // namespace

#define CS_CAT2(a, b) a##b
#define CS_CAT(a, b) CS_CAT2(a, b)

cudaError_t CS_CAT(launch_tpe_part, CS_TPE_PART)(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    return h->p.n == kNLo ? launch_tpe_n<kNLo>(h, mode, actions, mask, rflags, st) : launch_tpe_n<kNHi>(h, mode, actions, mask, rflags, st);
}

cudaError_t CS_CAT(launch_group_part, CS_TPE_PART)(const cs_flight_group* g, const uint8_t* const* d_actions, cudaStream_t st) {
    GroupActions acts;
    for (int i = 0; i < g->count; ++i) acts.a[i] = d_actions[i];
    for (int i = g->count; i < kMaxGroup; ++i) acts.a[i] = nullptr;
    return g->n == kNLo ? launch_group_n<kNLo>(g, acts, st) : launch_group_n<kNHi>(g, acts, st);
}

int CS_CAT(fused_lanes_part, CS_TPE_PART)() { return kFusedLanes; }

}  // namespace csf
