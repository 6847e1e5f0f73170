// Lane-per-agent step / reset kernel of flight_easy / flight (n_agents > 8, or lanes_per_env >= 16) and the launch of
// the generic belief-map kernel that follows it in the flight variant.  See flight_common.cuh for the file map.
#include "flight_internal.h"

namespace csf {
namespace {

// ------------------------------------------------------------------------------------------------
// The step / reset kernel.  A group of LPE lanes (LPE = power of two >= max(n_agents, target_num)) owns one env:
// lane a < n holds agent a (x, y, heading, cos, sin) and lane j < m holds target j, all in REGISTERS; positions
// travel between lanes by warp shuffles.  Every global load is issued up front; the kernel uses no shared memory.
// Every warp collective uses the FULL mask and sits in warp-uniform control flow (groups are told apart by
// predicates, not branches), so no partial-mask MATCH/REDUX sequences or divergence barriers are generated.
//   pass 0 (STEP): _agent_step -> _update_obs -> step bookkeeping            (flight_env_easy.py:255-314)
//   pass 1       : reset (selected envs in RESET mode; just-terminated envs under auto_reset) -> _update_obs (:79-182)
// actions == nullptr in MODE_STEP: uniform-random policy drawn in-kernel (alg=random, agent/agent.py:34-36)
// ------------------------------------------------------------------------------------------------
template <int LPE, int MODE, bool MAP>
__global__ void __launch_bounds__(kThreads, 8) flight_kernel(const __grid_constant__ FlightParams p, const uint8_t* __restrict__ actions,
                                                             const uint8_t* __restrict__ mask, uint32_t rflags, uint32_t seq) {
    constexpr int EPW = 32 / LPE;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr unsigned GBITS = (LPE == 32) ? 0xffffffffu : ((1u << (LPE & 31)) - 1u);

    const int tid = threadIdx.x, warp = tid >> 5, lane32 = tid & 31;
    const int wenv0 = (blockIdx.x * (kThreads / 32) + warp) * EPW;      // first env of this warp
    const int wcnt = min(EPW, p.E - wenv0);
    if (wcnt <= 0) return;                                               // whole warp idle (nothing is block-synchronised)
    const int n = p.n, m = p.m;
    const int g = lane32 / LPE, lane = lane32 % LPE, gbase = lane32 - lane;
    const bool active = g < wcnt;
    const int e = wenv0 + (active ? g : 0);
    const bool is_agent = active && lane < n, is_tgt = active && lane < m;
    const uint32_t env_id = p.env_id_base + (uint32_t)e;
#define GSHFL(v, q) __shfl_sync(FULL, (v), gbase + (q))
#define GBALLOT(pred) ((__ballot_sync(FULL, (pred)) >> gbase) & GBITS)

    // ---- every load of the step, issued before anything is consumed ----------------------------------------
    double ax = 0.0, ay = 0.0, yaw = 0.0, tx = 0.0, ty = 0.0;
    uint4 m0 = make_uint4(0, 0, 0, 0), m1 = make_uint4(0, 0, 0, 0);
    int act = 0;
    if (is_agent) {
        const double2 v = xy_ld(p, lane, e);
        ax = v.x; ay = v.y;
        yaw = *dyn_at(p, p.yaw_off + lane, e);
        if (MODE == MODE_STEP && actions != nullptr) act = actions[(size_t)e * n + lane];
    }
    if (is_tgt) {
        const double2 v = tgt_ld(p, lane, e);
        tx = v.x; ty = v.y;
    }
    if (active) {
        meta_ld(p, e, &m0, &m1);                                               // same addresses for the whole group
    }
    uint32_t found = m0.x, newf_last = m0.y, outmask = m0.z, time_step = m0.w;
    uint32_t episode = m1.x, flags = m1.y;
    float ep_reward = __uint_as_float(m1.z);

    double c_h = 0.0, s_h = 0.0;                 // cos/sin of the heading (agent lanes), for the fp32 outputs
    bool done = (flags & CS_FLAG_DONE) != 0;
    bool do_sense = false, emit = false, state_full = false, tgt_dirty = false, have_result = false;
    float res_reward = 0.f;
    uint32_t res_term = 0, res_win = 0, res_found = 0, t_key = 0;   // what step()/reset() report for this env
    float st_eps = 0.f, st_rew = 0.f, st_found = 0.f, st_wins = 0.f, st_len = 0.f;
    uint32_t sense_word = m1.w, prejob = 0;     // CS_META_SENSE: (call number << 1) | job parked in `pre`

    // ---- _agent_step -------------------------------------------------------------------------------------------
    if (MODE == MODE_STEP) {
        const bool stepping = active && !done;
        if (stepping && is_agent) {
            if (actions == nullptr) {
                // one Philox block serves 4 agents; action = word % 3 (np.random.randint(0, 3), agent.py:36)
                const cs_u4 w = cs_philox4x32_10(env_id, ((episode & 0xFFFFu) << 16) | ((time_step + 1u) & 0xFFFFu),
                                                 (uint32_t)(lane >> 2), 0u, p.seed, cs_stream_key(CS_STREAM_POLICY, episode));
                act = (int)(cs_word(w, lane & 3) % 3u);
            }
            double h = yaw + ((act == 1) ? p.turn : ((act == 2) ? -p.turn : 0.0));   // dyaw = [0, pi/18, -pi/18] (:259-262)
            if (h > p.two_pi) h -= p.two_pi;                                          // strict tests (:263-266)
            else if (h < 0.0) h += p.two_pi;
            { const double2 sc = heading_sincos(p, h); s_h = sc.x; c_h = sc.y; }
            yaw = h;
        }
        // Can any repulsion term be non-zero this step?  If every pair of OLD positions is farther apart than
        // force_dist + |v| (with slack), no agent receives a force, every displacement is <= |v|, and by
        // induction over the sequential update order no later agent does either (DESIGN.md 4.2).
        bool close = false;
        for (int q = 1; q < n; ++q) {
            const double xq = GSHFL(ax, q), yq = GSHFL(ay, q);
            const double dx = xq - ax, dy = yq - ay;
            close |= (q > lane && dx * dx + dy * dy < p.near2);
        }
        const bool close_g = GBALLOT(close && stepping && is_agent) != 0u;     // some pair of this env is close
        bool outside = false;
        if (stepping && is_agent && !close_g) {
            ax = ax + p.v * c_h;                          // x += v*cos(yaw)   (:267-268)
            ay = ay + p.v * s_h;
            outside = wall_reg(p, ax, ay, yaw, c_h);
        }
        if (__any_sync(FULL, close_g)) {
            // Repulsion path: the reference's sequential, in-place update (:271,:293-301) -- agent k sees its own
            // OLD position and the already-moved j<k.  Lanes keep their CURRENT position in registers, so iterating
            // k = 0..n-1 and letting every lane q evaluate its term against agent k's old position reproduces
            // exactly that; the terms of the (few) lanes in range are added on lane k in ascending q, the
            // reference's summation order.
            for (int k = 0; k < n; ++k) {
                const double x0 = GSHFL(ax, k), y0 = GSHFL(ay, k);
                const double dxq = ax - x0, dyq = ay - y0;
                const bool inr = close_g && is_agent && lane != k && (dxq * dxq + dyq * dyq < p.fd2) && (ax != x0 || ay != y0);
                uint32_t near_all = __ballot_sync(FULL, inr);
                double tfx = 0.0, tfy = 0.0;
                if (inr) {
                    const double ex = x0 - ax, ey = y0 - ay;
                    const double r2 = ex * ex + ey * ey;
                    tfx = p.fk * ex / r2;
                    tfy = p.fk * ey / r2;
                }
                double fx = 0.0, fy = 0.0;
                while (near_all) {                                          // warp-uniform; ascending lane = ascending q
                    const int src = __ffs(near_all) - 1;
                    near_all &= near_all - 1;
                    const double vx = __shfl_sync(FULL, tfx, src), vy = __shfl_sync(FULL, tfy, src);
                    if ((src & ~(LPE - 1)) == gbase) { fx += vx; fy += vy; }
                }
                if (close_g && is_agent && lane == k) {
                    ax = ax + p.v * c_h;
                    ay = ay + p.v * s_h;
                    ax += fx;
                    ay += fy;
                    outside = wall_reg(p, ax, ay, yaw, c_h);
                }
            }
        }
        if (stepping) {
            do_sense = true;
            t_key = time_step + 1u;
        } else if (active) {
            have_result = true;                            // masked no-op on a finished env
            res_reward = 0.f;
            res_term = 1;
            res_win = flags & CS_FLAG_WIN;
            res_found = (uint32_t)__popc(found);
        }
        const uint32_t ob = GBALLOT(outside);
        if (stepping) outmask = ob;
    }

    for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1) {
            const bool do_reset = active && ((MODE == MODE_RESET) ? (mask == nullptr || mask[e] != 0) : (p.auto_reset && done));
            if (!__any_sync(FULL, do_reset)) break;
            do_sense = do_reset;
            if (do_reset) {                                                   // reset (:79-180)
                episode += (rflags & CS_RESET_KEEP_EPISODE) ? 0u : 1u;
                found = 0; outmask = 0; time_step = 0; flags = 0; ep_reward = 0.f; done = false;
                if (!(rflags & CS_RESET_KEEP_TARGETS)) {
                    if (is_tgt) {
                        const double2 t = draw_target(p, p.tmpl, p.seed, env_id, episode, lane);
                        tx = t.x; ty = t.y;
                    }
                    tgt_dirty = true;
                }
                if (is_agent) {
                    const double lin = p.lin[lane];                                       // (:140-143)
                    switch (p.agent_mode) {
                        case 0: ax = lin; ay = 0.0; yaw = p.half_pi; break;
                        case 1: ax = lin; ay = p.Md / 2.0; yaw = p.half_pi; break;
                        case 2: ax = 0.0; ay = lin; yaw = 0.0; break;
                        default: ax = p.Md; ay = lin; yaw = p.pi; break;
                    }
                    c_h = p.cos0; s_h = p.sin0;
                }
                if (MAP && (rflags & CS_RESET_INIT)) {
                    float* map = p.prob_map + (size_t)e * p.map_stride;
                    for (int c = lane; c < p.map_stride; c += LPE) map[c] = 0.5f;         // flight_env.py:84-86 (tiled map incl. padding)
                }
                t_key = 0;
                emit = true;
                state_full = true;
                if (MODE == MODE_RESET) { have_result = true; res_reward = 0.f; res_term = 0; }
            }
        } else if (MODE == MODE_RESET) {
            continue;
        }

        // ---- _update_obs: detection + reward + win (:223-253) ----------------------------------------------
        uint32_t amask = 0;
        for (int q = 0; q < n; ++q) {
            const double xq = GSHFL(ax, q), yq = GSHFL(ay, q);
            const double dx = tx - xq, dy = ty - yq;
            if (dx * dx + dy * dy <= p.R2) amask |= 1u << q;                   // '<=' (:237)
        }
        bool got = false;
        if (do_sense && is_tgt && amask && !((found >> lane) & 1u)) {          // draw is irrelevant once found (:239)
            for (int blk = 0; 4 * blk < n && !got; ++blk) {
                const uint32_t bits = (amask >> (4 * blk)) & 0xFu;
                if (!bits) continue;
                const cs_u4 w = cs_detect_words(p.seed, env_id, episode, t_key, (uint32_t)blk, (uint32_t)lane);
                got = ((bits & 1u) && (long long)w.x <= p.thr) || ((bits & 2u) && (long long)w.y <= p.thr) ||
                      ((bits & 4u) && (long long)w.z <= p.thr) || ((bits & 8u) && (long long)w.w <= p.thr);
            }
        }
        const uint32_t newf = GBALLOT(got);
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
            if (lane == 0 && term) {
                st_eps = 1.f; st_rew = ep_reward; st_found = (float)nfound; st_wins = (flags & CS_FLAG_WIN) ? 1.f : 0.f;
                st_len = (float)time_step;
            }
        }
        // ---- belief map (flight_env.py:266,:275-303): a job for flight_map_generic_kernel, which runs next on the stream.
        //      Normally the job IS the state record (positions, CS_META_NEWFOUND); an env about to be reset inside this
        //      call parks the job of its last step in the side buffer, because pass 1 overwrites the record.
        if (MAP && do_sense) {
            sense_word = seq << 1;
            if (pass == 0 && done && p.auto_reset) {
                double* pj = p.pre + (size_t)e * p.pre_stride;
                int* ph = reinterpret_cast<int*>(pj + 2 * n);
                if (is_agent) *reinterpret_cast<double2*>(pj + 2 * lane) = make_double2(ax, ay);
                if (lane == 0) ph[0] = __popc(newf);
                if (is_tgt && ((newf >> lane) & 1u)) ph[1 + __popc(newf & ((1u << lane) - 1u))] = hit_cell(p, tx, ty);
                prejob = 1u;
            }
        }
    }
#undef GSHFL
#undef GBALLOT

    // ---- outputs, straight from registers -------------------------------------------------------------------
    if (active && emit) {
        if (is_agent) {
            xy_st(p, lane, e, ax, ay);
            *dyn_at(p, p.yaw_off + lane, e) = yaw;
            // get_obs row = agent part of get_state (flight_env_easy.py:218-221, :192-193)
            const float4 o = make_float4((float)((ax - p.half_M) * p.inv_half), (float)((ay - p.half_M) * p.inv_half),
                                         (float)c_h, (float)s_h);
            reinterpret_cast<float4*>(p.obs)[(size_t)e * n + lane] = o;
            reinterpret_cast<float4*>(p.state + (size_t)e * p.state_stride)[lane] = o;
        }
        if (lane == 0) {
            meta_st(p, e, make_uint4(found, newf_last, outmask, time_step),
                    make_uint4(episode, flags, __float_as_uint(ep_reward), MAP ? (sense_word | prejob) : 0u));
        }
        if (is_tgt) {
            // target part of the state row (:201-211): rewritten in full after a reset, otherwise only the 'find'
            // entry of a target found by this call
            float* srow = p.state + (size_t)e * p.state_stride + 4 * n + 3 * lane;
            if (state_full) {
                srow[0] = (float)((tx - p.half_M) * p.inv_half);
                srow[1] = (float)((ty - p.half_M) * p.inv_half);
                srow[2] = ((found >> lane) & 1u) ? 1.0f : 0.0f;
            } else if ((newf_last >> lane) & 1u) {
                srow[2] = 1.0f;
            }
            if (tgt_dirty) tgt_st(p, lane, e, make_double2(tx, ty));
        }
    }
    if (MAP && active && !emit && lane == 0 && m1.w != 0u)
        meta_at(p, 3, e)->y = 0u;      // not sensed by THIS call: no job for the map kernel
    if (active && have_result && lane == 0) {
        p.reward[e] = res_reward;
        p.terminated[e] = (uint8_t)res_term;
        p.win[e] = res_win ? 1 : 0;
        p.target_find[e] = (int32_t)res_found;
    }
    // ---- statistics of episodes that ended in this call: warp reduction, then one atomic per statistic per warp.
    //      Nothing is accumulated for ordinary steps (a same-address atomic per warp per step serialises in L2 and
    //      was the floor of the small configurations); env_steps = sum of finished episode lengths + live time_steps
    //      is assembled by cs_flight_stats.
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
                atomicAdd(p.stats + CS_STAT_EPISODES, (double)st_eps);
                atomicAdd(p.stats + CS_STAT_EP_REWARD, (double)st_rew);
                atomicAdd(p.stats + CS_STAT_TARGETS_FOUND, (double)st_found);
                atomicAdd(p.stats + CS_STAT_WINS, (double)st_wins);
                atomicAdd(p.stats + CS_STAT_EP_LEN, (double)st_len);
            }
        }
    }
}

template <int LPE>
cudaError_t launch_flight(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags,
                          cudaStream_t st) {
    if (h->p.variant) {
        if (mode == MODE_STEP)
            flight_kernel<LPE, MODE_STEP, true><<<h->grid, kThreads, 0, st>>>(h->p, actions, mask, rflags, h->seq);
        else
            flight_kernel<LPE, MODE_RESET, true><<<h->grid, kThreads, 0, st>>>(h->p, actions, mask, rflags, h->seq);
        // the belief maps of the envs the step / reset kernel just sensed (flight_env.py:266)
        const cudaError_t em = launch_map_generic(h, st);
        if (em != cudaSuccess) return em;
    } else {
        if (mode == MODE_STEP)
            flight_kernel<LPE, MODE_STEP, false><<<h->grid, kThreads, 0, st>>>(h->p, actions, mask, rflags, 0u);
        else
            flight_kernel<LPE, MODE_RESET, false><<<h->grid, kThreads, 0, st>>>(h->p, actions, mask, rflags, 0u);
    }
    cs_count_launch(1);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_lpa(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    switch (h->lpe) {
        case 1: return launch_flight<1>(h, mode, actions, mask, rflags, st);
        case 2: return launch_flight<2>(h, mode, actions, mask, rflags, st);
        case 4: return launch_flight<4>(h, mode, actions, mask, rflags, st);
        case 8: return launch_flight<8>(h, mode, actions, mask, rflags, st);
        case 16: return launch_flight<16>(h, mode, actions, mask, rflags, st);
        default: return launch_flight<32>(h, mode, actions, mask, rflags, st);
    }
}

}  // namespace csf
