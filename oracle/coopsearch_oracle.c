/*
 * coopsearch_oracle.c -- plain-C restatement of the reference env-step hot path.
 * TEST INFRASTRUCTURE: this file is the checker, never the product.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.
 *
 * It restates, in float64 with the reference's operation order,
 *   env/flight_env_easy.py:223-314   (_update_obs, _agent_step, _potential_energy_force, step)
 *   env/flight_env.py:232-345        (same + _update_prob_map, _percent_in_agent_viewrange)
 *   env/search_env.py:186-296        (_update_state, _update_obs, get_avail_agent_actions, step)
 * for a BATCH of env instances, so that 4096 x 200-step parity runs finish in seconds (the Python
 * oracle oracle/py_envs.py does ~10^4 env-steps/s).  Squares are taken with pow(v, 2.0) because that
 * is what Python's ** does on floats (SURVEY.md section 8c); the detection draw is the keyed Philox
 * word of oracle/philox.py.
 *
 * PINNING: tests/test_oracle_golden.py::test_c_oracle_* checks this file against the golden
 * trajectories produced by the unmodified reference (tests/golden/ npz files) -- integer state bit-exact,
 * float64 state to 1e-12 -- and against oracle/py_envs.py on random inputs.
 *
 * Build: make -C oracle   (gcc -O2 -shared; no reference sources are compiled or copied).  The C side is
 * single-threaded; oracle/c_oracle.py fans contiguous env blocks out over host threads (ctypes drops the GIL).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define META_FOUND 0
#define META_NEWFOUND 1
#define META_OUT 2
#define META_TIME 3
#define META_EPISODE 4
#define META_FLAGS 5
#define META_EPREWARD 6
#define META_WORDS 8
#define FLAG_WIN 1u
#define FLAG_DONE 2u

#define STREAM_DETECT 1u
#define STREAM_TARGET 2u
#define STREAM_POLICY 3u
#define STREAM_SEARCH 4u
/* key word 1 of a stream: the tag with the episode's bits 16..31 above it (csrc/cs_philox.cuh: cs_stream_key) */
#define STREAM_KEY(stream, episode) ((stream) | ((((uint32_t)(episode)) >> 16) << 8))

typedef struct of_spec {
    int32_t n, m, M, R, T, agent_mode, target_mode, variant, auto_reset;
    double v, detect_prob, safe_dist, force_dist;
    uint32_t seed;
} of_spec;

static void philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

void of_philox(const uint32_t* in6, uint32_t* out4) { philox(in6[0], in6[1], in6[2], in6[3], in6[4], in6[5], out4); }

static double u53(uint32_t hi, uint32_t lo) {
    uint64_t bits = ((uint64_t)(hi >> 5) << 26) + (uint64_t)(lo >> 6);
    return ((double)bits + 0.5) / 9007199254740992.0;
}

static int64_t threshold(double d) {
    if (d >= 1.0) return 0xFFFFFFFFLL;
    if (d < 0.0) return -1;
    return (int64_t)floor(d * 4294967296.0);
}

/* Python float ** 2 is libm pow(v, 2.0) (built with -fno-builtin-pow so that gcc does not fold it into v * v): glibc's pow is
 * not correctly rounded, and pow(v, 2.0) differs from v * v in the last bit for ~0.08 % of arguments (SURVEY.md section 8c).
 * The CUDA kernels square by multiplication; of_set_square(1) makes this oracle do the same, for the tests that demand
 * bit-identical float64 positions from the GPU.  Default 0 = the reference's arithmetic. */
static int g_square_mul = 0;
void of_set_square(int mul) { g_square_mul = mul; }
static double sq(double v) { return g_square_mul ? v * v : pow(v, 2.0); }

/* ---------------------------------------------------------------- belief map (flight_env.py:275-303) */
static int64_t belief_update(const of_spec* s, const double* xy, const double* tgt, uint32_t newf, double* map) {
    const int M = s->M, n = s->n;
    const double R2 = (double)(s->R * s->R);
    const double q = 1 - s->detect_prob;
    int hit[32][2], nh = 0;
    for (int j = 0; j < s->m; ++j)
        if ((newf >> j) & 1u) {
            double tx = tgt[2 * j], ty = tgt[2 * j + 1];
            int ci = (int)(tx > M ? M : tx), cj = (int)(ty > M ? M : ty);   /* int() truncation, then min(.., M-1) */
            hit[nh][0] = ci < M - 1 ? ci : M - 1;
            hit[nh][1] = cj < M - 1 ? cj : M - 1;
            ++nh;
        }
    double lo_x = xy[0], hi_x = xy[0], lo_y = xy[1], hi_y = xy[1];
    for (int a = 1; a < n; ++a) {
        if (xy[2 * a] < lo_x) lo_x = xy[2 * a];
        if (xy[2 * a] > hi_x) hi_x = xy[2 * a];
        if (xy[2 * a + 1] < lo_y) lo_y = xy[2 * a + 1];
        if (xy[2 * a + 1] > hi_y) hi_y = xy[2 * a + 1];
    }
    int i0 = (int)floor(lo_x - s->R) - 1, i1 = (int)ceil(hi_x + s->R);
    int j0 = (int)floor(lo_y - s->R) - 1, j1 = (int)ceil(hi_y + s->R);
    if (i0 < 0) i0 = 0;
    if (j0 < 0) j0 = 0;
    if (i1 > M - 1) i1 = M - 1;
    if (j1 > M - 1) j1 = M - 1;
    int64_t touched = 0;
    for (int i = i0; i <= i1; ++i)
        for (int j = j0; j <= j1; ++j) {
            int inside = 0;
            const int cx[4] = {i, i + 1, i, i + 1}, cy[4] = {j, j, j + 1, j + 1};
            for (int c = 0; c < 4; ++c)
                for (int a = 0; a < n; ++a)
                    if (sq((double)cx[c] - xy[2 * a]) + sq((double)cy[c] - xy[2 * a + 1]) < R2) { ++inside; break; }
            if (!inside) continue;
            ++touched;
            int is_hit = 0;
            for (int k = 0; k < nh; ++k) is_hit |= (hit[k][0] == i && hit[k][1] == j);
            double* cell = map + (size_t)i * M + j;
            if (is_hit) *cell = 1;
            else {
                double p = *cell;
                double frac = inside / 4.0;
                *cell = frac * q * p / (q * p + (1 - p));
            }
        }
    return touched;
}

/* ---------------------------------------------------------------- _update_obs */
static int sense(const of_spec* s, uint32_t env_id, uint32_t t, const double* xy, const double* tgt, uint32_t* meta,
                 uint32_t outbits, double* map, int64_t* touched) {
    const int n = s->n, m = s->m;
    const double R2 = (double)(s->R * s->R);
    const int64_t thr = threshold(s->detect_prob);
    uint32_t found = meta[META_FOUND], newf = 0, flags = meta[META_FLAGS];
    const uint32_t episode = meta[META_EPISODE];
    int rew = -1;
    for (int i = 0; i < n; ++i) {
        const double x = xy[2 * i], y = xy[2 * i + 1];
        for (int j = 0; j < m; ++j) {
            if (sq(tgt[2 * j] - x) + sq(tgt[2 * j + 1] - y) <= R2) {
                uint32_t w[4];
                philox(env_id, ((episode & 0xFFFFu) << 16) | (t & 0xFFFFu), (uint32_t)(i >> 2), (uint32_t)j, s->seed,
                       STREAM_KEY(STREAM_DETECT, episode), w);
                if (!((found >> j) & 1u) && (int64_t)w[i & 3] <= thr) {
                    found |= 1u << j;
                    newf |= 1u << j;
                    rew += 10;
                    if (__builtin_popcount(found) == m && !(flags & FLAG_WIN)) { rew += 100; flags |= FLAG_WIN; }
                }
            }
        }
        if ((outbits >> i) & 1u) rew -= 1;
    }
    meta[META_FOUND] = found; meta[META_NEWFOUND] = newf; meta[META_OUT] = outbits; meta[META_FLAGS] = flags;
    if (s->variant) *touched += belief_update(s, xy, tgt, newf, map);
    return rew;
}

/* ---------------------------------------------------------------- _agent_step */
static uint32_t move(const of_spec* s, double* xy, double* yaw, const uint8_t* act) {
    const int n = s->n;
    const double M = (double)s->M;
    const double turn[3] = {0, M_PI / 18, -M_PI / 18};
    const double fk = s->safe_dist * 0.8 * s->v;
    const double fd2 = sq(s->force_dist);
    uint32_t outbits = 0;
    for (int k = 0; k < n; ++k) {
        const double x0 = xy[2 * k], y0 = xy[2 * k + 1];
        double h = yaw[k] + turn[act[k] < 3 ? act[k] : 0];
        if (h > 2 * M_PI) h -= 2 * M_PI;
        else if (h < 0) h += 2 * M_PI;
        double x = x0 + s->v * cos(h);
        double y = y0 + s->v * sin(h);
        double fx = 0, fy = 0;
        for (int q = 0; q < n; ++q) {
            const double xa = xy[2 * q], ya = xy[2 * q + 1];
            if (q != k && sq(xa - x0) + sq(ya - y0) < fd2 && (xa != x0 || ya != y0)) {
                fx += fk * (x0 - xa) / (sq(x0 - xa) + sq(y0 - ya));
                fy += fk * (y0 - ya) / (sq(x0 - xa) + sq(y0 - ya));
            }
        }
        x += fx; y += fy;
        const int outside = s->variant ? (x < 0 || x >= M || y < 0 || y >= M) : (x < 0 || x > M || y < 0 || y > M);
        if (outside) {
            x = x < 0 ? 0 : (x > M ? M : x);
            y = y < 0 ? 0 : (y > M ? M : y);
            h = (h <= M_PI) ? M_PI - h : 3 * M_PI - h;
            outbits |= 1u << k;
        }
        xy[2 * k] = x; xy[2 * k + 1] = y; yaw[k] = h;
    }
    return outbits;
}

static void place(const of_spec* s, uint32_t env_id, const double* tmpl, int keep_targets, int keep_episode, int init,
                  double* xy, double* yaw, double* tgt, uint32_t* meta, double* map) {
    const int n = s->n, m = s->m;
    const double M = (double)s->M;
    const uint32_t episode = meta[META_EPISODE] + (keep_episode ? 0u : 1u);
    memset(meta, 0, META_WORDS * sizeof(uint32_t));
    meta[META_EPISODE] = episode;
    if (!keep_targets)
        for (int j = 0; j < m; ++j) {
            uint32_t w[4];
            philox(env_id, (episode & 0xFFFFu) << 16, (uint32_t)j, 0u, s->seed, STREAM_KEY(STREAM_TARGET, episode), w);
            const double u1 = u53(w[0], w[1]), u2 = u53(w[2], w[3]);
            double x, y;
            if (s->target_mode == 0) {
                x = tmpl[5 * j]; y = tmpl[5 * j + 1];
                if (tmpl[5 * j + 4] != 0.0) {
                    const double rad = sqrt(-2.0 * log(u1)), ang = 2.0 * M_PI * u2;
                    x += tmpl[5 * j + 2] * 2 * (rad * cos(ang) - 0.5);
                    y += tmpl[5 * j + 3] * 2 * (rad * sin(ang) - 0.5);
                }
            } else { x = M * u1; y = M * u2; }
            tgt[2 * j] = x; tgt[2 * j + 1] = y;
        }
    for (int a = 0; a < n; ++a) {
        const double lin = (n != 1) ? (double)(a * s->M) / (double)(n - 1) : M / 2;
        switch (s->agent_mode) {
            case 0: xy[2 * a] = lin; xy[2 * a + 1] = 0; yaw[a] = M_PI / 2; break;
            case 1: xy[2 * a] = lin; xy[2 * a + 1] = M / 2; yaw[a] = M_PI / 2; break;
            case 2: xy[2 * a] = 0; xy[2 * a + 1] = lin; yaw[a] = 0; break;
            default: xy[2 * a] = M; xy[2 * a + 1] = lin; yaw[a] = M_PI; break;
        }
    }
    if (s->variant && init)
        for (int c = 0; c < s->M * s->M; ++c) map[c] = 0.5;
}

/* tmpl rows already scaled by a = M/10: x, y, sx, sy, random */
void of_flight_reset(const of_spec* s, int E, uint32_t base, const double* tmpl, const uint8_t* mask, int keep_targets,
                     int keep_episode, int init, double* xy, double* yaw, double* tgt, uint32_t* meta, double* map,
                     int64_t* touched) {
    for (int e = 0; e < E; ++e) {
        if (mask && !mask[e]) continue;
        double* mp = s->variant ? map + (size_t)e * s->M * s->M : NULL;
        int64_t tc = 0;
        place(s, base + e, tmpl, keep_targets, keep_episode, init, xy + (size_t)e * 2 * s->n, yaw + (size_t)e * s->n,
              tgt + (size_t)e * 2 * s->m, meta + (size_t)e * META_WORDS, mp);
        (void)sense(s, base + e, 0, xy + (size_t)e * 2 * s->n, tgt + (size_t)e * 2 * s->m, meta + (size_t)e * META_WORDS, 0, mp, &tc);
        if (touched) *touched += tc;
    }
}

/* actions == NULL: uniform-random policy from the keyed stream (same words as the CUDA kernel) */
void of_flight_step(const of_spec* s, int E, uint32_t base, const double* tmpl, const uint8_t* actions, double* xy,
                    double* yaw, double* tgt, uint32_t* meta, double* map, double* reward, uint8_t* terminated,
                    uint8_t* win, int64_t* touched) {
    for (int e = 0; e < E; ++e) {
        uint32_t* mt = meta + (size_t)e * META_WORDS;
        double* pxy = xy + (size_t)e * 2 * s->n;
        double* pyaw = yaw + (size_t)e * s->n;
        double* ptg = tgt + (size_t)e * 2 * s->m;
        double* mp = s->variant ? map + (size_t)e * s->M * s->M : NULL;
        int64_t tc = 0;
        int done = (mt[META_FLAGS] & FLAG_DONE) != 0;
        if (!done) {
            uint8_t buf[32];
            const uint8_t* act = actions ? actions + (size_t)e * s->n : buf;
            if (!actions)
                for (int a = 0; a < s->n; ++a) {
                    uint32_t w[4];
                    philox(base + e, ((mt[META_EPISODE] & 0xFFFFu) << 16) | ((mt[META_TIME] + 1u) & 0xFFFFu), (uint32_t)(a >> 2),
                           0u, s->seed, STREAM_KEY(STREAM_POLICY, mt[META_EPISODE]), w);
                    buf[a] = (uint8_t)(w[a & 3] % 3u);
                }
            const uint32_t outbits = move(s, pxy, pyaw, act);
            const int rew = sense(s, base + e, mt[META_TIME] + 1u, pxy, ptg, mt, outbits, mp, &tc);
            mt[META_TIME] += 1;
            const int term = __builtin_popcount(mt[META_FOUND]) >= s->m || (int)mt[META_TIME] >= s->T;
            if (term) mt[META_FLAGS] |= FLAG_DONE;
            reward[e] = rew; terminated[e] = (uint8_t)term; win[e] = (mt[META_FLAGS] & FLAG_WIN) ? 1 : 0;
            done = term;
        } else {
            reward[e] = 0; terminated[e] = 1; win[e] = (mt[META_FLAGS] & FLAG_WIN) ? 1 : 0;
        }
        if (s->auto_reset && done) {
            place(s, base + e, tmpl, 0, 0, 0, pxy, pyaw, ptg, mt, mp);
            (void)sense(s, base + e, 0, pxy, ptg, mt, 0, mp, &tc);
        }
        if (touched && tc) *touched += tc;
    }
}

/* get_obs / get_state (flight_env_easy.py:190-221), float64 like the reference */
void of_flight_obs_state(const of_spec* s, int E, const double* xy, const double* yaw, const double* tgt,
                         const uint32_t* meta, double* obs, double* state) {
    const int n = s->n, m = s->m, S = 4 * n + 3 * m;
    const double M = (double)s->M;
    for (int e = 0; e < E; ++e) {
        const uint32_t found = meta[(size_t)e * META_WORDS + META_FOUND];
        for (int a = 0; a < n; ++a) {
            const double x = xy[((size_t)e * n + a) * 2], y = xy[((size_t)e * n + a) * 2 + 1], h = yaw[(size_t)e * n + a];
            const double f[4] = {(x - 0.5 * M) / (M / 2), (y - 0.5 * M) / (M / 2), cos(h), sin(h)};
            for (int k = 0; k < 4; ++k) {
                if (obs) obs[((size_t)e * n + a) * 4 + k] = f[k];
                if (state) state[(size_t)e * S + 4 * a + k] = f[k];
            }
        }
        if (state)
            for (int j = 0; j < m; ++j) {
                state[(size_t)e * S + 4 * n + 3 * j + 0] = (tgt[((size_t)e * m + j) * 2] - 0.5 * M) / (M / 2);
                state[(size_t)e * S + 4 * n + 3 * j + 1] = (tgt[((size_t)e * m + j) * 2 + 1] - 0.5 * M) / (M / 2);
                state[(size_t)e * S + 4 * n + 3 * j + 2] = ((found >> j) & 1u) ? 1.0 : 0.0;
            }
    }
}

/* =====================================================================================
 * search_env
 * ===================================================================================== */
typedef struct os_spec {
    int32_t n, m, M, R, agent_mode, target_mode, auto_reset;
    uint32_t seed;
} os_spec;

/* counters[e][4]: target_find, time_step, flags (1 done, 2 illegal), episode */
static void search_place_agents(const os_spec* s, int32_t* pos, int32_t* freq) {
    const int n = s->n, M = s->M;
    int cnt = 0;
    if (s->agent_mode == 0) {
        const int L = (int)ceil(sqrt((double)n)), b = (M - L) / 2;
        for (int i = b; i < b + L; ++i)
            for (int j = b; j < b + L; ++j)
                if (cnt < n) { pos[2 * cnt] = i; pos[2 * cnt + 1] = j; ++cnt; }
    } else if (s->agent_mode == 1) {
        const int L = (int)ceil(sqrt((double)n));
        for (int i = M - 1; i > M - 1 - L; --i)
            for (int j = 0; j < L; ++j)
                if (cnt < n) { pos[2 * cnt] = i; pos[2 * cnt + 1] = j; ++cnt; }
    } else {
        const int gap = (M - 1) / (n - 1);
        for (int i = 0; i < n; ++i) { pos[2 * i] = M - 1; pos[2 * i + 1] = i * gap; }
    }
    for (int a = 0; a < n; ++a) freq[pos[2 * a] * M + pos[2 * a + 1]] += 1;
}

static void search_place_targets(const os_spec* s, uint32_t env_id, uint32_t episode, int32_t* cells, uint8_t* tmap) {
    const int M = s->M, lo = M / 4, hi = 3 * M / 4;
    int got = 0;
    uint32_t k = 0;
    while (got < s->m) {
        uint32_t w[4];
        philox(env_id, (episode & 0xFFFFu) << 16, k++, 0u, s->seed, STREAM_KEY(STREAM_SEARCH, episode), w);
        const int x = (int)(w[0] % (uint32_t)M), y = (int)(w[1] % (uint32_t)M);
        if (tmap[x * M + y]) continue;
        if (s->target_mode == 1 && !(x <= lo || x >= hi || y <= lo || y >= hi)) continue;
        tmap[x * M + y] = 1;
        cells[2 * got] = x; cells[2 * got + 1] = y; ++got;
    }
}

/* reset of env e (search_env.py:69-183, init=False): the next episode, its targets, agents at their start cells */
static void search_reset_env(const os_spec* s, int e, uint32_t env_id, int keep_targets, int32_t* pos, int32_t* cells,
                             uint8_t* tmap, uint8_t* found, int32_t* freq, int32_t* counters) {
    const int M = s->M;
    int32_t* ct = counters + (size_t)e * 4;
    uint8_t* tm = tmap + (size_t)e * M * M;
    ct[0] = 0; ct[1] = 0; ct[2] = 0; ct[3] += 1;
    memset(tm, 0, (size_t)M * M);
    memset(found + (size_t)e * s->m, 0, s->m);
    if (keep_targets) {
        for (int k = 0; k < s->m; ++k) tm[cells[((size_t)e * s->m + k) * 2] * M + cells[((size_t)e * s->m + k) * 2 + 1]] = 1;
    } else {
        search_place_targets(s, env_id, (uint32_t)ct[3], cells + (size_t)e * s->m * 2, tm);
    }
    search_place_agents(s, pos + (size_t)e * s->n * 2, freq + (size_t)e * M * M);
}

void os_reset(const os_spec* s, int E, uint32_t base, const uint8_t* mask, int keep_targets, int32_t* pos, int32_t* cells,
              uint8_t* tmap, uint8_t* found, int32_t* freq, int32_t* counters) {
    for (int e = 0; e < E; ++e)
        if (!mask || mask[e]) search_reset_env(s, e, base + e, keep_targets, pos, cells, tmap, found, freq, counters);
}

/* step (search_env.py:246-296).  terms (may be NULL): [E][n+2] the reward's terms of this call, -1, 1/freq of each agent
 * and 10 * (targets found), zeros for an env that did not step; find_out (may be NULL): [E] target_find after the step of
 * the finished episode.  With s->auto_reset a terminating env is reset within the call, like the kernel: counters, agents,
 * targets and found flags then hold the new episode, reward / terminated / terms / find_out the finished one's step. */
void os_step(const os_spec* s, int E, uint32_t base, const uint8_t* actions, int32_t* pos, int32_t* cells, uint8_t* tmap,
             uint8_t* found, int32_t* freq, int32_t* counters, double* reward, uint8_t* terminated, double* terms,
             int32_t* find_out) {
    const int n = s->n, m = s->m, M = s->M, R2 = s->R * s->R;
    for (int e = 0; e < E; ++e) {
        int32_t* ct = counters + (size_t)e * 4;
        int32_t* p = pos + (size_t)e * n * 2;
        int32_t* fq = freq + (size_t)e * M * M;
        double* tr = terms ? terms + (size_t)e * (n + 2) : NULL;
        if (tr) memset(tr, 0, sizeof(double) * (size_t)(n + 2));
        if (ct[2] & 1) {
            reward[e] = 0; terminated[e] = 1;
            if (find_out) find_out[e] = ct[0];
            if (s->auto_reset) search_reset_env(s, e, base + e, 0, pos, cells, tmap, found, freq, counters);
            continue;
        }
        double rew = -1;
        int newfound = 0;
        ct[1] += 1;
        for (int i = 0; i < n; ++i) {
            uint8_t a;
            if (actions) a = actions[(size_t)e * n + i];
            else {
                /* uniform over the AVAILABLE moves (agent.py:34-36 picks among avail actions) */
                uint32_t w[4];
                philox(base + e, (((uint32_t)ct[3] & 0xFFFFu) << 16) | ((uint32_t)ct[1] & 0xFFFFu), (uint32_t)(i >> 2), 0u, s->seed,
                       STREAM_KEY(STREAM_POLICY, ct[3]), w);
                const int av[4] = {p[2 * i] > 0, p[2 * i + 1] > 0, p[2 * i] < M - 1, p[2 * i + 1] < M - 1};
                const int na = av[0] + av[1] + av[2] + av[3];
                int pick = (int)(w[i & 3] % (uint32_t)na);
                a = 0;
                for (int k = 0; k < 4; ++k)
                    if (av[k]) { if (pick == 0) { a = (uint8_t)k; break; } --pick; }
            }
            const int x = p[2 * i], y = p[2 * i + 1];
            if (a == 0 && x > 0) p[2 * i] -= 1;
            else if (a == 1 && y > 0) p[2 * i + 1] -= 1;
            else if (a == 2 && x < M - 1) p[2 * i] += 1;
            else if (a == 3 && y < M - 1) p[2 * i + 1] += 1;
            else { ct[2] |= 2; continue; }
            fq[p[2 * i] * M + p[2 * i + 1]] += 1;
        }
        for (int i = 0; i < n; ++i) {
            const int xa = p[2 * i], ya = p[2 * i + 1];
            rew += 1 / (double)fq[xa * M + ya];
            if (tr) tr[1 + i] = 1 / (double)fq[xa * M + ya];
            for (int k = 0; k < m; ++k) {
                const int dx = cells[((size_t)e * m + k) * 2] - xa, dy = cells[((size_t)e * m + k) * 2 + 1] - ya;
                if (dx * dx + dy * dy <= R2 && !found[(size_t)e * m + k]) {
                    rew += 10;
                    found[(size_t)e * m + k] = 1;
                    ct[0] += 1;
                    ++newfound;
                }
            }
        }
        if (tr) { tr[0] = -1; tr[n + 1] = 10.0 * newfound; }
        const int term = ct[0] >= m;
        if (term) ct[2] |= 1;
        reward[e] = rew;
        terminated[e] = (uint8_t)term;
        if (find_out) find_out[e] = ct[0];
        if (term && s->auto_reset) search_reset_env(s, e, base + e, 0, pos, cells, tmap, found, freq, counters);
    }
}

/* get_obs (search_env.py:203-227), get_state (:186-200), avail (:230-243); float32 outputs */
void os_views(const os_spec* s, int E, const int32_t* pos, const uint8_t* tmap, float* obs, float* state, uint8_t* avail) {
    const int n = s->n, M = s->M, R = s->R, S = 2 * R - 1, W = S * S + 2;
    for (int e = 0; e < E; ++e) {
        const uint8_t* tm = tmap + (size_t)e * M * M;
        const int32_t* p = pos + (size_t)e * n * 2;
        if (state) {
            float* st = state + (size_t)e * 2 * M * M;
            for (int c = 0; c < M * M; ++c) { st[2 * c] = tm[c] ? 1.f : 0.f; st[2 * c + 1] = 0.f; }
            for (int a = 0; a < n; ++a) st[2 * (p[2 * a] * M + p[2 * a + 1]) + 1] = 1.f;
        }
        for (int a = 0; a < n; ++a) {
            const int x = p[2 * a], y = p[2 * a + 1];
            if (obs) {
                float* o = obs + ((size_t)e * n + a) * W;
                for (int i = 0; i < S; ++i)
                    for (int j = 0; j < S; ++j) {
                        const int gx = i + x - R + 1, gy = j + y - R + 1;
                        float v = 0.f;
                        if (gx >= 0 && gx < M && gy >= 0 && gy < M) {
                            if ((R - 1 - i) * (R - 1 - i) + (R - 1 - j) * (R - 1 - j) > R * R) v = 0.5f;
                            else if (tm[gx * M + gy]) v = 1.f;
                        } else v = 0.5f;
                        o[i * S + j] = v;
                    }
                o[S * S] = (float)x; o[S * S + 1] = (float)y;
            }
            if (avail) {
                uint8_t* av = avail + ((size_t)e * n + a) * 4;
                av[0] = x > 0; av[1] = y > 0; av[2] = x < M - 1; av[3] = y < M - 1;
            }
        }
    }
}
