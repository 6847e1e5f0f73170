// search_env discrete-grid env-step hot path for B200 (sm_100a).
//
// Restates (reference: WZN1ng/Cooperative-Search, env/search_env.py):
//   reset                      :69-183   (agent layouts :146-180; target modes 0/1 :86-104)
//   _agent_step + step         :246-296  (move, freq_map, 1/freq reward, disc detection)
//   _update_obs / get_obs      :203-227  ((2R-1)^2 window + raw position)
//   _update_state / get_state  :186-200  (plane 0 targets (sticky), plane 1 agents)
//   get_avail_agent_actions    :230-243
//
// Design: one CTA (128 threads) per env instance.  Target presence and "not yet found" live as bit
// rows (one bit per cell) staged in shared memory; detection is an atomicAnd of each agent's disc row
// masks against the unfound rows (the returned old word says which targets THIS agent found, so
// simultaneous sightings are counted once); observation windows and the two state planes are emitted
// with fully coalesced stores straight from the bit rows.  The path is write-bandwidth bound:
// ~4n((2R-1)^2+2) + 8M^2 bytes per env-step (DESIGN.md section 5).
#include <math.h>
#include <new>
#include "cs_common.cuh"
#include "cs_philox.cuh"

namespace {

constexpr int kThreads = 128;
enum { CNT_FIND = 0, CNT_TIME = 1, CNT_FLAGS = 2, CNT_EPISODE = 3 };
enum : int { SF_DONE = 1, SF_ILLEGAL = 2 };
enum { MODE_STEP = 0, MODE_RESET = 1 };

struct SearchParams {
    int E, n, m, M, R, W;            // W = words per bit row
    int S, obs_len;                  // S = 2R-1, obs_len = S*S+2
    int agent_mode, target_mode, auto_reset;
    int stage_obs;                   // 1: observation block staged in shared memory (M <= 64 and it fits)
    uint32_t mg_half, mg_M, mg_S1, mg_span;   // ceil(2^32/d) for d = M/2, M, S+1, 2R+1
    uint32_t seed, env_id_base;
    int32_t* pos;
    uint32_t* target_bits;
    uint32_t* unfound_bits;
    int32_t* freq;
    int32_t* counters;
    const int32_t* cells;            // injected target cells [E][m][2] or nullptr
    float* obs;
    float* state;
    uint8_t* avail;
    float* reward;
    uint8_t* terminated;
    int32_t* target_find;
    double* stats;
    double* ep_reward;               // [E] fp64 sum of the running episode's step rewards -> CS_STAT_EP_REWARD
    int place_batches;               // cap on 128-candidate batches of target placement (search_init)
};

struct SearchSmem {
    uint32_t* tbits;     // [M*W]
    uint32_t* ubits;     // [M*W]
    uint32_t* abits;     // [M*W] agent presence
    int32_t* pos;        // [2n]
    int32_t* cand;       // [2*kThreads] candidate cells during target placement
    int* scal;           // [8]
    uint32_t* discmask;  // [S]   bit j set: window cell (i, j) lies outside the disc -> 0.5 (search_env.py:221-222)
    int* halfw;          // [2R+1] half width of the disc row at |dx| (detection, :263)
    uint8_t* obs_stage;  // [n*obs_len] bytes = 2*value of the observation block (0, 0.5, 1 and raw positions < 128),
                         // or nullptr (direct path)
};

__device__ __forceinline__ SearchSmem carve(const SearchParams& p, unsigned char* raw) {
    SearchSmem s;
    const int rows = p.M * p.W;
    s.tbits = reinterpret_cast<uint32_t*>(raw);
    s.ubits = s.tbits + rows;
    s.abits = s.ubits + rows;
    s.pos = reinterpret_cast<int32_t*>(s.abits + rows);
    s.cand = s.pos + 2 * p.n;
    s.scal = s.cand + 2 * kThreads;
    s.discmask = reinterpret_cast<uint32_t*>(s.scal + 8);
    s.halfw = reinterpret_cast<int*>(s.discmask + p.S);
    // 16-byte aligned staging block after the integer scratch
    const size_t used = sizeof(uint32_t) * (size_t)(3 * rows) + sizeof(int32_t) * (size_t)(2 * p.n + 2 * kThreads + 8 + p.S + 2 * p.R + 1);
    s.obs_stage = p.stage_obs ? reinterpret_cast<uint8_t*>(raw + ((used + 15) & ~(size_t)15)) : nullptr;
    return s;
}
size_t smem_base_bytes(const SearchParams& p) {
    const size_t used = sizeof(uint32_t) * (size_t)(3 * p.M * p.W) + sizeof(int32_t) * (size_t)(2 * p.n + 2 * kThreads + 8 + p.S + 2 * p.R + 1);
    return (used + 15) & ~(size_t)15;
}
// cells of the target_mode 1 edge band: x or y <= M/4 or >= 3M/4 (search_env.py:96-104)
int search_band_cells(int M) {
    const int inner = 3 * M / 4 - M / 4 - 1;
    return M * M - (inner > 0 ? inner * inner : 0);
}
// v / d with magic = ceil(2^32 / d); d == 1 gives magic 2^32 -> stored as 0 -> identity
__device__ __forceinline__ int fastdiv(int v, uint32_t magic) { return magic ? (int)__umulhi((uint32_t)v, magic) : v; }

// scal slots
enum { SC_NEWFOUND = 0, SC_ILLEGAL = 1, SC_GOT = 2, SC_NEXTK = 3 };

// ---- reset of one env by its CTA (search_env.py:69-183, init=False semantics) ------------------------
__device__ void search_reset(const SearchParams& p, const SearchSmem& s, int e, uint32_t rflags, int32_t* cnt_local) {
    const int tid = threadIdx.x, M = p.M, W = p.W, n = p.n;
    const int rows = M * W;
    const uint32_t env_id = p.env_id_base + (uint32_t)e;
    const int episode = cnt_local[CNT_EPISODE] + ((rflags & CS_RESET_KEEP_EPISODE) ? 0 : 1);
    for (int k = tid; k < rows; k += kThreads) { s.tbits[k] = 0; s.abits[k] = 0; }
    if (tid == 0) { s.scal[SC_GOT] = 0; s.scal[SC_NEXTK] = 0; }
    __syncthreads();
    if (rflags & CS_RESET_KEEP_TARGETS) {
        const int32_t* c = p.cells + (size_t)e * p.m * 2;
        for (int k = tid; k < p.m; k += kThreads) {
            const int x = c[2 * k], y = c[2 * k + 1];
            if (x >= 0 && x < M && y >= 0 && y < M) atomicOr(&s.tbits[x * W + (y >> 5)], 1u << (y & 31));
        }
    } else {
        // Rejection sampling in candidate order k = 0,1,...: candidate k is Philox(env, episode, k) ->
        // (w0 % M, w1 % M); accepted when the cell is free (mode 1: and in the edge band) -- the accept rule of
        // search_env.py:86-104.  Philox for a batch of candidates in parallel, acceptance in order by thread 0.
        // cs_search_create refuses requests that cannot be met; place_batches bounds the loop so that a met request
        // always completes (search_init states the bound) and nothing can spin forever
        const int lo = M / 4, hi = 3 * M / 4;
        for (int batch = 0; batch < p.place_batches; ++batch) {
            const int base = s.scal[SC_NEXTK];
            const cs_u4 w = cs_philox4x32_10(env_id, ((uint32_t)episode & 0xFFFFu) << 16, (uint32_t)(base + tid), 0u, p.seed,
                                             cs_stream_key(CS_STREAM_SEARCH, (uint32_t)episode));
            s.cand[2 * tid] = (int)(w.x % (uint32_t)M);
            s.cand[2 * tid + 1] = (int)(w.y % (uint32_t)M);
            __syncthreads();
            if (tid == 0) {
                int got = s.scal[SC_GOT];
                for (int k = 0; k < kThreads && got < p.m; ++k) {
                    const int x = s.cand[2 * k], y = s.cand[2 * k + 1];
                    const uint32_t bit = 1u << (y & 31);
                    uint32_t* word = &s.tbits[x * W + (y >> 5)];
                    if (*word & bit) continue;
                    if (p.target_mode == 1 && !(x <= lo || x >= hi || y <= lo || y >= hi)) continue;
                    *word |= bit;
                    ++got;
                }
                s.scal[SC_GOT] = got;
                s.scal[SC_NEXTK] = base + kThreads;
            }
            __syncthreads();
            if (s.scal[SC_GOT] >= p.m) break;
        }
    }
    __syncthreads();
    for (int k = tid; k < rows; k += kThreads) s.ubits[k] = s.tbits[k];
    // agent layouts (:146-180)
    for (int a = tid; a < n; a += kThreads) {
        int x, y;
        if (p.agent_mode == 0) {
            const int L = (int)ceil(sqrt((double)n)), b = (M - L) / 2;
            x = b + a / L; y = b + a % L;
        } else if (p.agent_mode == 1) {
            const int L = (int)ceil(sqrt((double)n));
            x = M - 1 - a / L; y = a % L;
        } else {
            const int gap = (M - 1) / (n - 1);
            x = M - 1; y = a * gap;
        }
        s.pos[2 * a] = x; s.pos[2 * a + 1] = y;
        atomicAdd(&p.freq[(size_t)e * M * M + x * M + y], 1);         // freq_map is never cleared (:39 vs :70-80)
    }
    if (tid == 0) {
        cnt_local[CNT_FIND] = 0; cnt_local[CNT_TIME] = 0; cnt_local[CNT_FLAGS] = 0; cnt_local[CNT_EPISODE] = episode;
        p.ep_reward[e] = 0.0;
    }
    __syncthreads();
}

// ---- get_obs / get_state / avail of one env (:186-243) ------------------------------------------------
__device__ __forceinline__ uint32_t bit_at(const uint32_t* rows, int W, int x, int y) {
    return (rows[x * W + (y >> 5)] >> (y & 31)) & 1u;
}

__device__ void search_emit(const SearchParams& p, const SearchSmem& s, int e) {
    const int tid = threadIdx.x, M = p.M, W = p.W, n = p.n, R = p.R, S = p.S;
    const int rows = M * W;
    for (int k = tid; k < rows; k += kThreads) s.abits[k] = 0;
    __syncthreads();
    for (int a = tid; a < n; a += kThreads) {
        const int x = s.pos[2 * a], y = s.pos[2 * a + 1];
        atomicOr(&s.abits[x * W + (y >> 5)], 1u << (y & 31));
        uint8_t* av = p.avail + ((size_t)e * n + a) * 4;
        *reinterpret_cast<uchar4*>(av) = make_uchar4(x > 0, y > 0, x < M - 1, y < M - 1);
    }
    __syncthreads();
    // state [M][M][2]: plane 0 targets (found ones stay 1), plane 1 agents; two cells = one 16-byte store
    if ((M & 1) == 0) {
        float4* st = reinterpret_cast<float4*>(p.state + (size_t)e * 2 * M * M);
        const int half = M >> 1;
        for (int c2 = tid; c2 < M * half; c2 += kThreads) {
            const int x = fastdiv(c2, p.mg_half), y = (c2 - x * half) * 2;
            const uint32_t tw = s.tbits[x * W + (y >> 5)] >> (y & 31), aw = s.abits[x * W + (y >> 5)] >> (y & 31);
            st[c2] = make_float4((float)(tw & 1u), (float)(aw & 1u), (float)((tw >> 1) & 1u), (float)((aw >> 1) & 1u));
        }
    } else {
        float2* st = reinterpret_cast<float2*>(p.state + (size_t)e * 2 * M * M);
        for (int c = tid; c < M * M; c += kThreads) {
            const int x = fastdiv(c, p.mg_M), y = c - x * M;
            st[c] = make_float2((float)bit_at(s.tbits, W, x, y), (float)bit_at(s.abits, W, x, y));
        }
    }
    // obs [n][S*S+2]: one thread per (agent, window row) builds the row from the target bit row, staged in shared
    // memory (conflict-free: consecutive tasks are S words apart, S odd), then copied out with 16-byte stores.
    float* ob = p.obs + (size_t)e * n * p.obs_len;
    const int R2 = R * R;
    if (s.obs_stage != nullptr) {
        const int tasks = n * (S + 1);
        for (int t = tid; t < tasks; t += kThreads) {
            const int a = fastdiv(t, p.mg_S1), i = t - a * (S + 1);
            const int x = s.pos[2 * a], y = s.pos[2 * a + 1];
            uint8_t* o = s.obs_stage + a * p.obs_len;
            if (i == S) {                                              // raw integer position (:205-208)
                o[S * S] = (uint8_t)(2 * x);
                o[S * S + 1] = (uint8_t)(2 * y);
                continue;
            }
            const int gx = i + x - R + 1, gy0 = y - R + 1;
            unsigned long long field = 0ull;
            const bool row_ok = gx >= 0 && gx < M;
            if (row_ok) {
                unsigned long long row = s.tbits[gx * W];
                if (W > 1) row |= (unsigned long long)s.tbits[gx * W + 1] << 32;
                field = gy0 >= 0 ? (row >> gy0) : (row << (-gy0));
            }
            // columns inside the map: j in [max(0,-gy0), min(S-1, M-1-gy0)]; everything else, everything outside the
            // disc and every off-map row reads 0.5 (:220-226).  Staged byte = 2*value.
            const int jlo = max(0, -gy0), jhi = min(S - 1, M - 1 - gy0);
            uint32_t inmap = 0;
            if (row_ok && jlo <= jhi) inmap = (jhi >= 31 ? 0xffffffffu : ((2u << jhi) - 1u)) & ~((1u << jlo) - 1u);
            const uint32_t halfm = ~inmap | s.discmask[i];
            const uint32_t ones = (uint32_t)field & ~halfm;
            uint8_t* orow = o + i * S;
            for (int j = 0; j < S; ++j)
                orow[j] = (uint8_t)(((halfm >> j) & 1u) + 2u * ((ones >> j) & 1u));
        }
        __syncthreads();
        const int total = n * p.obs_len;
        if ((total & 3) == 0) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(s.obs_stage);
            float4* dst = reinterpret_cast<float4*>(ob);
            for (int k = tid; k < (total >> 2); k += kThreads) {
                const uint32_t w = src[k];
                dst[k] = make_float4(0.5f * (float)(w & 0xffu), 0.5f * (float)((w >> 8) & 0xffu),
                                     0.5f * (float)((w >> 16) & 0xffu), 0.5f * (float)(w >> 24));
            }
        } else {
            for (int k = tid; k < total; k += kThreads) ob[k] = 0.5f * (float)s.obs_stage[k];
        }
    } else {
        // large maps / very many agents: direct per-element path
        const int total = n * p.obs_len;
        for (int idx = tid; idx < total; idx += kThreads) {
            const int a = idx / p.obs_len, k = idx - a * p.obs_len;
            const int x = s.pos[2 * a], y = s.pos[2 * a + 1];
            float v;
            if (k >= S * S) {
                v = (float)(k == S * S ? x : y);
            } else {
                const int i = k / S, j = k - i * S;
                const int gx = i + x - R + 1, gy = j + y - R + 1;
                const int di = R - 1 - i, dj = R - 1 - j;
                if (gx < 0 || gx >= M || gy < 0 || gy >= M || di * di + dj * dj > R2) v = 0.5f;
                else v = (float)bit_at(s.tbits, W, gx, gy);
            }
            ob[idx] = v;
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(kThreads) search_kernel(const SearchParams p, const uint8_t* __restrict__ actions,
                                                          const uint8_t* __restrict__ mask, uint32_t rflags, int random_policy) {
    extern __shared__ __align__(16) unsigned char raw[];
    __shared__ int32_t cnt[4];
    __shared__ double s_red[kThreads / 32];
    __shared__ double s_ep_reward;
    const SearchSmem s = carve(p, raw);
    const int tid = threadIdx.x, e = blockIdx.x, M = p.M, W = p.W, n = p.n;
    const int rows = M * W;
    const uint32_t env_id = p.env_id_base + (uint32_t)e;
    if (MODE == MODE_RESET && mask != nullptr && mask[e] == 0) return;

    if (tid < 4) cnt[tid] = p.counters[(size_t)e * 4 + tid];
    if (tid == 0) { s.scal[SC_NEWFOUND] = 0; s.scal[SC_ILLEGAL] = 0; }
    {
        const uint32_t* gt = p.target_bits + (size_t)e * rows;
        const uint32_t* gu = p.unfound_bits + (size_t)e * rows;
        for (int k = tid; k < rows; k += kThreads) { s.tbits[k] = gt[k]; s.ubits[k] = gu[k]; }
        const int32_t* gp = p.pos + (size_t)e * 2 * n;
        for (int k = tid; k < 2 * n; k += kThreads) s.pos[k] = gp[k];
        const int R = p.R, R2 = R * R;
        for (int i = tid; i < p.S; i += kThreads) {              // window rows: which columns fall outside the disc
            uint32_t mk = 0;
            const int di = R - 1 - i;
            for (int j = 0; j < p.S && j < 32; ++j) {
                const int dj = R - 1 - j;
                if (di * di + dj * dj > R2) mk |= 1u << j;
            }
            s.discmask[i] = mk;
        }
        for (int d = tid; d <= 2 * R; d += kThreads) {           // detection rows: half width at dx = d - R
            const int dx = d - R;
            int w = 0;
            while ((w + 1) * (w + 1) + dx * dx <= R2) ++w;
            s.halfw[d] = w;
        }
    }
    __syncthreads();

    bool emit = false, bits_dirty = false;
    if (MODE == MODE_STEP) {
        bool done = (cnt[CNT_FLAGS] & SF_DONE) != 0;
        if (!done) {
            int32_t* fq = p.freq + (size_t)e * M * M;
            const int t1 = cnt[CNT_TIME] + 1;
            // ---- _agent_step (:280-296)
            for (int a = tid; a < n; a += kThreads) {
                int x = s.pos[2 * a], y = s.pos[2 * a + 1];
                int act;
                if (!random_policy) {
                    act = actions[(size_t)e * n + a];
                } else {
                    const cs_u4 w = cs_philox4x32_10(env_id, (((uint32_t)cnt[CNT_EPISODE] & 0xFFFFu) << 16) | ((uint32_t)t1 & 0xFFFFu),
                                                     (uint32_t)(a >> 2), 0u, p.seed, cs_stream_key(CS_STREAM_POLICY, (uint32_t)cnt[CNT_EPISODE]));
                    const int av0 = x > 0, av1 = y > 0, av2 = x < M - 1, av3 = y < M - 1;
                    int pick = (int)(cs_word(w, a & 3) % (uint32_t)(av0 + av1 + av2 + av3));
                    act = 0;
                    if (av0) { if (pick == 0) act = 0; --pick; }
                    if (av1 && pick >= 0) { if (pick == 0) act = 1; --pick; }
                    if (av2 && pick >= 0) { if (pick == 0) act = 2; --pick; }
                    if (av3 && pick >= 0) { if (pick == 0) act = 3; --pick; }
                }
                bool ok = true;
                if (act == 0 && x > 0) x -= 1;
                else if (act == 1 && y > 0) y -= 1;
                else if (act == 2 && x < M - 1) x += 1;
                else if (act == 3 && y < M - 1) y += 1;
                else ok = false;                                    // reference raises (:293): flag, agent stays
                if (ok) {
                    s.pos[2 * a] = x; s.pos[2 * a + 1] = y;
                    atomicAdd(&fq[x * M + y], 1);
                } else {
                    atomicOr(&s.scal[SC_ILLEGAL], 1);
                }
            }
            __syncthreads();
            if (tid == 32) s_ep_reward = p.ep_reward[e];     // the episode's reward so far, loaded while detection runs
            // ---- reward: sum_i 1/freq[p_i] in fp64 (:257-259)
            double part = 0.0;
            for (int a = tid; a < n; a += kThreads) part += 1.0 / (double)__ldcg(&fq[s.pos[2 * a] * M + s.pos[2 * a + 1]]);
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            if ((tid & 31) == 0) s_red[tid >> 5] = part;
            // ---- detection: disc rows of every agent against the unfound bit rows (:261-267)
            const int R = p.R, span = 2 * R + 1;
            for (int task = tid; task < n * span; task += kThreads) {
                const int a = fastdiv(task, p.mg_span), dx = task - a * span - R;
                const int x = s.pos[2 * a] + dx;
                if (x < 0 || x >= M) continue;
                const int w = s.halfw[dx + R];                      // half width of the disc row: dy^2 <= R^2 - dx^2
                const int y0 = max(0, s.pos[2 * a + 1] - w), y1 = min(M - 1, s.pos[2 * a + 1] + w);
                for (int wd = y0 >> 5; wd <= (y1 >> 5); ++wd) {
                    const int lo = max(y0, wd * 32) - wd * 32, hi = min(y1, wd * 32 + 31) - wd * 32;
                    const uint32_t m = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
                    if (s.ubits[x * W + wd] & m) {
                        const uint32_t old = atomicAnd(&s.ubits[x * W + wd], ~m);
                        const int c = __popc(old & m);
                        if (c) atomicAdd(&s.scal[SC_NEWFOUND], c);
                    }
                }
            }
            __syncthreads();
            const int newf = s.scal[SC_NEWFOUND];
            const int found = cnt[CNT_FIND] + newf;
            const bool term = found >= p.m;                                  // (:270-271)
            __syncthreads();
            if (tid == 0) {
                double fsum = 0.0;
                for (int k = 0; k < kThreads / 32; ++k) fsum += s_red[k];
                const double rew = -1.0 + fsum + 10.0 * (double)newf;       // MOVE_COST + freq + REWARD_FIND (:250-265)
                cnt[CNT_FIND] = found;
                cnt[CNT_TIME] = t1;
                cnt[CNT_FLAGS] |= (term ? SF_DONE : 0) | (s.scal[SC_ILLEGAL] ? SF_ILLEGAL : 0);
                // no per-step statistic: a same-address atomic per CTA per step serialises in L2; env_steps is
                // assembled by cs_search_stats from finished-episode lengths + live time_steps
                if (s.scal[SC_ILLEGAL]) atomicAdd(p.stats + CS_STAT_ILLEGAL, 1.0);
                const double ep_rew = s_ep_reward + rew;                     // fp64, before the fp32 cast of the output
                p.ep_reward[e] = ep_rew;
                if (term) {
                    atomicAdd(p.stats + CS_STAT_EPISODES, 1.0);
                    atomicAdd(p.stats + CS_STAT_EP_REWARD, ep_rew);
                    atomicAdd(p.stats + CS_STAT_TARGETS_FOUND, (double)found);
                    atomicAdd(p.stats + CS_STAT_WINS, 1.0);
                    atomicAdd(p.stats + CS_STAT_EP_LEN, (double)t1);
                }
                p.reward[e] = (float)rew;
                p.terminated[e] = term ? 1 : 0;
                p.target_find[e] = found;
            }
            done = term;
            emit = true;
            bits_dirty = true;
            __syncthreads();
        } else if (tid == 0) {
            p.reward[e] = 0.f;
            p.terminated[e] = 1;
        }
        if (p.auto_reset && done) {
            search_reset(p, s, e, 0u, cnt);
            emit = true;
            bits_dirty = true;
        }
    } else {
        search_reset(p, s, e, rflags, cnt);
        emit = true;
        bits_dirty = true;
        if (tid == 0) {
            p.reward[e] = 0.f;
            p.terminated[e] = 0;
            p.target_find[e] = 0;
        }
    }
    if (!emit) return;
    __syncthreads();
    if (bits_dirty) {
        uint32_t* gt = p.target_bits + (size_t)e * rows;
        uint32_t* gu = p.unfound_bits + (size_t)e * rows;
        for (int k = tid; k < rows; k += kThreads) { gt[k] = s.tbits[k]; gu[k] = s.ubits[k]; }
        int32_t* gp = p.pos + (size_t)e * 2 * n;
        for (int k = tid; k < 2 * n; k += kThreads) gp[k] = s.pos[k];
        if (tid < 4) p.counters[(size_t)e * 4 + tid] = cnt[tid];
    }
    search_emit(p, s, e);
}

// sum of the live time_step counters, for cs_search_stats
__global__ void __launch_bounds__(256) search_live_steps_kernel(const int32_t* __restrict__ counters, int E, double* __restrict__ out) {
    unsigned long long acc = 0;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < E; e += gridDim.x * blockDim.x) {
        const int4 c = reinterpret_cast<const int4*>(counters)[e];
        if (!(c.z & SF_DONE)) acc += (unsigned)c.y;            // a finished episode is already in CS_STAT_EP_LEN
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, (double)acc);
}

}  // namespace

struct cs_search {
    cs_search_cfg cfg;
    SearchParams p;
    size_t smem_bytes;
    int32_t* d_cells;
    uint8_t* d_actions;
    double* d_live;
};

namespace {
cudaError_t launch_search(cs_search* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags,
                          int random_policy, cudaStream_t st) {
    if (mode == MODE_STEP)
        search_kernel<MODE_STEP><<<h->p.E, kThreads, h->smem_bytes, st>>>(h->p, actions, mask, rflags, random_policy);
    else
        search_kernel<MODE_RESET><<<h->p.E, kThreads, h->smem_bytes, st>>>(h->p, actions, mask, rflags, random_policy);
    cs_count_launch(1);
    return cudaGetLastError();
}
}  // namespace

namespace { int search_init(cs_search* h); }

extern "C" {

int cs_search_create(const cs_search_cfg* cfg, cs_search** out) {
    CS_REQUIRE(cfg && out, "cs_search_create: null argument");
    CS_REQUIRE(cfg->struct_size == sizeof(cs_search_cfg), "cs_search_create: cfg.struct_size %u != %zu (ABI mismatch)",
               cfg->struct_size, sizeof(cs_search_cfg));
    CS_REQUIRE(cfg->num_envs > 0, "num_envs must be > 0");
    CS_REQUIRE(cfg->n_agents >= 1 && cfg->n_agents <= 4096, "n_agents out of range");
    CS_REQUIRE(cfg->map_size >= 2 && cfg->map_size <= 1024, "map_size out of range");
    CS_REQUIRE(cfg->view_range >= 1 && cfg->view_range <= 64, "view_range out of range");
    CS_REQUIRE(cfg->target_num >= 1 && cfg->target_num <= cfg->map_size * cfg->map_size, "target_num must fit the grid");
    CS_REQUIRE(cfg->agent_mode >= 0 && cfg->agent_mode <= 2, "Unknown agent mode");          // search_env.py:180
    CS_REQUIRE(cfg->target_mode == 0 || cfg->target_mode == 1, "Unknown target mode");        // :143 (modes 2,3: inject cells)
    CS_REQUIRE(cfg->agent_mode != 2 || cfg->n_agents >= 2, "agent_mode 2 divides by n_agents-1 (search_env.py:171)");
    CS_REQUIRE(cfg->target_mode != 1 || cfg->target_num <= search_band_cells(cfg->map_size),
               "target_mode 1: target_num %d exceeds the %d cells of the edge band (the reference never finishes placing them)",
               cfg->target_num, search_band_cells(cfg->map_size));
    {
        const int L = (int)ceil(sqrt((double)cfg->n_agents));
        CS_REQUIRE(cfg->agent_mode == 2 || L <= cfg->map_size, "agents do not fit the map");
    }
    cs_search* h = new (std::nothrow) cs_search();
    if (!h) { cs_set_error("out of host memory"); return CS_ERR_NOMEM; }
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    const int rc = search_init(h);
    if (rc != CS_OK) {            // free whatever exists: a retry with fewer envs must find the memory back
        cs_search_destroy(h);
        cudaGetLastError();
        return rc;
    }
    *out = h;
    return CS_OK;
}

}  // extern "C"

namespace {
// everything cs_search_create computes and allocates, in one place so that a failure half way frees what exists
int search_init(cs_search* h) {
    const cs_search_cfg* cfg = &h->cfg;
    CS_CUDA(cudaSetDevice(cfg->device));
    SearchParams& p = h->p;
    p.E = cfg->num_envs; p.n = cfg->n_agents; p.m = cfg->target_num; p.M = cfg->map_size; p.R = cfg->view_range;
    p.W = (p.M + 31) / 32; p.S = 2 * p.R - 1; p.obs_len = p.S * p.S + 2;
    p.agent_mode = cfg->agent_mode; p.target_mode = cfg->target_mode; p.auto_reset = cfg->auto_reset;
    p.seed = cfg->seed; p.env_id_base = cfg->env_id_base;
    auto magic = [](int d) { return (uint32_t)((0x100000000ULL + (uint64_t)d - 1) / (uint64_t)d); };
    p.mg_half = magic(p.M / 2 > 0 ? p.M / 2 : 1); p.mg_M = magic(p.M); p.mg_S1 = magic(p.S + 1); p.mg_span = magic(2 * p.R + 1);
    const size_t stage_bytes = ((size_t)p.n * p.obs_len + 15) & ~(size_t)15;      // one byte (2*value) per element
    p.stage_obs = (p.M <= 64 && p.S <= 32 && smem_base_bytes(p) + stage_bytes <= 100 * 1024) ? 1 : 0;
    h->smem_bytes = smem_base_bytes(p) + (p.stage_obs ? stage_bytes : 0);
    CS_REQUIRE(h->smem_bytes <= 200 * 1024, "map too large for the shared-memory bit rows");
    {
        // the limit is per KERNEL, not per handle: only ever raise it (a later, smaller handle must not lower it under
        // an earlier one's launches)
        static size_t cur_limit = 48 * 1024;
        if (h->smem_bytes > cur_limit) {
            CS_CUDA(cudaFuncSetAttribute(search_kernel<MODE_STEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
            CS_CUDA(cudaFuncSetAttribute(search_kernel<MODE_RESET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
            cur_limit = h->smem_bytes;
        }
    }
    {
        // Target placement draws uniform candidates over all M^2 cells and accepts the eligible free ones (all cells; mode 1:
        // the edge band).  A given eligible cell is missed by N candidates with probability (1 - 1/M^2)^N <= e^(-N/M^2);
        // over the Q eligible cells, N = M^2 (ln Q + c) leaves one unvisited with probability <= e^-c (the coupon-collector
        // tail).  Every eligible cell visited means every accepted request (m <= Q) is placed in full; c = 70 puts a
        // shortfall at <= 4e-31 per reset.  Envs stop at the m-th accepted cell (c5, m = 1000 of 4096: ~1150 candidates).
        const double MM = (double)p.M * p.M;
        const double Q = p.target_mode == 1 ? (double)search_band_cells(p.M) : MM;
        p.place_batches = (int)ceil(MM * (log(Q) + 70.0) / kThreads);
    }
    const size_t E = (size_t)p.E, rows = (size_t)p.M * p.W, MM = (size_t)p.M * p.M;
#define CS_ALLOC0(ptr, bytes)                                   \
    CS_CUDA(cudaMalloc(reinterpret_cast<void**>(&(ptr)), (bytes))); \
    CS_CUDA(cudaMemset((ptr), 0, (bytes)))
    CS_ALLOC0(p.pos, E * 2 * p.n * sizeof(int32_t));
    CS_ALLOC0(p.target_bits, E * rows * sizeof(uint32_t));
    CS_ALLOC0(p.unfound_bits, E * rows * sizeof(uint32_t));
    CS_ALLOC0(p.freq, E * MM * sizeof(int32_t));
    CS_ALLOC0(p.counters, E * 4 * sizeof(int32_t));
    CS_ALLOC0(p.obs, E * p.n * p.obs_len * sizeof(float));
    CS_ALLOC0(p.state, E * 2 * MM * sizeof(float));
    CS_ALLOC0(p.avail, E * p.n * 4);
    CS_ALLOC0(p.reward, E * sizeof(float));
    CS_ALLOC0(p.terminated, E);
    CS_ALLOC0(p.target_find, E * sizeof(int32_t));
    CS_ALLOC0(p.stats, CS_NUM_STATS * sizeof(double));
    CS_ALLOC0(h->d_actions, E * p.n);
    CS_ALLOC0(h->d_live, sizeof(double));
    CS_ALLOC0(p.ep_reward, E * sizeof(double));
#undef CS_ALLOC0
    // episode counter starts at -1 so that the first reset opens episode 0
    CS_CUDA(cudaMemset2D(p.counters + CNT_EPISODE, 4 * sizeof(int32_t), 0xFF, sizeof(int32_t), E));
    return CS_OK;
}
}  // namespace

extern "C" {

void cs_search_destroy(cs_search* h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    SearchParams& p = h->p;
    cudaFree(p.pos); cudaFree(p.target_bits); cudaFree(p.unfound_bits); cudaFree(p.freq); cudaFree(p.counters);
    cudaFree(p.obs); cudaFree(p.state); cudaFree(p.avail); cudaFree(p.reward); cudaFree(p.terminated);
    cudaFree(p.target_find); cudaFree(p.stats); cudaFree(p.ep_reward); cudaFree(h->d_cells); cudaFree(h->d_actions); cudaFree(h->d_live);
    delete h;
}

int cs_search_buffers_get(cs_search* h, cs_search_buffers* b) {
    CS_REQUIRE(h && b, "cs_search_buffers_get: null argument");
    const SearchParams& p = h->p;
    b->pos = p.pos; b->target_bits = p.target_bits; b->unfound_bits = p.unfound_bits; b->freq = p.freq;
    b->counters = p.counters; b->words_per_row = p.W; b->obs = p.obs; b->state = p.state; b->avail = p.avail;
    b->reward = p.reward; b->terminated = p.terminated; b->target_find = p.target_find; b->stats = p.stats;
    return CS_OK;
}

int cs_search_env_info(const cs_search* h, int32_t* out4) {
    CS_REQUIRE(h && out4, "cs_search_env_info: null argument");
    out4[0] = 4;                                   // n_actions      (search_env.py:62)
    out4[1] = 2 * h->p.M * h->p.M;                 // state_shape    (:63)
    out4[2] = h->p.obs_len;                        // obs_shape      (:64)
    out4[3] = 500;                                 // episode_limit  (:65)
    return CS_OK;
}

int cs_search_set_targets(cs_search* h, const int32_t* d_cells, void* stream) {
    CS_REQUIRE(h && d_cells, "cs_search_set_targets: null argument");
    CS_CUDA(cudaSetDevice(h->cfg.device));
    const size_t bytes = (size_t)h->p.E * h->p.m * 2 * sizeof(int32_t);
    if (!h->d_cells) CS_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->d_cells), bytes));
    CS_CUDA(cudaMemcpyAsync(h->d_cells, d_cells, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    h->p.cells = h->d_cells;
    return CS_OK;
}

int cs_search_reset(cs_search* h, const uint8_t* d_mask, uint32_t flags, void* stream) {
    CS_REQUIRE(h, "cs_search_reset: null handle");
    CS_REQUIRE(!(flags & CS_RESET_KEEP_TARGETS) || h->p.cells, "CS_RESET_KEEP_TARGETS needs cs_search_set_targets first");
    CS_CUDA(launch_search(h, MODE_RESET, nullptr, d_mask, flags, 0, (cudaStream_t)stream));
    return CS_OK;
}

int cs_search_step(cs_search* h, const uint8_t* d_actions, void* stream) {
    CS_REQUIRE(h && d_actions, "cs_search_step: null argument");
    CS_CUDA(launch_search(h, MODE_STEP, d_actions, nullptr, 0u, 0, (cudaStream_t)stream));
    return CS_OK;
}

int cs_search_step_random(cs_search* h, int32_t k, void* stream) {
    CS_REQUIRE(h && k >= 0, "cs_search_step_random: bad argument");
    for (int i = 0; i < k; ++i) CS_CUDA(launch_search(h, MODE_STEP, nullptr, nullptr, 0u, 1, (cudaStream_t)stream));
    return CS_OK;
}

int cs_search_step_host(cs_search* h, const cs_search_host_io* io, void* stream) {
    CS_REQUIRE(h && io && io->actions, "cs_search_step_host: null argument");
    const SearchParams& p = h->p;
    const size_t E = (size_t)p.E;
    cudaStream_t st = (cudaStream_t)stream;
    CS_CUDA(cudaSetDevice(h->cfg.device));
    CS_CUDA(cudaMemcpyAsync(h->d_actions, io->actions, E * p.n, cudaMemcpyHostToDevice, st));
    CS_CUDA(launch_search(h, MODE_STEP, h->d_actions, nullptr, 0u, 0, st));
    if (io->reward) CS_CUDA(cudaMemcpyAsync(io->reward, p.reward, E * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (io->terminated) CS_CUDA(cudaMemcpyAsync(io->terminated, p.terminated, E, cudaMemcpyDeviceToHost, st));
    if (io->obs) CS_CUDA(cudaMemcpyAsync(io->obs, p.obs, E * p.n * p.obs_len * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (io->state) CS_CUDA(cudaMemcpyAsync(io->state, p.state, E * 2 * p.M * p.M * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (io->avail) CS_CUDA(cudaMemcpyAsync(io->avail, p.avail, E * p.n * 4, cudaMemcpyDeviceToHost, st));
    CS_CUDA(cudaStreamSynchronize(st));
    return CS_OK;
}

int cs_search_stats(cs_search* h, double* h_out, void* stream) {
    CS_REQUIRE(h && h_out, "cs_search_stats: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    CS_CUDA(cudaSetDevice(h->cfg.device));
    CS_CUDA(cudaMemsetAsync(h->d_live, 0, sizeof(double), st));
    const int grid = (h->p.E + 255) / 256 < CS_NUM_SMS_B200 * 4 ? (h->p.E + 255) / 256 : CS_NUM_SMS_B200 * 4;
    search_live_steps_kernel<<<grid, 256, 0, st>>>(h->p.counters, h->p.E, h->d_live);
    cs_count_launch(1);
    CS_CUDA(cudaGetLastError());
    double live = 0.0;
    CS_CUDA(cudaMemcpyAsync(h_out, h->p.stats, CS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, st));
    CS_CUDA(cudaMemcpyAsync(&live, h->d_live, sizeof(double), cudaMemcpyDeviceToHost, st));
    CS_CUDA(cudaStreamSynchronize(st));
    h_out[CS_STAT_ENV_STEPS] = h_out[CS_STAT_EP_LEN] + live;      // finished episodes + episodes still running
    return CS_OK;
}

}  // extern "C"
