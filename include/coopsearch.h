/*
 * coopsearch.h -- C ABI of libcoopsearch.so (B200 / sm_100a batched env-step hot path).
 *
 * The reference (WZN1ng/Cooperative-Search) is pure Python and has no FFI; its "plugin
 * interface" for this path is the duck-typed SMAC-style env protocol that
 * common/rollout.py:24-201 and main.py:114,134 call.  Every entry point below names the
 * reference method it replaces.  Python binds these with ctypes
 * (cooperative-search_b200/_lib.py); INTEGRATION.md shows the stub a reference
 * maintainer would add.
 *
 * Conventions
 *   - plain C types only; every function returns CS_OK (0) or a negative cs_status;
 *     cs_last_error() gives a thread-local message.  Nothing throws across the ABI.
 *   - a handle owns its device memory (state + output buffers).  cs_*_buffers() exposes
 *     the device pointers so the host language can wrap them zero-copy.
 *   - all calls taking a `stream` (a cudaStream_t passed as void*) are asynchronous on
 *     that stream and never synchronise; *_host calls take HOST pointers, do their own
 *     H2D/D2H copies on the given stream and return after the results are in host memory.
 *   - a handle is not thread-safe; use one handle per host thread / stream.
 *   - global env ids are env_id_base + local index; every random draw is keyed by the
 *     GLOBAL id, so results do not depend on how envs are sharded over GPUs.
 */
#ifndef COOPSEARCH_H_
#define COOPSEARCH_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CS_ABI_VERSION 2
#define CS_MAX_AGENTS 32   /* flight envs: out-of-map flags live in one 32-bit word   */
#define CS_MAX_TARGETS 32  /* flight envs: found flags live in one 32-bit word        */
#define CS_NUM_STATS 8

typedef enum cs_status {
    CS_OK = 0,
    CS_ERR_INVALID = -1,      /* bad argument / config (reference: raise Exception(...))   */
    CS_ERR_CUDA = -2,         /* a CUDA runtime call failed                                */
    CS_ERR_NOMEM = -3,
    CS_ERR_UNSUPPORTED = -4
} cs_status;

/* cs_*_reset flags */
#define CS_RESET_INIT 1u          /* reset(init=True): flight variant refills prob_map=0.5
                                     (env/flight_env.py:84-86)                              */
#define CS_RESET_KEEP_TARGETS 2u  /* keep the target coordinates/cells currently in the
                                     state buffers (parity tests inject the reference's)   */
#define CS_RESET_KEEP_EPISODE 4u  /* do not advance the per-env episode counter            */

/* meta words of a flight env (uint32 each), see cs_flight_buffers.dyn */
enum { CS_META_FOUND = 0, CS_META_NEWFOUND = 1, CS_META_OUT = 2, CS_META_TIME = 3,
       CS_META_EPISODE = 4, CS_META_FLAGS = 5, CS_META_EPREWARD = 6, CS_META_SENSE = 7,  /* flight variant: non-zero iff the latest step/reset call sensed the env (bit 0: its first job is parked in the side buffer) */
       CS_META_WORDS = 8 };
#define CS_FLAG_WIN 1u
#define CS_FLAG_DONE 2u

/* indices into the stats vector (doubles); the vector all-reduced over NCCL (SURVEY 8e) */
enum { CS_STAT_EPISODES = 0, CS_STAT_EP_REWARD = 1, CS_STAT_TARGETS_FOUND = 2, CS_STAT_WINS = 3,
       CS_STAT_EP_LEN = 4, CS_STAT_ENV_STEPS = 5, CS_STAT_ILLEGAL = 6, CS_STAT_TOUCHED = 7 };

int cs_version(void);
const char* cs_last_error(void);
/* number of kernels this library has launched in the calling process (bench "gpu_launches") */
uint64_t cs_launch_count(void);

/* lanes per env the handle's step kernel was instantiated with (tuning visibility) */
struct cs_flight;
int cs_flight_lanes_per_env(const struct cs_flight* env);
/* test hook: d_in6 [count][6] = Philox counter(4) + key(2) -> d_out4 [count][4] words */
int cs_debug_philox(const uint32_t* d_in6, uint32_t* d_out4, int32_t count, void* stream);

/* test hook, host only: evaluates the heading trig table (csrc/flight.cu: heading_sincos) a handle with this
 * time_limit would use; returns the number of table entries.  from_table[i] = 0 where the fallback is used. */
int cs_debug_heading_lut(int32_t time_limit, const double* h_in, int32_t count, double* sin_out, double* cos_out,
                         int32_t* from_table);

/* measurement hook: how cs_flight_obs_full writes the observation rows (0 = TMA bulk stores, default; 1 = plain stores) */
int cs_debug_flight_obs_path(struct cs_flight* env, int32_t path);

/* Row gather / scatter on the device: dst row d_dst_idx[i] <- src row d_src_idx[i] for i < count (a NULL index array =
 * identity), rows of row_bytes bytes.  The data movement of the device replay ring (common/replay_buffer.py:36-79:
 * store_episode, sample, sample_latest). */
int cs_rows_copy(void* d_dst, const void* d_src, uint64_t row_bytes, const int64_t* d_dst_idx, const int64_t* d_src_idx, int64_t count,
                 void* stream);
/* Pinned host memory for the *_host entry points. */
int cs_host_alloc(void** out, uint64_t bytes);
int cs_host_free(void* p);

/* ===================================================================================
 * flight_easy / flight  (env/flight_env_easy.py, env/flight_env.py)
 * =================================================================================== */
typedef struct cs_flight_cfg {
    uint32_t struct_size;   /* sizeof(cs_flight_cfg), ABI check                            */
    int32_t num_envs;       /* E: env instances owned by this handle (this GPU's shard)    */
    int32_t n_agents;       /* args.n_agents      (flight_env_easy.py:22)                  */
    int32_t target_num;     /* args.target_num    (:19)                                    */
    int32_t map_size;       /* args.map_size      (:18)                                    */
    int32_t view_range;     /* args.view_range    (:23)                                    */
    int32_t time_limit;     /* args.time_limit    (:25), <= 65535                          */
    int32_t agent_mode;     /* 0..3               (:139-180)                               */
    int32_t target_mode;    /* 0 file template, 1 uniform (:95-136)                        */
    int32_t variant;        /* 0 = flight_easy (wall test '>'), 1 = flight (prob map, '>=')*/
    int32_t auto_reset;     /* 1: a terminated env is reset inside the same step call      */
    int32_t count_touched;  /* 1: accumulate #prob-map cells updated into CS_STAT_TOUCHED  */
    int32_t lanes_per_env;  /* 0 = automatic; 1 or 4 (n_agents <= 8): thread-per-env step kernel with
                               that many threads per env (flight variant: + the tiled belief-map
                               kernel); flight variant, 8: step + belief map fused in one kernel;
                               otherwise 2, 8, 16, 32: lane-per-agent kernel (flight variant: +
                               generic map kernel)                                                 */
    int32_t device;         /* CUDA device ordinal                                         */
    double velocity;        /* args.agent_velocity                                         */
    double detect_prob;     /* args.detect_prob                                            */
    double safe_dist;       /* args.safe_dist                                              */
    double force_dist;      /* args.force_dist                                             */
    uint32_t seed;          /* Philox key word 0                                           */
    uint32_t env_id_base;   /* global id of local env 0                                    */
    int32_t map_overlap;    /* flight variant: 1 = the belief-map kernel of a step / reset call runs on
                               the handle's OWN stream, concurrently with the next call's step kernel
                               (the step does not read the map).  Every entry point that reads or writes
                               the map joins that stream first; a caller that touches prob_map directly,
                               or captures calls into a CUDA graph, calls cs_flight_map_sync (before the
                               capture begins and before it ends).  0 = everything on the caller's stream */
    int32_t reserved0;
} cs_flight_cfg;

typedef struct cs_flight cs_flight;

/* Device pointers of a flight handle.  fp64 internal state, fp32/u8 outputs.  The state layout is chosen per handle
 * (structure of arrays from 32768 envs, one record per env below) and described by strides, in doubles:
 *   dyn : element (row r, env e) at dyn[r*dyn_row_stride + e*dyn_env_stride]; rows 0..2n-1 = x0,y0,..,x(n-1),y(n-1),
 *         rows yaw_off..yaw_off+n-1 = headings, rows meta_off..meta_off+3 = the CS_META_WORDS uint32 meta words
 *         (two per row: word w of env e is the (w & 1)-th uint32 of element (meta_off + w/2, e))
 *   tgt : element (row r, env e) at tgt[r*tgt_row_stride + e*tgt_env_stride]; row 2j = x of target j, row 2j+1 = y
 *         (target_pos, flight_env_easy.py:113)                                                                    */
typedef struct cs_flight_buffers {
    int64_t dyn_row_stride, dyn_env_stride, tgt_row_stride, tgt_env_stride;
    double* dyn;
    int32_t dyn_doubles;
    int32_t yaw_off;        /* = 2n   (first heading row)                                  */
    int32_t meta_off;       /* first of the four meta rows                                 */
    int32_t state_len;      /* 4n + 3m                                                     */
    int32_t state_stride;   /* floats between consecutive state rows (state_len rounded up
                               to a multiple of 4 so rows start 16-byte aligned)           */
    double* tgt;
    float* obs;             /* [E][n][4]     get_obs   (flight_env_easy.py:218-221)        */
    float* state;           /* [E][state_stride], first 4n+3m of a row = get_state (:190-216) */
    float* reward;          /* [E]           step()[0] (:314)                              */
    uint8_t* terminated;    /* [E]           step()[1]                                     */
    uint8_t* win;           /* [E]           step()[2] (win_flag)                          */
    int32_t* target_find;   /* [E]           attribute target_find (rollout.py:79)         */
    float* prob_map;        /* variant 1 else NULL.  TILED: 4x4-cell tiles of 64 bytes, cell prob_map[i][j]
                               (i<->x) of env e at prob_map[e*map_env_stride + ((i>>2)*map_tiles + (j>>2))*16
                               + (i&3)*4 + (j&3)]; cs_flight_map_export / _import convert from / to the
                               reference's row-major [E][M][M]                              */
    double* stats;          /* [CS_NUM_STATS] running sums over finished episodes          */
    int32_t map_tiles;      /* tiles per map side = ceil(M/4)                              */
    int32_t map_env_stride; /* floats per env in prob_map = map_tiles^2 * 16               */
    void* slab;             /* the one allocation behind reward..state, obs (checkpointing) */
    uint64_t slab_bytes;
} cs_flight_buffers;

/* FlightSearchEnvEasy.__init__ / FlightSearchEnv.__init__ (flight_env_easy.py:15-69).
 * Allocates state; envs are NOT reset until cs_flight_reset is called. */
int cs_flight_create(const cs_flight_cfg* cfg, cs_flight** out);
void cs_flight_destroy(cs_flight* env);
int cs_flight_buffers_get(cs_flight* env, cs_flight_buffers* out);
/* get_env_info (flight_env_easy.py:71-77): out4 = n_actions, state_shape, obs_shape, episode_limit */
int cs_flight_env_info(const cs_flight* env, int32_t* out4);
/* circle_dict of main.py:19-32 for target_mode 0: host array [m][5] doubles
 * (x, y, dx, dy, deter=='f' ? 1 : 0) in FILE units (the a = map_size/10 scale is applied inside,
 * flight_env_easy.py:97-103). */
int cs_flight_set_target_template(cs_flight* env, const double* host_rows, int32_t rows);
/* reset(init) (flight_env_easy.py:79-182) for envs with mask[e] != 0 (device u8 [E]; NULL = all). */
int cs_flight_reset(cs_flight* env, const uint8_t* d_mask, uint32_t flags, void* stream);
/* step(act_list) (flight_env_easy.py:303-314).  d_actions: device u8 [E][n], values 0..2.
 * Envs whose DONE flag is set are a masked no-op (reward 0, terminated 1) unless auto_reset. */
int cs_flight_step(cs_flight* env, const uint8_t* d_actions, void* stream);
/* Grouped device step: several flight_easy handles of the same shape (independent env batches = rollout workers,
 * n_agents <= 8, same n_agents / lanes_per_env / device) advance one step in ONE kernel launch.  d_actions: host
 * array of `count` device pointers, u8 [E_i][n] each.  Results land in every handle's own buffers, exactly as
 * `count` cs_flight_step calls would leave them.  At most 128 handles per group; the handles must outlive the group
 * (it keeps their device pointers), and like a handle a group is used from one host thread / stream at a time. */
typedef struct cs_flight_group cs_flight_group;
int cs_flight_group_create(cs_flight* const* envs, int32_t count, cs_flight_group** out);
int cs_flight_group_step(cs_flight_group* group, const uint8_t* const* d_actions, void* stream);
void cs_flight_group_destroy(cs_flight_group* group);
/* k steps under the uniform-random policy drawn in-kernel (alg=random, agent/agent.py:34-36). */
int cs_flight_step_random(cs_flight* env, int32_t k, void* stream);
/* Reference-shaped observation of the flight variant (flight_env.py:223-230):
 * d_out [E][n][M*M+4] = prob_map.ravel() || (x^,y^,cos,sin). */
int cs_flight_obs_full(cs_flight* env, float* d_out, void* stream);
/* self.prob_map as the reference holds it (flight_env.py:53): d_out / d_in = device [E][M][M] row-major floats,
 * converted from / into the handle's tiled map. */
int cs_flight_map_export(cs_flight* env, float* d_out, void* stream);
int cs_flight_map_import(cs_flight* env, const float* d_in, void* stream);
/* Makes `stream` wait for the latest belief-map kernel of the handle (no-op unless map_overlap). */
int cs_flight_map_sync(cs_flight* env, void* stream);
/* Host-buffer step: the call a CPU-side rollout makes.  h_actions [E][n] u8.  Any output pointer
 * may be NULL (not copied).  Blocks until outputs are in host memory. */
#define CS_HOST_NO_SYNC 1u        /* cs_*_host_io.flags: enqueue only; the caller synchronises the stream */
typedef struct cs_flight_host_io {
    const uint8_t* actions;
    float* reward;
    uint8_t* terminated;
    uint8_t* win;
    float* obs;
    float* state;           /* compact [E][4n+3m] */
    void* slab;             /* if non-NULL: ONE D2H copy of reward|target_find|terminated|win|state in
                               the layout of cs_flight_slab_layout; the pointers above are ignored */
    uint32_t flags;         /* CS_HOST_NO_SYNC */
} cs_flight_host_io;
int cs_flight_step_host(cs_flight* env, const cs_flight_host_io* io, void* stream);
/* cs_flight_step_host for `count` independent env batches (rollout workers) in one call: batch i is enqueued on
 * streams[i % n_streams]; all streams are synchronised once at the end unless every io carries CS_HOST_NO_SYNC. */
int cs_flight_step_host_many(cs_flight* const* envs, const cs_flight_host_io* ios, int32_t count, void* const* streams,
                             int32_t n_streams);
/* Compact host-buffer step (the fast form of cs_flight_step_host).  Per step and env the device sends 16 + 16n bytes:
 * a 16-byte record (reward, found mask, target_find, terminated, win, reset flag; one flat D2H copy, plus one small entry
 * per env that was reset inside the call) and the n agent rows, which the copy engine writes IN PLACE into the agent
 * part of the library's reference-shaped host rows (= get_obs, flight_env_easy.py:192-193,218-221) with one strided D2H
 * copy.  A few host threads (CS_HOST_THREADS) spread the records over the result arrays, flip the find flags whose bit
 * changed and rewrite target coordinates after a reset.  `state` is pinned host memory.
 * The views stay valid (and are updated in place) until the handle is destroyed. */
typedef struct cs_flight_host_views {
    float* reward;          /* [E]                   step()[0]                                        */
    int32_t* target_find;   /* [E]                                                                    */
    uint8_t* terminated;    /* [E]                   step()[1]                                        */
    uint8_t* win;           /* [E]                   step()[2]                                        */
    float* state;           /* [E][state_stride]     get_state(); get_obs() = floats 0..4n-1 of a row */
    int32_t state_stride;   /* floats between rows                                                    */
    uint64_t h2d_bytes_per_step, d2h_bytes_per_step;
} cs_flight_host_views;
int cs_flight_host_compact_begin(cs_flight* env, cs_flight_host_views* out);
/* h_actions: HOST u8 [E][n] (pinned for full speed).  flags: CS_HOST_NO_SYNC = enqueue only (H2D, step, pack, D2H) --
 * the caller then calls cs_flight_host_expand, with sync = 1 to wait for `stream` first. */
int cs_flight_step_host_compact(cs_flight* env, const uint8_t* h_actions, uint32_t flags, void* stream);
int cs_flight_host_expand(cs_flight* env, void* stream, int32_t sync);
/* many independent env batches in one call: batch i on streams[i % n_streams]; unless CS_HOST_NO_SYNC, batch by batch
 * the stream is synchronised and the rows rebuilt (host work of batch i overlaps the transfers of batch i+1) */
int cs_flight_step_host_compact_many(cs_flight* const* envs, const uint8_t* const* h_actions, int32_t count, void* const* streams,
                                     int32_t n_streams, uint32_t flags);
int cs_flight_host_expand_many(cs_flight* const* envs, int32_t count, void* const* streams, int32_t n_streams, int32_t sync);
/* Pooled form of the compact host-buffer step for many env batches (rollout workers) of one GPU: the batches' host rows,
 * records, agent rows and actions are segments of single allocations, so that ONE call steps every batch with one H2D copy
 * of all actions, one grouped step launch (cs_flight_group_step; per-batch launches when the handles do not group), one
 * pack launch and two D2H copies -- a flat copy of the dense result arrays (reward, target_find, terminated, win, found
 * masks: 14 bytes per env; the host views of the first four ARE that pinned block) and the strided copy that writes all
 * agent rows in place.  Host work per step: the find flags whose bit changed and the rows of envs that were reset.  Batches must agree in n_agents, target_num, auto_reset and device and must not have compact host buffers yet;
 * afterwards cs_flight_host_compact_begin(env) returns the env's segment of the pooled arrays.  Destroy the pool before
 * its envs. */
typedef struct cs_flight_host_pool cs_flight_host_pool;
int cs_flight_host_pool_create(cs_flight* const* envs, int32_t count, cs_flight_host_pool** out);
void cs_flight_host_pool_destroy(cs_flight_host_pool* pool);
/* batch i's views (as cs_flight_host_compact_begin) and its segment of the pool's pinned action buffer [E_i][n] */
int cs_flight_host_pool_views(cs_flight_host_pool* pool, int32_t i, cs_flight_host_views* out, uint8_t** h_actions);
/* h_actions: HOST u8 [sum of num_envs][n], batch after batch (pinned for full speed), or NULL = the pool's own buffer.
 * flags: CS_HOST_NO_SYNC = enqueue only; then cs_flight_host_pool_expand (sync = 1 waits for `stream` first). */
int cs_flight_host_pool_step(cs_flight_host_pool* pool, const uint8_t* h_actions, uint32_t flags, void* stream);
int cs_flight_host_pool_expand(cs_flight_host_pool* pool, void* stream, int32_t sync);
/* out8 = { slab bytes, offsets of reward, target_find, terminated, win, obs (unused: = slab bytes), state, state row
 * pitch in bytes }.  The slab does not carry obs separately: obs[e][a][0..3] = state row e, floats 4a..4a+3. */
int cs_flight_slab_layout(const cs_flight* env, uint64_t* out8);
/* Copies the stats vector to host (synchronises the stream). */
int cs_flight_stats(cs_flight* env, double* h_out, void* stream);

/* Episode-batch writer: the padded episode arrays RolloutWorker.generate_episode builds (common/rollout.py:43-132),
 * for every env of the handle, in caller-owned DEVICE memory.  T = episode_limit; A = n_actions = 3.
 * Usage: reset -> cs_flight_record_begin -> for t in 0..T-1: cs_flight_step(actions_t); cs_flight_record(t, actions_t)
 * on a handle WITHOUT auto_reset (a finished env is a masked no-op and keeps its padding rows). */
typedef struct cs_episode_buffers {
    float* o;               /* [E][T][n][4]       obs before the step              (rollout.py:45,66)   */
    float* s;               /* [E][T][4n+3m]      state before the step            (:46,67)             */
    uint8_t* u;             /* [E][T][n][1]       actions                          (:68)                */
    float* r;               /* [E][T][1]          reward                           (:71)                */
    uint8_t* avail_u;       /* [E][T][n][A]                                        (:70)                */
    float* o_next;          /* [E][T][n][4]       obs after the step               (:82-86)             */
    float* s_next;          /* [E][T][4n+3m]                                                            */
    uint8_t* avail_u_next;  /* [E][T][n][A]                                        (:90-97)             */
    uint8_t* u_onehot;      /* [E][T][n][A]                                        (:57-58,69)          */
    uint8_t* padded;        /* [E][T][1]          1 past the end of the episode    (:73,115)            */
    uint8_t* terminated;    /* [E][T][1]          env flag; 1 in the padding       (:72,116)            */
    float* episode_reward;  /* [E]                                                 (:74)                */
    uint8_t* win_tag;       /* [E]                terminated and win               (:64)                */
    int32_t* targets_find;  /* [E]                                                 (:79)                */
    int32_t* length;        /* [E]                steps taken                                            */
} cs_episode_buffers;
int cs_flight_record_begin(cs_flight* env, const cs_episode_buffers* bufs, int32_t T, void* stream);
int cs_flight_record(cs_flight* env, const cs_episode_buffers* bufs, int32_t t, int32_t T, const uint8_t* d_actions, void* stream);

/* ===================================================================================
 * search_env  (env/search_env.py)
 * =================================================================================== */
typedef struct cs_search_cfg {
    uint32_t struct_size;
    int32_t num_envs;
    int32_t n_agents;       /* search_env.py:25 */
    int32_t target_num;     /* :21 */
    int32_t map_size;       /* :20 */
    int32_t view_range;     /* :26 */
    int32_t agent_mode;     /* 0 centre square, 1 bottom-left, 2 bottom row (:146-180) */
    int32_t target_mode;    /* 0 uniform cells, 1 edge band (:86-104) */
    int32_t auto_reset;
    int32_t device;
    uint32_t seed;
    uint32_t env_id_base;
} cs_search_cfg;

typedef struct cs_search cs_search;

typedef struct cs_search_buffers {
    int32_t* pos;           /* [E][n][2]  agent_pos                                        */
    uint32_t* target_bits;  /* [E][M][W]  bit y of row x: target_map[x][y] (sticky)        */
    uint32_t* unfound_bits; /* [E][M][W]  targets not yet found                            */
    int32_t* freq;          /* [E][M][M]  freq_map, never cleared (search_env.py:39)       */
    int32_t* counters;      /* [E][4]     target_find, time_step, flags(done|illegal), episode */
    int32_t words_per_row;  /* W = ceil(M/32)                                              */
    float* obs;             /* [E][n][(2R-1)^2+2]  get_obs   (:203-227)                    */
    float* state;           /* [E][M][M][2]        get_state (:186-200)                    */
    uint8_t* avail;         /* [E][n][4]           get_avail_agent_actions (:230-243)      */
    float* reward;          /* [E] */
    uint8_t* terminated;    /* [E] */
    int32_t* target_find;   /* [E] */
    double* stats;          /* [CS_NUM_STATS] */
} cs_search_buffers;

int cs_search_create(const cs_search_cfg* cfg, cs_search** out);
void cs_search_destroy(cs_search* env);
int cs_search_buffers_get(cs_search* env, cs_search_buffers* out);
/* get_env_info (search_env.py:60-66): n_actions, state_shape, obs_shape, episode_limit */
int cs_search_env_info(const cs_search* env, int32_t* out4);
/* Inject target cells for CS_RESET_KEEP_TARGETS: d_cells device int32 [E][m][2]. */
int cs_search_set_targets(cs_search* env, const int32_t* d_cells, void* stream);
/* reset (search_env.py:69-183); init=False semantics, freq_map is never cleared. */
int cs_search_reset(cs_search* env, const uint8_t* d_mask, uint32_t flags, void* stream);
/* step(act_list) (search_env.py:246-296); d_actions u8 [E][n] in 0..3.  An illegal move
 * (reference raises, :293) sets the env's illegal flag and leaves that agent in place. */
int cs_search_step(cs_search* env, const uint8_t* d_actions, void* stream);
int cs_search_step_random(cs_search* env, int32_t k, void* stream);
typedef struct cs_search_host_io {
    const uint8_t* actions;
    float* reward;
    uint8_t* terminated;
    float* obs;
    float* state;
    uint8_t* avail;
} cs_search_host_io;
int cs_search_step_host(cs_search* env, const cs_search_host_io* io, void* stream);
int cs_search_stats(cs_search* env, double* h_out, void* stream);

/* ===================================================================================
 * simple_spread  (env/simple_spread.py; SURVEY 8f "next" row 4)
 * =================================================================================== */
typedef struct cs_spread_cfg {
    uint32_t struct_size;
    int32_t num_envs;
    int32_t n_agents;       /* simple_spread.py:23 */
    int32_t target_num;     /* :21 */
    int32_t map_size;       /* :20 */
    int32_t time_limit;     /* :25 -- the reference hard-codes 100 */
    int32_t auto_reset;     /* 1: an env that terminates is reset inside the same call (the step still reports it) */
    int32_t device;
    uint32_t seed, env_id_base;   /* reset placement is keyed by (seed, global env id, episode): shard invariant */
} cs_spread_cfg;
typedef struct cs_spread cs_spread;
typedef struct cs_spread_buffers {
    double* pos;            /* [E][n + m][2]  agents, then targets (float64 like the reference's Python floats)    */
    int32_t* meta;          /* [E][4]         time_step, episode, done, 0                                          */
    float* obs;             /* [E][n][obs_dim]   get_obs()   (:78-101,112-114), obs_dim = 2 + 2(n-1) + 4m          */
    float* state;           /* [E][state_dim]    get_state() (:116-128), state_dim = 2n + 2m                       */
    float* reward;          /* [E]            step()[0] (:141-167)                                                 */
    double* reward64;       /* [E]            the same in float64                                                  */
    uint8_t* terminated;    /* [E]            step()[1] (:176-178)                                                 */
    uint8_t* occupied;      /* [E][m]         (:96-110)                                                            */
    double* stats;          /* [CS_NUM_STATS] episodes, reward sum, episode length sum                             */
    double* episode_reward; /* [E]            total_reward of the running episode (:175)                           */
    int32_t obs_dim, state_dim;
} cs_spread_buffers;
int cs_spread_create(const cs_spread_cfg* cfg, cs_spread** out);                  /* SimpleSpreadEnv.__init__ (:16-39) */
void cs_spread_destroy(cs_spread* env);
int cs_spread_env_info(const cs_spread* env, int32_t* out4);                      /* get_env_info (:41-46) */
int cs_spread_buffers_get(cs_spread* env, cs_spread_buffers* out);
/* reset (:48-70) of the envs with d_mask[e] != 0 (NULL = all).  CS_RESET_KEEP_TARGETS keeps every coordinate currently in
 * `pos` (a layout the caller injected), CS_RESET_KEEP_EPISODE does not advance the episode counter. */
int cs_spread_reset(cs_spread* env, const uint8_t* d_mask, uint32_t flags, void* stream);
int cs_spread_step(cs_spread* env, const uint8_t* d_actions, void* stream);       /* step (:169-180); actions u8 [E][n] in 0..4 */
int cs_spread_step_random(cs_spread* env, int32_t k, void* stream);               /* k steps, actions drawn in the kernel */
/* HOST buffers: H2D of the actions, the step, D2H of whatever is non-NULL; synchronises the stream */
int cs_spread_step_host(cs_spread* env, const uint8_t* h_actions, float* h_reward, uint8_t* h_terminated, float* h_obs, float* h_state, void* stream);
int cs_spread_stats(cs_spread* env, double* h_out, void* stream);

/* ===================================================================================
 * batched agent network + action selection  (network/base_net.py, agent/agent.py; SURVEY 8f "next" row 1)
 * =================================================================================== */
typedef struct cs_policy_cfg {
    uint32_t struct_size;
    int32_t device;
    int32_t n_agents;       /* args.n_agents                                                   */
    int32_t obs_dim;        /* args.obs_shape (4 for flight_easy)                              */
    int32_t n_actions;      /* args.n_actions                                                  */
    int32_t hidden_dim;     /* args.rnn_hidden_dim, must be 64                                 */
    int32_t last_action;    /* args.last_action: append the last action one-hot (agent.py:44-45) */
    int32_t reuse_network;  /* args.reuse_network: append the agent id one-hot (agent.py:46-47)  */
    int32_t conv_out_dim;   /* args.conv_out_dim where args.conv (the `flight` agents, network/base_net.py:10-20),
                               else 0: that many conv features of the env's map lead the fc1 input   */
} cs_policy_cfg;
/* HOST pointers in torch's own layouts (RNN.state_dict(), network/base_net.py:22-28): Linear.weight is (out, in),
 * GRUCell.weight_ih / weight_hh are (3*hidden, hidden) with gate order r | z | n. */
typedef struct cs_policy_weights {
    const float *fc1_w, *fc1_b;        /* (64, in), (64)        fc1                         */
    const float *w_ih, *w_hh;          /* (192, 64) each        rnn.weight_ih / weight_hh   */
    const float *b_ih, *b_hh;          /* (192) each                                        */
    const float *fc2a_w, *fc2a_b;      /* (64, 64), (64)        fc2.0                       */
    const float *fc2b_w, *fc2b_b;      /* (n_actions, 64), (n_actions)   fc2.2              */
} cs_policy_weights;
typedef struct cs_policy_io {          /* DEVICE pointers; row r = env r / n_agents, agent r % n_agents */
    int32_t rows;
    int32_t evaluate;                  /* 1: greedy (agent.py:71 `evaluate or ...`)                       */
    float epsilon;                     /* probability of a uniform available action when !evaluate        */
    uint32_t seed, t;                  /* Philox key / counter of the epsilon draws (row, t)              */
    const float* obs;                  /* [rows][obs_dim]    = get_obs()                                  */
    const uint8_t* last_action;        /* [rows] or NULL; 255 = no action yet (rollout.py:31 zeros)       */
    const uint8_t* avail;              /* [rows][n_actions] or NULL (= all available)                     */
    float* hidden;                     /* [rows][64] in/out  (policy.eval_hidden, init_hidden = zeros)    */
    float* q;                          /* [rows][n_actions] out or NULL                                   */
    uint8_t* actions;                  /* [rows] out; may be the same buffer as last_action               */
    int32_t precision;                 /* 0 = fp32 on CUDA cores; 1 = bf16 operands on the tcgen05 tensor cores,
                                          fp32 accumulation and hidden state (both: input width <= 256)   */
    int32_t mode;                      /* 0 = masked argmax / epsilon-greedy (agent.py:66-75);
                                          1 = softmax sampling of alg=reinforce (agent.py:77-97)            */
    const float* feat;                 /* [rows / n_agents][conv_out_dim] from cs_policy_conv_features, or NULL  */
} cs_policy_io;
typedef struct cs_policy cs_policy;
/* RNN(input_shape, args) + load_state_dict (policy/qmix.py:40-59).  The fc1 input width (conv_out_dim + obs_dim
 * [+ n_actions] [+ n_agents]) may be up to 256; larger widths return CS_ERR_INVALID. */
int cs_policy_create(const cs_policy_cfg* cfg, const cs_policy_weights* host_weights, cs_policy** out);
void cs_policy_destroy(cs_policy* policy);
/* Agents.choose_action for every (env, agent) row at once (agent/agent.py:33-97, alg != random) */
int cs_policy_act(cs_policy* policy, const cs_policy_io* io, void* stream);
/* Conv front end of the `flight` agents (network/base_net.py:10-20,31-41; args of common/arguments.py:246-265):
 * Conv2d(1, dim_1, kernel_size_1, stride_1) -> ReLU -> Conv2d(dim_1, dim_2, kernel_size_2, stride_2, padding_2) -> ReLU ->
 * Linear(dim_2 * conv_size^2, out_dim).  HOST weight pointers in torch's layouts: Conv2d.weight (out, in, kh, kw),
 * Linear.weight (out, in). */
typedef struct cs_policy_conv_cfg {
    uint32_t struct_size;
    int32_t map_size, dim_1, kernel_size_1, stride_1, dim_2, kernel_size_2, stride_2, padding_2, out_dim;
} cs_policy_conv_cfg;
typedef struct cs_policy_conv_weights {
    const float *c1_w, *c1_b;          /* conv.0 */
    const float *c2_w, *c2_b;          /* conv.2 */
    const float *lin_w, *lin_b;        /* linear */
} cs_policy_conv_weights;
int cs_policy_set_conv(cs_policy* policy, const cs_policy_conv_cfg* cfg, const cs_policy_conv_weights* host_weights);
/* The conv features of every env's belief map, read ONCE per env from the flight handle's TILED device map
 * (cs_flight_buffers.prob_map / map_tiles / map_env_stride) -- the reference replicates the map into every agent's
 * observation row (flight_env.py:223-230) and convolves it once per agent.  d_feat: device [num_envs][out_dim]. */
int cs_policy_conv_features(cs_policy* policy, const float* d_map_tiled, int32_t map_tiles, int32_t map_env_stride, int32_t num_envs,
                            float* d_feat, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* COOPSEARCH_H_ */
