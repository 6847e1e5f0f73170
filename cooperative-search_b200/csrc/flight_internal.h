// Host-side internals shared by the flight_*.cu translation units (not part of the C ABI).
#pragma once
#include <cuda.h>
#include "flight_common.cuh"

constexpr int kTpeMaxAgents = 8;       // thread-per-env kernels are instantiated for n_agents 1..8
#ifndef CS_TPE_THREADS
#define CS_TPE_THREADS 64
#endif
constexpr int kTpeThreads = CS_TPE_THREADS;   // threads per CTA of the thread-per-env kernels
constexpr int kMaxGroup = 128;         // handles per grouped launch

// Compact host-buffer path (cs_flight_step_host_compact): what the device sends per step and where the host keeps the
// reference-shaped results it expands them into.
struct cs_flight_compact {
    unsigned char* d_pack;       // device: [E records][cap reset entries][counter]
    unsigned char* h_pack;       // pinned host mirror
    size_t pack_bytes, rec_bytes, ent_bytes, off_entries, off_counter;
    int cap;                     // reset entries that fit (envs that were reset inside one call)
    float* reward; int32_t* target_find; uint8_t* terminated; uint8_t* win;   // host results, library-owned
    float* state;                // [E][state_stride]
    uint32_t* shadow_found;      // found mask the host rows currently show
    bool dirty;                  // the host rows must be refreshed in full (first step, after cs_flight_reset / import)
    bool pooled;                 // the arrays are segments of a cs_flight_host_pool's (which owns them)
    struct cs_flight_host_pool* pool;   // that pool, and this env's batch index in it
    int pool_index;
};

struct cs_flight {
    cs_flight_cfg cfg;
    csf::FlightParams p;
    int lpe;              // lanes per env of the lane-per-agent kernel
    bool tpe;             // thread-per-env step kernel (n_agents <= kTpeMaxAgents and lanes_per_env in {0, 1, 4})
    int tpe_k;            // threads that share one env's target loop in that kernel (1, 4; 8 in the fused kernel)
    bool fused;           // flight variant: step + belief map in ONE kernel, 8 lanes per env (lanes_per_env = 8, map_size <= 63)
    bool tiled;           // flight variant: thread-per-env step kernel, then flight_map_tile_kernel (the default, map_size <= 63)
    // two-kernel form: job records double buffered over calls; with cfg.map_overlap the map kernel runs on map_stream
    unsigned char* d_jobs;
    int job_parity;
    cudaStream_t map_stream;
    cudaEvent_t ev_step;
    struct MapEvent { cudaEvent_t ev; unsigned long long capture_id; bool valid; } ev_map[2];
    int last_map;         // index into ev_map of the latest map launch, -1 = none
    size_t map_smem;
    int grid, map_grid;
    uint32_t seq;         // generic map path: value of CS_META_SENSE >> 1 that marks "sensed by the latest call" (constant: launches captured in CUDA graphs replay it)
    double* d_tmpl;
    uint8_t* d_actions;   // device staging of the *_host entry point's actions
    double* d_live;       // scratch of cs_flight_stats
    int obs_path;         // 0 = TMA bulk stores for the map observation, 1 = plain stores (A/B measurement)
    uint8_t* d_slab;      // one allocation behind reward | target_find | terminated | win | obs | state
    size_t slab_bytes, host_bytes, off_reward, off_tf, off_term, off_win, off_obs, off_state;
    longlong2* d_lut_meta;
    double2* d_lut;
    float4* d_lut_cells;
    bool have_tmpl;
    cs_flight_compact* hc;
};

// what differs between the handles of a grouped launch (everything else of FlightParams must be equal)
struct GroupEntry {
    int E;
    uint32_t env_id_base, seed, pad;
    long long dyn_rs, dyn_es, tgt_rs, tgt_es;
    double* dyn; double* tgt; float* obs; float* state; float* reward; uint8_t* terminated; uint8_t* win; int32_t* target_find;
    double* stats; const double* tmpl;
};
struct GroupTable { GroupEntry h[kMaxGroup]; };
struct GroupActions { const uint8_t* a[kMaxGroup]; };

struct cs_flight_group {
    int count, n, k, grid_x, device;
    cs_flight* envs[kMaxGroup];
    GroupTable table;
};

// Host-buffer steps of many env batches with pooled buffers (cs_flight_host_pool_*, flight_hostio.cu): the batches' host
// rows, records, agent rows and actions are segments of single allocations, so that a step of ALL batches is one H2D
// copy, one grouped step launch, one grouped pack launch and two D2H copies.
struct PoolGeom { int first[kMaxGroup + 1]; };       // env offset of every batch in the pooled arrays
struct cs_flight_host_pool {
    int count, device, total;
    cs_flight* envs[kMaxGroup];
    PoolGeom geo;
    cs_flight_group* group;      // grouped step launch when the handles allow it (flight_easy, thread-per-env), else null
    GroupTable table;            // per-batch buffers for the grouped pack kernel
    const uint8_t* act_ptrs[kMaxGroup];
    uint8_t* h_actions; uint8_t* d_actions;          // [total][n] (pinned / device)
    // result block (device / pinned mirror): reward f32[total] | target_find i32[total] | terminated u8[total] |
    // win u8[total] | found mask u32[total] | counter | reset entries.  The host views of the first four ARE the mirror.
    unsigned char* d_rec; unsigned char* h_rec;
    size_t rec_block_bytes, off_tf, off_term, off_win, off_found, off_entries, off_counter, ent_bytes;
    size_t fast_bytes;           // what every step copies: records, counter and the first cap_fast entries
    int cap, cap_fast;
    cudaEvent_t ev_rec;          // the record block has arrived (the strided copy of the agent rows is still running)
    float* d_agent;              // device [total][4n]
    float* h_state;              // pinned [total][state_stride]
    uint32_t* shadow_found;      // found mask the host rows currently show
};

namespace csf {

// flight_tpe.cu, one translation unit per pair of n_agents (part P: 2P+1, 2P+2)
cudaError_t launch_tpe_part0(cs_flight*, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t);
cudaError_t launch_tpe_part1(cs_flight*, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t);
cudaError_t launch_tpe_part2(cs_flight*, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t);
cudaError_t launch_tpe_part3(cs_flight*, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t);
cudaError_t launch_group_part0(const cs_flight_group*, const uint8_t* const* d_actions, cudaStream_t);
cudaError_t launch_group_part1(const cs_flight_group*, const uint8_t* const* d_actions, cudaStream_t);
cudaError_t launch_group_part2(const cs_flight_group*, const uint8_t* const* d_actions, cudaStream_t);
cudaError_t launch_group_part3(const cs_flight_group*, const uint8_t* const* d_actions, cudaStream_t);
int fused_lanes_part0();

// flight_lpa.cu: lane-per-agent step / reset kernel (+ the generic belief-map kernel of the flight variant)
cudaError_t launch_lpa(cs_flight*, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t);

// flight_mapk.cu: belief-map kernels that run as their own launch
cudaError_t launch_map_tile(cs_flight*, cudaStream_t);
cudaError_t launch_map_generic(cs_flight*, cudaStream_t);
cudaError_t map_set_smem_limit(size_t generic_bytes);

// flight_aux.cu
cudaError_t launch_obs_full(cs_flight*, float* d_out, cudaStream_t);
cudaError_t launch_map_export(cs_flight*, float* d_out, cudaStream_t);
cudaError_t launch_map_import(cs_flight*, const float* d_in, cudaStream_t);
cudaError_t launch_record_begin(cs_flight*, const cs_episode_buffers&, int T, cudaStream_t);
cudaError_t launch_record(cs_flight*, const cs_episode_buffers&, int t, int T, const uint8_t* actions, cudaStream_t);
cudaError_t launch_live_steps(cs_flight*, cudaStream_t);
cudaError_t launch_pack(cs_flight*, cudaStream_t);
cudaError_t launch_pack_pool(cs_flight_host_pool*, cudaStream_t);

// flight_host.cu
cudaError_t flight_dispatch(cs_flight*, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t);
cudaError_t flight_map_join(cs_flight*, cudaStream_t);

// flight_hostio.cu
void flight_compact_release(cs_flight*);
void flight_compact_mark_dirty(cs_flight*);

}  // namespace csf
