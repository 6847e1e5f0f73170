// cs_flight handle and the C ABI of the flight_easy / flight envs (include/coopsearch.h).  Kernels live in
// flight_tpe.cu / flight_lpa.cu / flight_aux.cu; see flight_common.cuh for the file map.
#include <new>
#include <vector>
#include "flight_internal.h"

using namespace csf;

namespace {

// lanes per env of the lane-per-agent kernel: the smallest power of two that gives every agent and every target its own lane
int pick_lpe(const cs_flight_cfg& c) {
    int need = c.n_agents > c.target_num ? c.n_agents : c.target_num;
    if (c.lanes_per_env > need) need = c.lanes_per_env;
    int lpe = 1;
    while (lpe < need) lpe <<= 1;
    return lpe > 32 ? 32 : lpe;
}

unsigned long long capture_id(cudaStream_t st) {
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    unsigned long long id = 0;
    if (cudaStreamGetCaptureInfo(st, &status, &id) != cudaSuccess) { cudaGetLastError(); return 0; }
    return status == cudaStreamCaptureStatusActive ? id : 0;
}

// `st` waits for a map-stream event -- only where that is meaningful: an event recorded in the SAME capture (or, outside
// captures, a really recorded one).  An event from another context is covered by stream order: cs_flight_map_sync joins
// the map stream before a capture begins and before it ends.
cudaError_t wait_map_event(cs_flight* h, int idx, cudaStream_t st) {
    if (idx < 0 || !h->ev_map[idx].valid || h->ev_map[idx].capture_id != capture_id(st)) return cudaSuccess;
    return cudaStreamWaitEvent(st, h->ev_map[idx].ev, 0);
}

cudaError_t launch_step(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    switch ((h->p.n - 1) / 2) {
        case 0: return launch_tpe_part0(h, mode, actions, mask, rflags, st);
        case 1: return launch_tpe_part1(h, mode, actions, mask, rflags, st);
        case 2: return launch_tpe_part2(h, mode, actions, mask, rflags, st);
        default: return launch_tpe_part3(h, mode, actions, mask, rflags, st);
    }
}

cudaError_t dispatch(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    if (!h->tpe) return launch_lpa(h, mode, actions, mask, rflags, st);
    if (!h->tiled) return launch_step(h, mode, actions, mask, rflags, st);
    // flight variant, two-kernel form: step / reset kernel (leaves one job record per env), then the tiled map kernel.
    // Job records are double buffered over calls: with map_overlap the map kernel runs on the handle's own stream,
    // concurrently with the NEXT call's step kernel, which writes the other buffer; before a buffer is rewritten the
    // map kernel that read it (two calls ago) must be done.
    const int par = h->job_parity;
    h->p.jobs = h->d_jobs + (size_t)par * (size_t)h->p.E * (size_t)h->p.job_stride;
    cudaError_t e = cudaSuccess;
    if (h->cfg.map_overlap) e = wait_map_event(h, par, st);
    if (e == cudaSuccess) e = launch_step(h, mode, actions, mask, rflags, st);
    if (e != cudaSuccess) return e;
    if (!h->cfg.map_overlap) {
        e = launch_map_tile(h, st);
    } else {
        e = cudaEventRecord(h->ev_step, st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(h->map_stream, h->ev_step, 0);
        if (e == cudaSuccess) e = launch_map_tile(h, h->map_stream);
        if (e == cudaSuccess) e = cudaEventRecord(h->ev_map[par].ev, h->map_stream);
        if (e == cudaSuccess) {
            h->ev_map[par].valid = true;
            h->ev_map[par].capture_id = capture_id(h->map_stream);
            h->last_map = par;
        }
    }
    h->job_parity = par ^ 1;
    return e;
}

// the caller's stream waits for the latest belief-map kernel (no-op unless map_overlap)
cudaError_t map_join(cs_flight* h, cudaStream_t st) {
    if (!h->tiled || !h->cfg.map_overlap) return cudaSuccess;
    return wait_map_event(h, h->last_map, st);
}

inline int up2(int v) { return (v + 1) & ~1; }

// Host-side heading table (see heading_sincos): clusters k = 1..36 around k*pi/18, window = rounding drift after
// `time_limit` steps with a 1.5x margin (measured drift: +-3.4e-14 after 200 steps ~ 1.7e-16 per step).
struct HeadingLut {
    std::vector<longlong2> meta;
    std::vector<double2> tab;
};

inline double ulp_of(double v) {
    long long b;
    memcpy(&b, &v, 8);
    ++b;
    double w;
    memcpy(&w, &b, 8);
    return w - v;
}

void build_heading_lut(int time_limit, HeadingLut* out) {
    const double drift = ((double)time_limit + 16.0) * 2.6e-16;
    out->meta.assign(37, make_longlong2(0, 0));
    out->tab.clear();
    for (int k = 1; k <= 36; ++k) {
        const double centre = (double)k * M_PI / 18.0;
        long long cb;
        memcpy(&cb, &centre, 8);
        long long half = (long long)ceil(drift / ulp_of(centre * 0.999)) + 4;
        if (half > 16384) half = 16384;             // very long episodes: the tail falls back to sincos()
        const long long base = (long long)out->tab.size();
        for (long long off = -half; off <= half; ++off) {
            const long long bits = cb + off;
            double h;
            memcpy(&h, &bits, 8);
            out->tab.push_back(make_double2(sin(h), cos(h)));     // HOST libm: the reference's own bits
        }
        out->meta[k] = make_longlong2(cb, base | (half << 32));
    }
}

// host mirror of the device lookup (tests call it through cs_debug_heading_lut)
void host_heading_sincos(const HeadingLut& lut, double h, double* sn, double* c, int* from_table) {
    const int k = (int)nearbyint(h * (18.0 / M_PI));
    *from_table = 1;
    if (k == 0 && fabs(h) < 7.450580596923828e-09) { *sn = h; *c = 1.0; return; }
    if (k >= 1 && k <= 36) {
        long long hb;
        memcpy(&hb, &h, 8);
        const long long off = hb - lut.meta[k].x, half = lut.meta[k].y >> 32;
        if (off >= -half && off <= half) {
            const double2 v = lut.tab[(size_t)((lut.meta[k].y & 0xffffffffLL) + half + off)];
            *sn = v.x; *c = v.y;
            return;
        }
    }
    *from_table = 0;
    *sn = sin(h); *c = cos(h);
}


// Table of the fused belief-map sweep (flight_map.cuh): the 10 corner bits of a float4 of cells -- x0 = corners
// j..j+4 of corner row i (bits 0..4), x1 = the same of corner row i+1 (bits 5..9) -- give, for each of the 4 cells,
// w = corners-in-view / 4 (exact) and u = (corners-in-view == 0).  (1-d) is applied by the sweep as an fp32 pair.
void build_cell_lut(std::vector<float>* out) {
    out->assign(1024 * 8, 0.0f);
    for (unsigned idx = 0; idx < 1024; ++idx)
        for (int k = 0; k < 4; ++k) {
            const int cnt = __builtin_popcount(idx & (0x63u << k));
            (*out)[idx * 8 + k] = 0.25f * (float)cnt;
            (*out)[idx * 8 + 4 + k] = cnt == 0 ? 1.0f : 0.0f;
        }
}

}  // namespace

namespace csf {
cudaError_t flight_dispatch(cs_flight* h, int mode, const uint8_t* actions, const uint8_t* mask, uint32_t rflags, cudaStream_t st) {
    return dispatch(h, mode, actions, mask, rflags, st);
}
cudaError_t flight_map_join(cs_flight* h, cudaStream_t st) { return map_join(h, st); }
}  // namespace csf

namespace {

// everything cs_flight_create allocates, in one place so that a failure half way frees what exists
int flight_alloc(cs_flight* h) {
    const cs_flight_cfg* cfg = &h->cfg;
    FlightParams& p = h->p;
    const int n = p.n, m = p.m;
    const size_t E = (size_t)p.E;
    CS_CUDA(cudaMalloc(&p.dyn, E * p.rec * sizeof(double)));
    CS_CUDA(cudaMemset(p.dyn, 0, E * p.rec * sizeof(double)));
    // episode counter starts at -1 so that the first reset opens episode 0
    CS_CUDA(cudaMemset2D(reinterpret_cast<uint32_t*>(p.dyn + (size_t)(p.meta_off + CS_META_EPISODE / 2) * p.dyn_rs) + (CS_META_EPISODE & 1),
                         (size_t)p.dyn_es * sizeof(double), 0xFF, sizeof(uint32_t), E));
    CS_CUDA(cudaMalloc(&p.tgt, E * 2 * m * sizeof(double)));
    CS_CUDA(cudaMemset(p.tgt, 0, E * 2 * m * sizeof(double)));
    {
        // all step outputs live in one slab so that the host-buffer step can fetch them with a single D2H copy
        auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
        size_t off = 0;
        h->off_reward = off; off = al(off + E * sizeof(float));
        h->off_tf = off; off = al(off + E * sizeof(int32_t));
        h->off_term = off; off = al(off + E);
        h->off_win = off; off = al(off + E);
        h->off_state = off; off = al(off + E * p.state_stride * sizeof(float));
        h->host_bytes = off;                  // what the host-buffer step copies: obs rows are the state rows' first 4n floats
        h->off_obs = off; off = al(off + E * 4 * n * sizeof(float));
        h->slab_bytes = off;
        CS_CUDA(cudaMalloc(&h->d_slab, off));
        CS_CUDA(cudaMemset(h->d_slab, 0, off));
        p.reward = reinterpret_cast<float*>(h->d_slab + h->off_reward);
        p.target_find = reinterpret_cast<int32_t*>(h->d_slab + h->off_tf);
        p.terminated = h->d_slab + h->off_term;
        p.win = h->d_slab + h->off_win;
        p.obs = reinterpret_cast<float*>(h->d_slab + h->off_obs);
        p.state = reinterpret_cast<float*>(h->d_slab + h->off_state);
    }
    CS_CUDA(cudaMalloc(&h->d_live, sizeof(double)));
    CS_CUDA(cudaMalloc(&p.stats, CS_NUM_STATS * sizeof(double)));
    CS_CUDA(cudaMemset(p.stats, 0, CS_NUM_STATS * sizeof(double)));
    CS_CUDA(cudaMalloc(&h->d_tmpl, (size_t)m * 5 * sizeof(double)));
    CS_CUDA(cudaMemset(h->d_tmpl, 0, (size_t)m * 5 * sizeof(double)));
    p.tmpl = h->d_tmpl;
    if (cfg->variant) {
        CS_CUDA(cudaMalloc(&p.prob_map, E * p.map_stride * sizeof(float)));
        CS_CUDA(cudaMemset(p.prob_map, 0, E * p.map_stride * sizeof(float)));
        if (!h->fused && !h->tiled) {
            CS_CUDA(cudaMalloc(&p.pre, E * p.pre_stride * sizeof(double)));
            CS_CUDA(cudaMemset(p.pre, 0, E * p.pre_stride * sizeof(double)));
        }
        if (h->tiled) {
            CS_CUDA(cudaMalloc(&h->d_jobs, 2 * E * p.job_stride));
            CS_CUDA(cudaMemset(h->d_jobs, 0, 2 * E * p.job_stride));
            p.jobs = h->d_jobs;
            if (cfg->map_overlap) {
                CS_CUDA(cudaStreamCreateWithFlags(&h->map_stream, cudaStreamNonBlocking));
                CS_CUDA(cudaEventCreateWithFlags(&h->ev_step, cudaEventDisableTiming));
                CS_CUDA(cudaEventCreateWithFlags(&h->ev_map[0].ev, cudaEventDisableTiming));
                CS_CUDA(cudaEventCreateWithFlags(&h->ev_map[1].ev, cudaEventDisableTiming));
            }
        }
        std::vector<float> cells;
        build_cell_lut(&cells);
        CS_CUDA(cudaMalloc(&h->d_lut_cells, cells.size() * sizeof(float)));
        CS_CUDA(cudaMemcpy(h->d_lut_cells, cells.data(), cells.size() * sizeof(float), cudaMemcpyHostToDevice));
        p.lut_cells = h->d_lut_cells;
    }
    CS_CUDA(cudaMalloc(&h->d_actions, E * n));
    {
        HeadingLut lut;
        build_heading_lut(cfg->time_limit, &lut);
        CS_CUDA(cudaMalloc(&h->d_lut_meta, lut.meta.size() * sizeof(longlong2)));
        CS_CUDA(cudaMemcpy(h->d_lut_meta, lut.meta.data(), lut.meta.size() * sizeof(longlong2), cudaMemcpyHostToDevice));
        CS_CUDA(cudaMalloc(&h->d_lut, lut.tab.size() * sizeof(double2)));
        CS_CUDA(cudaMemcpy(h->d_lut, lut.tab.data(), lut.tab.size() * sizeof(double2), cudaMemcpyHostToDevice));
        p.lut_meta = h->d_lut_meta;
        p.lut = h->d_lut;
    }
    return CS_OK;
}

}  // namespace

extern "C" {

int cs_flight_create(const cs_flight_cfg* cfg, cs_flight** out) {
    CS_REQUIRE(cfg && out, "cs_flight_create: null argument");
    CS_REQUIRE(cfg->struct_size == sizeof(cs_flight_cfg), "cs_flight_create: cfg.struct_size %u != %zu (ABI mismatch)",
               cfg->struct_size, sizeof(cs_flight_cfg));
    CS_REQUIRE(cfg->num_envs > 0, "num_envs must be > 0");
    CS_REQUIRE(cfg->n_agents >= 1 && cfg->n_agents <= CS_MAX_AGENTS, "n_agents must be in 1..%d", CS_MAX_AGENTS);
    CS_REQUIRE(cfg->target_num >= 1 && cfg->target_num <= CS_MAX_TARGETS, "target_num must be in 1..%d", CS_MAX_TARGETS);
    CS_REQUIRE(cfg->map_size >= 2 && cfg->map_size <= 4096, "map_size out of range");
    CS_REQUIRE(cfg->view_range >= 1, "view_range must be >= 1");
    CS_REQUIRE(cfg->time_limit >= 1 && cfg->time_limit <= 65535, "time_limit must be in 1..65535");
    CS_REQUIRE(cfg->agent_mode >= 0 && cfg->agent_mode <= 3, "No such agent mode");      // flight_env_easy.py:180
    CS_REQUIRE(cfg->target_mode == 0 || cfg->target_mode == 1, "No such target mode");   // flight_env_easy.py:136
    CS_REQUIRE(cfg->variant == 0 || cfg->variant == 1, "variant must be 0 (flight_easy) or 1 (flight)");
    const int l = cfg->lanes_per_env;
    CS_REQUIRE(l == 0 || l == 1 || l == 2 || l == 4 || l == 8 || l == 16 || l == 32, "lanes_per_env must be 0 or a power of two <= 32");

    cs_flight* h = new (std::nothrow) cs_flight();
    if (!h) { cs_set_error("out of host memory"); return CS_ERR_NOMEM; }
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    {
        const cudaError_t e = cudaSetDevice(cfg->device);
        if (e != cudaSuccess) { delete h; CS_CUDA(e); }
    }

    FlightParams& p = h->p;
    const int n = cfg->n_agents, m = cfg->target_num, M = cfg->map_size;
    p.E = cfg->num_envs; p.n = n; p.m = m; p.M = M; p.T = cfg->time_limit;
    p.variant = cfg->variant; p.auto_reset = cfg->auto_reset; p.agent_mode = cfg->agent_mode;
    p.target_mode = cfg->target_mode; p.count_touched = cfg->count_touched;
    p.yaw_off = 2 * n;
    p.meta_off = up2(3 * n);
    p.rec = p.meta_off + CS_META_WORDS / 2;
    p.state_len = 4 * n + 3 * m;
    p.state_stride = (p.state_len + 3) & ~3;
    // constants, computed exactly as the reference's Python floats are
    p.Md = (double)M;
    p.half_M = 0.5 * (double)M;
    p.inv_half = 1.0 / ((double)M / 2.0);
    p.R = (double)cfg->view_range;
    p.R2 = (double)cfg->view_range * (double)cfg->view_range;
    p.v = cfg->velocity;
    p.fk = cfg->safe_dist * 0.8 * cfg->velocity;                 // safe_dist*POTENTIAL_FORCE_FACTOR*velocity (:299)
    p.fd2 = cfg->force_dist * cfg->force_dist;
    const double reach = cfg->force_dist + 1.01 * fabs(cfg->velocity) + 1e-9;
    p.near2 = reach * reach;
    p.q_miss = 1.0 - cfg->detect_prob;                           // (1 - detect_prob) (flight_env.py:292)
    p.pi = M_PI; p.two_pi = 2 * M_PI; p.three_pi = 3 * M_PI; p.half_pi = M_PI / 2; p.turn = M_PI / 18;
    if (cfg->detect_prob >= 1.0) p.thr = 0xFFFFFFFFLL;
    else if (cfg->detect_prob < 0.0) p.thr = -1;
    else p.thr = (long long)floor(cfg->detect_prob * 4294967296.0);
    p.seed = cfg->seed; p.env_id_base = cfg->env_id_base;
    p.inv_turn = 18.0 / M_PI;
    for (int a = 0; a < CS_MAX_AGENTS; ++a)
        p.lin[a] = (n != 1) ? (double)(a * M) / (double)(n - 1) : (double)M / 2.0;
    {
        const double h0 = (cfg->agent_mode <= 1) ? M_PI / 2 : (cfg->agent_mode == 2 ? 0.0 : M_PI);
        p.cos0 = cos(h0);
        p.sin0 = sin(h0);
    }

    p.span_cap = 1; p.span_shift = 0;
    while (p.span_cap < 2 * cfg->view_range) { p.span_cap <<= 1; ++p.span_shift; }
    h->lpe = pick_lpe(*cfg);
    // lanes_per_env: 0 = automatic; 1 or 4 = thread-per-env kernel with that many threads per env; larger = lane-per-agent kernel
    h->tpe = n <= kTpeMaxAgents && (cfg->lanes_per_env == 0 || cfg->lanes_per_env == 1 || cfg->lanes_per_env == 4);
    // the flight variant (map_size <= 63, n_agents <= 8): thread-per-env step kernel + tiled map kernel; lanes_per_env = 8
    // asks for the fused single-kernel form; everything else takes the lane-per-agent step kernel + generic map kernel
    h->fused = cfg->variant == 1 && n <= kTpeMaxAgents && M <= 63 && cfg->lanes_per_env == 8;
    h->tiled = cfg->variant == 1 && h->tpe && M <= 63;
    if (h->fused) h->tpe = true;
    if (cfg->variant == 1 && !h->fused && !h->tiled) h->tpe = false;
    // measured on B200 (tools/sweep_step.sh): one thread per env wins from ~32k envs per launch (2.7e9 against 1.7e9
    // env-steps/s at 65536 envs, 5.0e9 against 2.4e9 at 1M); below that a launch cannot fill the GPU with one thread
    // per env and 4 threads per env match the lane-per-agent kernel's latency
    h->tpe_k = p.E >= 32768 ? 1 : 4;
    if (cfg->lanes_per_env == 1 || cfg->lanes_per_env == 4) h->tpe_k = cfg->lanes_per_env;
    if (const char* kenv = getenv("CS_TPE_K")) {                               // tuning sweeps only
        const int kv = atoi(kenv);
        if (kv == 1 || kv == 4) h->tpe_k = kv;
    }
    if (h->fused) h->tpe_k = fused_lanes_part0();
    p.s_lut = 0;
    p.s_warp = 76;                                        // 37 x 16 B heading-table index, padded
    {
        // belief map geometry: 4x4-cell tiles; scratch of the fused kernel (bytes per env) and of the generic kernel
        // (8-byte words per warp)
        p.tiles = (M + 3) / 4;
        p.map_stride = p.tiles * p.tiles * 16;
        const int Rwords = up2(M + 2) < 64 ? up2(M + 2) : 64;
        p.fm_list = Rwords * 8;
        p.fm_clo = p.fm_list + ((p.tiles * p.tiles * 2 + 15) & ~15);
        p.fm_job = p.fm_clo + ((n * 4 + 15) & ~15);
        p.fm_jobsz = (2 * n * 8 + (1 + m) * 4 + 15) & ~15;
        p.fm_env = p.fm_job + 2 * p.fm_jobsz;
        p.job_stride = 16 + 2 * p.fm_jobsz;
        p.ms_box = 0;
        p.ms_xy = p.ms_box + 2 * n;
        p.ms_hit = p.ms_xy + 2 * n;
        p.ms_warp = up2(p.ms_hit + (m + 1) / 2);
        const int per_cta = kThreads / 32;                                     // generic kernel: one warp per env
        h->map_smem = (size_t)per_cta * p.ms_warp * sizeof(unsigned long long);
        h->map_grid = (p.E + per_cta - 1) / per_cta;
        p.pre_stride = up2(2 * n + (m + 2) / 2);
    }
    h->smem_bytes = (size_t)(kThreads / 32) * p.s_warp * sizeof(double);
    const int env_per_cta = (kThreads / 32) * (32 / h->lpe);
    h->grid = (p.E + env_per_cta - 1) / env_per_cta;
    // structure of arrays exactly where one thread owns one env (flight_tpe_kernel<N, 1>), records otherwise
    if (h->tpe && h->tpe_k == 1) { p.dyn_rs = (long long)p.E; p.dyn_es = 1; p.tgt_rs = (long long)p.E; p.tgt_es = 1; }
    else { p.dyn_rs = 1; p.dyn_es = p.rec; p.tgt_rs = 1; p.tgt_es = 2 * m; }
    h->seq = 1u;
    h->last_map = -1;

    int rc = CS_OK;
    {
        cudaError_t e = lpa_set_smem_limit(h->smem_bytes);
        if (e == cudaSuccess && cfg->variant) e = map_set_smem_limit(h->map_smem);
        if (e != cudaSuccess) { cs_set_error("cudaFuncSetAttribute -> %s", cudaGetErrorString(e)); rc = CS_ERR_CUDA; }
    }
    if (rc == CS_OK) rc = flight_alloc(h);
    if (rc != CS_OK) {            // free whatever exists: a retry with fewer envs must find the memory back
        cs_flight_destroy(h);
        cudaGetLastError();
        return rc;
    }
    *out = h;
    return CS_OK;
}

void cs_flight_destroy(cs_flight* h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    cudaFree(h->p.dyn); cudaFree(h->p.tgt); cudaFree(h->d_slab); cudaFree(h->p.stats); cudaFree(h->d_live);
    cudaFree(h->d_tmpl); cudaFree(h->p.prob_map); cudaFree(h->p.pre); cudaFree(h->d_actions); cudaFree(h->d_lut_meta); cudaFree(h->d_lut);
    cudaFree(h->d_lut_cells);
    if (h->map_stream) { cudaStreamSynchronize(h->map_stream); cudaStreamDestroy(h->map_stream); }
    if (h->ev_step) cudaEventDestroy(h->ev_step);
    if (h->ev_map[0].ev) cudaEventDestroy(h->ev_map[0].ev);
    if (h->ev_map[1].ev) cudaEventDestroy(h->ev_map[1].ev);
    cudaFree(h->d_jobs);
    flight_compact_release(h);
    delete h;
}

int cs_flight_buffers_get(cs_flight* h, cs_flight_buffers* b) {
    CS_REQUIRE(h && b, "cs_flight_buffers_get: null argument");
    const FlightParams& p = h->p;
    b->dyn_row_stride = p.dyn_rs; b->dyn_env_stride = p.dyn_es; b->tgt_row_stride = p.tgt_rs; b->tgt_env_stride = p.tgt_es;
    b->dyn = p.dyn; b->dyn_doubles = p.rec; b->yaw_off = p.yaw_off; b->meta_off = p.meta_off; b->state_len = p.state_len; b->state_stride = p.state_stride;
    b->tgt = p.tgt; b->obs = p.obs; b->state = p.state; b->reward = p.reward; b->terminated = p.terminated;
    b->win = p.win; b->target_find = p.target_find; b->prob_map = p.prob_map; b->stats = p.stats;
    b->map_tiles = p.tiles; b->map_env_stride = p.map_stride;
    b->slab = h->d_slab; b->slab_bytes = h->slab_bytes;
    return CS_OK;
}

int cs_flight_env_info(const cs_flight* h, int32_t* out4) {
    CS_REQUIRE(h && out4, "cs_flight_env_info: null argument");
    out4[0] = 3;                       // n_actions       (flight_env_easy.py:32)
    out4[1] = h->p.state_len;          // state_shape     (:33)
    out4[2] = 4;                       // obs_shape       (:35)
    out4[3] = h->p.T;                  // episode_limit   (:76)
    return CS_OK;
}

int cs_flight_lanes_per_env(const cs_flight* h) { return h ? (h->tpe ? h->tpe_k : h->lpe) : CS_ERR_INVALID; }

// tuning / measurement hook: how cs_flight_obs_full writes the observation rows (0 = TMA bulk stores, 1 = plain stores)
int cs_debug_flight_obs_path(cs_flight* h, int32_t path) {
    CS_REQUIRE(h && (path == 0 || path == 1), "cs_debug_flight_obs_path: bad argument");
    h->obs_path = path;
    return CS_OK;
}

// test hook (host only, no GPU needed): the heading table's sin/cos for `count` headings
int cs_debug_heading_lut(int32_t time_limit, const double* h_in, int32_t count, double* sin_out, double* cos_out,
                         int32_t* from_table) {
    CS_REQUIRE(h_in && sin_out && cos_out && time_limit >= 1, "cs_debug_heading_lut: bad argument");
    HeadingLut lut;
    build_heading_lut(time_limit, &lut);
    for (int i = 0; i < count; ++i) {
        int ft = 0;
        host_heading_sincos(lut, h_in[i], &sin_out[i], &cos_out[i], &ft);
        if (from_table) from_table[i] = ft;
    }
    return (int)lut.tab.size();
}

int cs_flight_set_target_template(cs_flight* h, const double* rows, int32_t nrows) {
    CS_REQUIRE(h && rows, "cs_flight_set_target_template: null argument");
    CS_REQUIRE(nrows >= h->p.m, "target template has %d rows, target_num is %d", nrows, h->p.m);
    const int m = h->p.m;
    double* tmp = new (std::nothrow) double[(size_t)m * 5];
    if (!tmp) { cs_set_error("out of host memory"); return CS_ERR_NOMEM; }
    const double a = (double)h->p.M / 10.0;                  // a = map_size/10  (flight_env_easy.py:97)
    for (int j = 0; j < m; ++j) {
        tmp[5 * j + 0] = a * rows[5 * j + 0];
        tmp[5 * j + 1] = a * rows[5 * j + 1];
        tmp[5 * j + 2] = a * rows[5 * j + 2];
        tmp[5 * j + 3] = a * rows[5 * j + 3];
        tmp[5 * j + 4] = rows[5 * j + 4];
    }
    cudaError_t e = cudaSetDevice(h->cfg.device);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_tmpl, tmp, (size_t)m * 5 * sizeof(double), cudaMemcpyHostToDevice);
    delete[] tmp;
    CS_CUDA(e);
    h->have_tmpl = true;
    return CS_OK;
}

int cs_flight_reset(cs_flight* h, const uint8_t* d_mask, uint32_t flags, void* stream) {
    CS_REQUIRE(h, "cs_flight_reset: null handle");
    CS_REQUIRE((flags & CS_RESET_KEEP_TARGETS) || h->p.target_mode == 1 || h->have_tmpl,
               "target_mode 0 needs cs_flight_set_target_template before reset");
    CS_CUDA(dispatch(h, MODE_RESET, nullptr, d_mask, flags, (cudaStream_t)stream));
    flight_compact_mark_dirty(h);        // the compact host path refreshes its rows in full on the next step
    return CS_OK;
}

int cs_flight_step(cs_flight* h, const uint8_t* d_actions, void* stream) {
    CS_REQUIRE(h && d_actions, "cs_flight_step: null argument");
    CS_CUDA(dispatch(h, MODE_STEP, d_actions, nullptr, 0u, (cudaStream_t)stream));
    flight_compact_mark_dirty(h);        // a device-resident step: the compact host path refreshes its rows in full next time
    return CS_OK;
}

int cs_flight_step_random(cs_flight* h, int32_t k, void* stream) {
    CS_REQUIRE(h && k >= 0, "cs_flight_step_random: bad argument");
    for (int i = 0; i < k; ++i) CS_CUDA(dispatch(h, MODE_STEP, nullptr, nullptr, 0u, (cudaStream_t)stream));
    flight_compact_mark_dirty(h);
    return CS_OK;
}

int cs_flight_obs_full(cs_flight* h, float* d_out, void* stream) {
    CS_REQUIRE(h && d_out, "cs_flight_obs_full: null argument");
    CS_REQUIRE(h->p.variant == 1, "cs_flight_obs_full: only the flight (prob map) variant has a map observation");
    CS_CUDA(map_join(h, (cudaStream_t)stream));
    CS_CUDA(launch_obs_full(h, d_out, (cudaStream_t)stream));
    return CS_OK;
}

int cs_flight_map_export(cs_flight* h, float* d_out, void* stream) {
    CS_REQUIRE(h && d_out, "cs_flight_map_export: null argument");
    CS_REQUIRE(h->p.variant == 1, "cs_flight_map_export: only the flight (prob map) variant has a map");
    CS_CUDA(map_join(h, (cudaStream_t)stream));
    CS_CUDA(launch_map_export(h, d_out, (cudaStream_t)stream));
    return CS_OK;
}

int cs_flight_map_import(cs_flight* h, const float* d_in, void* stream) {
    CS_REQUIRE(h && d_in, "cs_flight_map_import: null argument");
    CS_REQUIRE(h->p.variant == 1, "cs_flight_map_import: only the flight (prob map) variant has a map");
    CS_CUDA(map_join(h, (cudaStream_t)stream));
    CS_CUDA(launch_map_import(h, d_in, (cudaStream_t)stream));
    if (h->tiled && h->cfg.map_overlap) {
        // later map kernels (own stream) must see the imported map: order them after this copy
        CS_CUDA(cudaEventRecord(h->ev_step, (cudaStream_t)stream));
        CS_CUDA(cudaStreamWaitEvent(h->map_stream, h->ev_step, 0));
    }
    return CS_OK;
}

int cs_flight_map_sync(cs_flight* h, void* stream) {
    CS_REQUIRE(h, "cs_flight_map_sync: null handle");
    CS_CUDA(map_join(h, (cudaStream_t)stream));
    return CS_OK;
}

int cs_flight_slab_layout(const cs_flight* h, uint64_t* out8) {
    CS_REQUIRE(h && out8, "cs_flight_slab_layout: null argument");
    out8[0] = h->host_bytes; out8[1] = h->off_reward; out8[2] = h->off_tf; out8[3] = h->off_term; out8[4] = h->off_win;
    out8[5] = h->off_obs; out8[6] = h->off_state; out8[7] = (uint64_t)h->p.state_stride * sizeof(float);
    return CS_OK;
}

int cs_flight_step_host(cs_flight* h, const cs_flight_host_io* io, void* stream) {
    CS_REQUIRE(h && io && io->actions, "cs_flight_step_host: null argument");
    const FlightParams& p = h->p;
    const size_t E = (size_t)p.E;
    cudaStream_t st = (cudaStream_t)stream;
    CS_CUDA(cudaSetDevice(h->cfg.device));
    CS_CUDA(cudaMemcpyAsync(h->d_actions, io->actions, E * p.n, cudaMemcpyHostToDevice, st));
    CS_CUDA(dispatch(h, MODE_STEP, h->d_actions, nullptr, 0u, st));
    CS_CUDA(map_join(h, st));             // a host-buffer step is complete when it returns: the belief map too
    if (io->slab) {
        // one copy for everything: reward | target_find | terminated | win | state (cs_flight_slab_layout); the obs
        // rows are the first 4n floats of the state rows and are not sent twice
        CS_CUDA(cudaMemcpyAsync(io->slab, h->d_slab, h->host_bytes, cudaMemcpyDeviceToHost, st));
    } else {
        if (io->reward) CS_CUDA(cudaMemcpyAsync(io->reward, p.reward, E * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (io->terminated) CS_CUDA(cudaMemcpyAsync(io->terminated, p.terminated, E, cudaMemcpyDeviceToHost, st));
        if (io->win) CS_CUDA(cudaMemcpyAsync(io->win, p.win, E, cudaMemcpyDeviceToHost, st));
        if (io->obs) CS_CUDA(cudaMemcpyAsync(io->obs, p.obs, E * 4 * p.n * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (io->state)   // compact [E][state_len] on the host, padded rows on the device
            CS_CUDA(cudaMemcpy2DAsync(io->state, p.state_len * sizeof(float), p.state, p.state_stride * sizeof(float),
                                      p.state_len * sizeof(float), E, cudaMemcpyDeviceToHost, st));
    }
    if (!(io->flags & CS_HOST_NO_SYNC)) CS_CUDA(cudaStreamSynchronize(st));
    return CS_OK;
}

// Many independent env batches (rollout workers) in one call: batch i is enqueued on streams[i % n_streams] without
// synchronising, then every stream is synchronised once (unless all ios carry CS_HOST_NO_SYNC).  Saves the per-call
// overhead of the host language, which dominates a host-buffer step of a few thousand envs.
int cs_flight_step_host_many(cs_flight* const* envs, const cs_flight_host_io* ios, int32_t count, void* const* streams, int32_t n_streams) {
    CS_REQUIRE(envs && ios && streams && count >= 0 && n_streams >= 1, "cs_flight_step_host_many: bad argument");
    bool sync = false;
    for (int i = 0; i < count; ++i) {
        cs_flight_host_io io = ios[i];
        sync |= !(io.flags & CS_HOST_NO_SYNC);
        io.flags |= CS_HOST_NO_SYNC;
        const int rc = cs_flight_step_host(envs[i], &io, streams[i % n_streams]);
        if (rc != CS_OK) return rc;
    }
    if (sync)
        for (int s = 0; s < n_streams && s < count; ++s) CS_CUDA(cudaStreamSynchronize((cudaStream_t)streams[s]));
    return CS_OK;
}

// ---- grouped device step (flight_tpe_group_kernel) ------------------------------------------------------------
int cs_flight_group_create(cs_flight* const* envs, int32_t count, cs_flight_group** out) {
    CS_REQUIRE(envs && out && count >= 1 && count <= kMaxGroup, "cs_flight_group_create: count must be in 1..%d", kMaxGroup);
    cs_flight_group* g = new (std::nothrow) cs_flight_group();
    if (!g) { cs_set_error("out of host memory"); return CS_ERR_NOMEM; }
    memset(g, 0, sizeof(*g));
    // the configuration shared by the group: handle 0's parameter block with the per-handle fields blanked
    auto shared_part = [](const FlightParams& src) {
        FlightParams c = src;
        c.E = 0; c.env_id_base = 0; c.seed = 0; c.dyn_rs = c.dyn_es = c.tgt_rs = c.tgt_es = 0;
        c.dyn = nullptr; c.tgt = nullptr; c.obs = nullptr; c.state = nullptr; c.reward = nullptr; c.terminated = nullptr; c.win = nullptr;
        c.target_find = nullptr; c.stats = nullptr; c.tmpl = nullptr; c.pre = nullptr; c.prob_map = nullptr; c.jobs = nullptr; c.lut_cells = nullptr;
        c.lut_meta = nullptr; c.lut = nullptr;       // per-handle copies of the same table (same time_limit)
        return c;
    };
    for (int i = 0; i < count; ++i) {
        cs_flight* h = envs[i];
        bool ok = h && h->tpe && h->p.variant == 0 && (i == 0 || (h->p.n == g->n && h->tpe_k == g->k && h->cfg.device == g->device));
        if (ok && i > 0) {
            const FlightParams a = shared_part(envs[0]->p), b = shared_part(h->p);
            ok = memcmp(&a, &b, sizeof(FlightParams)) == 0;
        }
        if (!ok) {
            delete g;
            cs_set_error("cs_flight_group_create: handle %d is not a flight_easy handle with n_agents <= %d, or differs from handle 0 in its configuration (everything but num_envs, env_id_base and seed must be equal) / threads per env / device", i, kTpeMaxAgents);
            return CS_ERR_INVALID;
        }
        if (i == 0) { g->n = h->p.n; g->k = h->tpe_k; g->device = h->cfg.device; }
        const long long threads = (long long)h->p.E * h->tpe_k;
        const int gx = (int)((threads + kTpeThreads - 1) / kTpeThreads);
        if (gx > g->grid_x) g->grid_x = gx;
        if (h->p.E > g->max_E) g->max_E = h->p.E;
        if (i == 0) g->all_even = true;
        if (h->p.E % 2) g->all_even = false;
        g->envs[i] = h;
        GroupEntry& t = g->table.h[i];
        const FlightParams& p = h->p;
        t.E = p.E; t.env_id_base = p.env_id_base; t.seed = p.seed; t.dyn_rs = p.dyn_rs; t.dyn_es = p.dyn_es; t.tgt_rs = p.tgt_rs; t.tgt_es = p.tgt_es;
        t.dyn = p.dyn; t.tgt = p.tgt; t.obs = p.obs; t.state = p.state; t.reward = p.reward; t.terminated = p.terminated; t.win = p.win;
        t.target_find = p.target_find; t.stats = p.stats; t.tmpl = p.tmpl;
    }
    g->count = count;
    *out = g;
    return CS_OK;
}

void cs_flight_group_destroy(cs_flight_group* g) {
    delete g;
}

int cs_flight_group_step(cs_flight_group* g, const uint8_t* const* d_actions, void* stream) {
    CS_REQUIRE(g && d_actions, "cs_flight_group_step: null argument");
    for (int i = 0; i < g->count; ++i) CS_REQUIRE(d_actions[i] != nullptr, "cs_flight_group_step: null actions for handle %d", i);
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    switch ((g->n - 1) / 2) {
        case 0: e = launch_group_part0(g, d_actions, st); break;
        case 1: e = launch_group_part1(g, d_actions, st); break;
        case 2: e = launch_group_part2(g, d_actions, st); break;
        default: e = launch_group_part3(g, d_actions, st); break;
    }
    CS_CUDA(e);
    for (int i = 0; i < g->count; ++i) flight_compact_mark_dirty(g->envs[i]);
    return CS_OK;
}

// Episode-batch writer (see flight_record_kernel).  Buffers are caller-owned device memory.
int cs_flight_record_begin(cs_flight* h, const cs_episode_buffers* b, int32_t T, void* stream) {
    CS_REQUIRE(h && b && T >= 1, "cs_flight_record_begin: bad argument");
    const FlightParams& p = h->p;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t ET = (size_t)p.E * T, O = 4 * (size_t)p.n, S = (size_t)p.state_len, A = 3 * (size_t)p.n;
    CS_CUDA(cudaSetDevice(h->cfg.device));
    CS_CUDA(cudaMemsetAsync(b->o, 0, ET * O * sizeof(float), st));
    CS_CUDA(cudaMemsetAsync(b->s, 0, ET * S * sizeof(float), st));
    CS_CUDA(cudaMemsetAsync(b->o_next, 0, ET * O * sizeof(float), st));
    CS_CUDA(cudaMemsetAsync(b->s_next, 0, ET * S * sizeof(float), st));
    CS_CUDA(cudaMemsetAsync(b->u, 0, ET * p.n, st));
    CS_CUDA(cudaMemsetAsync(b->u_onehot, 0, ET * A, st));
    CS_CUDA(cudaMemsetAsync(b->avail_u, 0, ET * A, st));
    CS_CUDA(cudaMemsetAsync(b->avail_u_next, 0, ET * A, st));
    CS_CUDA(cudaMemsetAsync(b->r, 0, ET * sizeof(float), st));
    CS_CUDA(cudaMemsetAsync(b->padded, 1, ET, st));                       // rollout.py:115-116
    CS_CUDA(cudaMemsetAsync(b->terminated, 1, ET, st));
    CS_CUDA(cudaMemsetAsync(b->episode_reward, 0, (size_t)p.E * sizeof(float), st));
    CS_CUDA(cudaMemsetAsync(b->win_tag, 0, (size_t)p.E, st));
    CS_CUDA(cudaMemsetAsync(b->targets_find, 0, (size_t)p.E * sizeof(int32_t), st));
    CS_CUDA(cudaMemsetAsync(b->length, 0, (size_t)p.E * sizeof(int32_t), st));
    CS_CUDA(launch_record_begin(h, *b, T, st));
    return CS_OK;
}

int cs_flight_record(cs_flight* h, const cs_episode_buffers* b, int32_t t, int32_t T, const uint8_t* d_actions, void* stream) {
    CS_REQUIRE(h && b && d_actions && t >= 0 && t < T, "cs_flight_record: bad argument");
    CS_CUDA(launch_record(h, *b, t, T, d_actions, (cudaStream_t)stream));
    return CS_OK;
}

int cs_flight_stats(cs_flight* h, double* h_out, void* stream) {
    CS_REQUIRE(h && h_out, "cs_flight_stats: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    CS_CUDA(cudaSetDevice(h->cfg.device));
    CS_CUDA(map_join(h, st));            // CS_STAT_TOUCHED is accumulated by the map kernel
    // env_steps = lengths of the finished episodes + steps of the episodes still running
    CS_CUDA(cudaMemsetAsync(h->d_live, 0, sizeof(double), st));
    CS_CUDA(launch_live_steps(h, st));
    double live = 0.0;
    CS_CUDA(cudaMemcpyAsync(h_out, h->p.stats, CS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, st));
    CS_CUDA(cudaMemcpyAsync(&live, h->d_live, sizeof(double), cudaMemcpyDeviceToHost, st));
    CS_CUDA(cudaStreamSynchronize(st));
    h_out[CS_STAT_ENV_STEPS] = h_out[CS_STAT_EP_LEN] + live;
    return CS_OK;
}

}  // extern "C"
