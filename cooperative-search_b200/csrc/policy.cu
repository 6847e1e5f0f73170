// Batched agent network + action selection (SURVEY.md 8f rank 1): policy_tc_kernel (policy_tc.cuh: tcgen05 tensor
// cores, bf16 operands, the default) and policy_kernel (CUDA cores, fp32, one warp per 4 rows: the accuracy reference).
//
// What is restated here (reference: WZN1ng/Cooperative-Search):
//   RNN.forward without the conv front end   network/base_net.py:30-47   fc1 -> ReLU -> GRUCell(64) -> Linear -> ReLU -> Linear
//   input assembly                           agent/agent.py:38-50        obs || last-action one-hot || agent-id one-hot
//   action choice                            agent/agent.py:66-75        q[avail == 0] = -inf; argmax, or a uniform available action with prob. epsilon
//   softmax sampling (alg=reinforce)         agent/agent.py:77-97        Categorical((1-eps) softmax(q) + eps/n_avail, unavailable = 0)
// The dop actor (agent/agent.py:62-63) is the same RNN class with the actor's weights: load those.
// The reference evaluates one (1, in) row per agent per step with a host<->device round trip each; here every (env, agent)
// row of a step is one warp-iteration of a persistent kernel whose CTAs keep the ~120 KB of weights in shared memory.
// fp32 with explicit FMAs, k ascending; sigmoid / tanh from expf / tanhf (no fast-math).
#include <math.h>
#include <new>
#include <vector>
#include "cs_common.cuh"
#include "cs_philox.cuh"

namespace {

constexpr int kH = 64;                 // args.rnn_hidden_dim (common/arguments.py)
constexpr int kPolicyThreads = 512;          // 16 warps per SM at 128 registers: one CTA per SM holds the weights
constexpr int kMaxIn = 32, kMaxActions = 8, kMaxConvOut = 16;
constexpr int kMaxInWide = 256;        // input widths 33..256 (search: (2R-1)^2 + 2 obs values + 4 + n) take the wide instantiations
constexpr int kRowsPerWarp = 4;

// ------------------------------------------------------------------------------------------------
// Conv front end of the `flight` agents (network/base_net.py:10-20,31-41; common/arguments.py:246-265):
//   prob_map [1, M, M] -> Conv2d(1, d1, k1, s1) -> ReLU -> Conv2d(d1, d2, k2, s2, p2) -> ReLU -> flatten -> Linear -> feat[out]
// The reference feeds every agent its own copy of the map (flight_env.py:223-230: 40 KB of observation per env and step)
// and runs the conv once per agent.  The features depend on the env's map only, so here one CTA reads the TILED device
// map of an env once (no observation rows are materialised), de-tiles it into shared memory and leaves `out` floats per
// env; the agents' fc1 input is features || (x^, y^, cos, sin) || last action || agent id.  fp32, explicit FMAs.
// ------------------------------------------------------------------------------------------------
struct ConvParams {
    int E, M, tiles, map_stride, d1, k1, s1, d2, k2, s2, p2, cs, out;
    int w_floats;                // c1_w [d1][k1*k1] | c1_b [d1] | c2_w [d2][d1][k2*k2] | c2_b [d2] | lin_w [out][d2*cs*cs] | lin_b [out]
    const float* map;
    const float* w;
    float* feat;                 // [E][out]
};
constexpr int kConvThreads = 256;

__global__ void __launch_bounds__(kConvThreads) flight_conv_kernel(const __grid_constant__ ConvParams p) {
    extern __shared__ __align__(16) float csm[];
    const int tid = threadIdx.x, M = p.M, cs = p.cs, cs2 = cs * cs;
    float* wsm = csm;
    float* img = wsm + ((p.w_floats + 3) & ~3);
    float* a1 = img + ((M * M + 3) & ~3);
    float* a2 = a1 + p.d1 * cs2;
    for (int i = tid; i < p.w_floats; i += kConvThreads) wsm[i] = p.w[i];
    const float* w1 = wsm;
    const float* b1 = w1 + p.d1 * p.k1 * p.k1;
    const float* w2 = b1 + p.d1;
    const float* b2 = w2 + p.d2 * p.d1 * p.k2 * p.k2;
    const float* wl = b2 + p.d2;
    const float* bl = wl + p.out * p.d2 * cs2;
    const int K = p.d2 * cs2;
    for (int e = blockIdx.x; e < p.E; e += gridDim.x) {
        __syncthreads();                                             // weights loaded / the previous env is done with img, a1, a2
        const float4* src = reinterpret_cast<const float4*>(p.map + (size_t)e * p.map_stride);
        for (int f = tid; f < p.map_stride / 4; f += kConvThreads) {
            const int tile = f >> 2, r = f & 3;
            const int tr = tile / p.tiles, tc = tile - tr * p.tiles;
            const int i = 4 * tr + r, j0 = 4 * tc;
            if (i >= M) continue;
            const float4 v = __ldcs(src + f);
            float* d = img + i * M + j0;
            d[0] = v.x;
            if (j0 + 1 < M) d[1] = v.y;
            if (j0 + 2 < M) d[2] = v.z;
            if (j0 + 3 < M) d[3] = v.w;
        }
        __syncthreads();
        for (int idx = tid; idx < p.d1 * cs2; idx += kConvThreads) {
            const int c = idx / cs2, rem = idx - c * cs2, oy = rem / cs, ox = rem - oy * cs;
            float acc = b1[c];
            const float* wp = w1 + c * p.k1 * p.k1;
            const float* ip = img + (oy * p.s1) * M + ox * p.s1;
            for (int ky = 0; ky < p.k1; ++ky)
                for (int kx = 0; kx < p.k1; ++kx) acc = fmaf(ip[ky * M + kx], wp[ky * p.k1 + kx], acc);
            a1[idx] = fmaxf(acc, 0.f);
        }
        __syncthreads();
        for (int idx = tid; idx < K; idx += kConvThreads) {
            const int c = idx / cs2, rem = idx - c * cs2, oy = rem / cs, ox = rem - oy * cs;
            float acc = b2[c];
            for (int ci = 0; ci < p.d1; ++ci)
                for (int ky = 0; ky < p.k2; ++ky) {
                    const int iy = oy * p.s2 - p.p2 + ky;
                    if (iy < 0 || iy >= cs) continue;
                    for (int kx = 0; kx < p.k2; ++kx) {
                        const int ix = ox * p.s2 - p.p2 + kx;
                        if (ix < 0 || ix >= cs) continue;
                        acc = fmaf(a1[ci * cs2 + iy * cs + ix], w2[((c * p.d1 + ci) * p.k2 + ky) * p.k2 + kx], acc);
                    }
                }
            a2[idx] = fmaxf(acc, 0.f);
        }
        __syncthreads();
        // Linear: 16 lanes per output
        const int o = tid >> 4, part = tid & 15;
        float acc = 0.f;
        if (o < p.out)
            for (int k = part; k < K; k += 16) acc = fmaf(a2[k], wl[o * K + k], acc);
        for (int s = 8; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
        if (o < p.out && part == 0) p.feat[(size_t)e * p.out + o] = acc + bl[o];
    }
}

struct PolicyParams {
    int rows, n_agents, obs_dim, n_actions, in_dim, use_last, use_id, evaluate;
    int mode;                    // 0 = argmax / epsilon-greedy (agent.py:66-75), 1 = softmax sampling (agent.py:77-97)
    float epsilon;
    uint32_t seed, t;
    const float* w;              // packed fp32 weights, see pack order in cs_policy_create
    const unsigned char* wtc;    // bf16 weights in the canonical UMMA layout + fp32 biases (policy_tc.cuh)
    const float* feat;           // [rows / n_agents][feat_dim]: conv features of each env's belief map, or null
    int feat_dim;
    const float* obs;            // [rows][obs_dim]
    const uint8_t* last_action;  // [rows] or null (255 = none yet: zero one-hot)
    const uint8_t* avail;        // [rows][n_actions] or null (= all available)
    float* hidden;               // [rows][64], in/out
    float* q;                    // [rows][n_actions] or null
    uint8_t* actions;            // [rows] out (may alias last_action)
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// element k of the network input of row r: [conv features of the env's map ||] obs || last-action one-hot || agent-id
// one-hot (network/base_net.py:31-41, agent/agent.py:38-50); la = the row's last action (255 = none yet)
__device__ __forceinline__ float policy_input(const PolicyParams& p, int r, int la, int k) {
    const int F = p.feat_dim, A = p.n_actions;
    if (k < F) return p.feat[(size_t)(r / p.n_agents) * F + k];
    k -= F;
    if (k < p.obs_dim) return p.obs[(size_t)r * p.obs_dim + k];
    k -= p.obs_dim;
    if (p.use_last) {
        if (k < A) return la == k ? 1.f : 0.f;
        k -= A;
    }
    if (p.use_id && k < p.n_agents) return (r % p.n_agents) == k ? 1.f : 0.f;
    return 0.f;
}

// Agents.choose_action from the action values of row r (agent/agent.py:66-97): stores q, picks the action.
__device__ __forceinline__ void policy_choose_action(const PolicyParams& p, int r, const float* qv) {
    const int A = p.n_actions;
    int best = -1, navail = 0;
    float bq = -INFINITY;
    unsigned okmask = 0;
#pragma unroll
    for (int a = 0; a < kMaxActions; ++a) {
        if (a >= A) continue;
        if (p.q) p.q[(size_t)r * A + a] = qv[a];
        const bool ok = !p.avail || p.avail[(size_t)r * A + a] != 0;
        navail += ok ? 1 : 0;
        okmask |= ok ? (1u << a) : 0u;
        if (ok && (best < 0 || qv[a] > bq)) { best = a; bq = qv[a]; }     // first maximum, like torch.argmax
    }
    int act = best < 0 ? 0 : best;
    if (p.mode == 1 && navail > 0) {
        // _choose_action_from_softmax: prob = (1 - eps) softmax(q) + eps / n_avail, unavailable actions 0, then
        // argmax (eps == 0 and evaluate) or a Categorical sample (which renormalises)
        float mx = -INFINITY, pr[kMaxActions], sum = 0.f, tot = 0.f;
#pragma unroll
        for (int a = 0; a < kMaxActions; ++a) if (a < A) mx = fmaxf(mx, qv[a]);
#pragma unroll
        for (int a = 0; a < kMaxActions; ++a) { pr[a] = a < A ? expf(qv[a] - mx) : 0.f; sum += pr[a]; }
#pragma unroll
        for (int a = 0; a < kMaxActions; ++a) {
            pr[a] = ((okmask >> a) & 1u) ? (1.f - p.epsilon) * (pr[a] / sum) + p.epsilon / (float)navail : 0.f;
            tot += pr[a];
        }
        if (p.epsilon == 0.f && p.evaluate) {
            float bp = -1.f;
#pragma unroll
            for (int a = 0; a < kMaxActions; ++a) if (a < A && pr[a] > bp) { bp = pr[a]; act = a; }
        } else {
            const cs_u4 w = cs_philox4x32_10((uint32_t)r, p.t, 0u, 0u, p.seed, CS_STREAM_POLICY);
            const float target = (float)(w.z >> 8) * (1.0f / 16777216.0f) * tot;
            float cum = 0.f;
            int pick = -1, last_ok = act;
#pragma unroll
            for (int a = 0; a < kMaxActions; ++a) {
                if (!((okmask >> a) & 1u)) continue;
                last_ok = a;
                cum += pr[a];
                if (pick < 0 && target < cum) pick = a;
            }
            act = pick < 0 ? last_ok : pick;
        }
    } else if (p.mode == 0 && !p.evaluate && p.epsilon > 0.f && navail > 0) {
        // agent.py:71-74: np.random.rand() >= epsilon -> argmax, else a uniform available action
        const cs_u4 w = cs_philox4x32_10((uint32_t)r, p.t, 0u, 0u, p.seed, CS_STREAM_POLICY);
        const float uu = (float)(w.x >> 8) * (1.0f / 16777216.0f);
        if (uu < p.epsilon) {
            int pick = (int)(w.y % (uint32_t)navail);
#pragma unroll
            for (int a = 0; a < kMaxActions; ++a)
                if (((okmask >> a) & 1u) && pick-- == 0) act = a;
        }
    }
    p.actions[r] = (uint8_t)act;
}

// S = 32-wide slices of the input row a lane holds (elements lane + 32 j): 1 for widths <= 32, kMaxInWide / 32 above
template <int S>
__global__ void __launch_bounds__(kPolicyThreads, 1) policy_kernel(const __grid_constant__ PolicyParams p) {
    extern __shared__ __align__(16) float wsm[];
    constexpr unsigned FULL = 0xffffffffu;
    const int in_dim = p.in_dim, A = p.n_actions;
    // packed layout (floats): W1T [in][64] | b1 [64] | WihT [64][192] | bih [192] | WhhT [64][192] | bhh [192] | W2T [64][64] | b2 [64] | W3 [A][64] | b3 [A]
    const int total = in_dim * kH + kH + 2 * (kH * 3 * kH + 3 * kH) + kH * kH + kH + A * kH + A;
    for (int i = threadIdx.x; i < total; i += kPolicyThreads) wsm[i] = p.w[i];
    __syncthreads();
    const float* W1T = wsm;
    const float* b1 = W1T + in_dim * kH;
    const float* WihT = b1 + kH;
    const float* bih = WihT + kH * 3 * kH;
    const float* WhhT = bih + 3 * kH;
    const float* bhh = WhhT + kH * 3 * kH;
    const float* W2T = bhh + 3 * kH;
    const float* b2 = W2T + kH * kH;
    const float* W3 = b2 + kH;
    const float* b3 = W3 + A * kH;

    // RPW consecutive rows per warp iteration: every weight read from shared memory serves RPW rows (the matvecs are
    // bound by the 12 shared-memory loads per k, not by the FMAs)
    constexpr int RPW = kRowsPerWarp;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpc = kPolicyThreads / 32;
    for (int rb = (blockIdx.x * wpc + warp) * RPW; rb < p.rows; rb += gridDim.x * wpc * RPW) {
        int row[RPW];
        float inv[RPW][S], x0[RPW], x1[RPW], h0[RPW], h1[RPW];
#pragma unroll
        for (int u = 0; u < RPW; ++u) {
            const int r = min(rb + u, p.rows - 1);                      // a short last block repeats its last row (writes are guarded)
            row[u] = r;
            // input elements `lane + 32 j` (agent/agent.py:38-50)
            if constexpr (S == 1) {
                inv[u][0] = lane < in_dim ? policy_input(p, r, (p.use_last && p.last_action) ? (int)p.last_action[r] : 255, lane) : 0.f;
            } else {
                const int la = (p.use_last && p.last_action) ? (int)p.last_action[r] : 255;
#pragma unroll
                for (int j = 0; j < S; ++j) inv[u][j] = lane + 32 * j < in_dim ? policy_input(p, r, la, lane + 32 * j) : 0.f;
            }
            x0[u] = b1[lane]; x1[u] = b1[lane + 32];
            h0[u] = p.hidden[(size_t)r * kH + lane]; h1[u] = p.hidden[(size_t)r * kH + lane + 32];
        }
        __syncwarp();                                                    // all rows' last actions are read before any is rewritten
        // fc1 + ReLU: outputs j = lane, lane + 32; k ascending over the whole width
        if constexpr (S == 1) {
            for (int k = 0; k < in_dim; ++k) {
                const float w0 = W1T[k * kH + lane], w1 = W1T[k * kH + lane + 32];
#pragma unroll
                for (int u = 0; u < RPW; ++u) {
                    const float v = __shfl_sync(FULL, inv[u][0], k);
                    x0[u] = fmaf(v, w0, x0[u]);
                    x1[u] = fmaf(v, w1, x1[u]);
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < S; ++j) {
                const int kend = min(32, in_dim - 32 * j);             // slice j holds elements 32 j .. 32 j + kend - 1
                for (int kk = 0; kk < kend; ++kk) {
                    const int k = 32 * j + kk;
                    const float w0 = W1T[k * kH + lane], w1 = W1T[k * kH + lane + 32];
#pragma unroll
                    for (int u = 0; u < RPW; ++u) {
                        const float v = __shfl_sync(FULL, inv[u][j], kk);
                        x0[u] = fmaf(v, w0, x0[u]);
                        x1[u] = fmaf(v, w1, x1[u]);
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < RPW; ++u) { x0[u] = fmaxf(x0[u], 0.f); x1[u] = fmaxf(x1[u], 0.f); }
        // GRUCell: gates r | z | n, outputs j = lane + 32 * o
        float gi[RPW][6], gh[RPW][6];
#pragma unroll
        for (int u = 0; u < RPW; ++u)
#pragma unroll
            for (int o = 0; o < 6; ++o) { gi[u][o] = bih[lane + 32 * o]; gh[u][o] = bhh[lane + 32 * o]; }
        for (int k = 0; k < kH; ++k) {
            float wi[6], wh[6];
#pragma unroll
            for (int o = 0; o < 6; ++o) { wi[o] = WihT[k * 3 * kH + lane + 32 * o]; wh[o] = WhhT[k * 3 * kH + lane + 32 * o]; }
#pragma unroll
            for (int u = 0; u < RPW; ++u) {
                const float xk = __shfl_sync(FULL, k < 32 ? x0[u] : x1[u], k & 31);
                const float hk = __shfl_sync(FULL, k < 32 ? h0[u] : h1[u], k & 31);
#pragma unroll
                for (int o = 0; o < 6; ++o) {
                    gi[u][o] = fmaf(xk, wi[o], gi[u][o]);
                    gh[u][o] = fmaf(hk, wh[o], gh[u][o]);
                }
            }
        }
        float hn0[RPW], hn1[RPW], y0[RPW], y1[RPW];
#pragma unroll
        for (int u = 0; u < RPW; ++u) {
            const float r0 = sigmoidf_(gi[u][0] + gh[u][0]), r1 = sigmoidf_(gi[u][1] + gh[u][1]);
            const float z0 = sigmoidf_(gi[u][2] + gh[u][2]), z1 = sigmoidf_(gi[u][3] + gh[u][3]);
            const float n0 = tanhf(gi[u][4] + r0 * gh[u][4]), n1 = tanhf(gi[u][5] + r1 * gh[u][5]);
            hn0[u] = (1.f - z0) * n0 + z0 * h0[u];
            hn1[u] = (1.f - z1) * n1 + z1 * h1[u];
            if (rb + u < p.rows) {
                p.hidden[(size_t)row[u] * kH + lane] = hn0[u];
                p.hidden[(size_t)row[u] * kH + lane + 32] = hn1[u];
            }
            y0[u] = b2[lane]; y1[u] = b2[lane + 32];
        }
        // fc2: Linear + ReLU, then Linear to the action values
        for (int k = 0; k < kH; ++k) {
            const float w0 = W2T[k * kH + lane], w1 = W2T[k * kH + lane + 32];
#pragma unroll
            for (int u = 0; u < RPW; ++u) {
                const float hk = __shfl_sync(FULL, k < 32 ? hn0[u] : hn1[u], k & 31);
                y0[u] = fmaf(hk, w0, y0[u]);
                y1[u] = fmaf(hk, w1, y1[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < RPW; ++u) {
            const float ya = fmaxf(y0[u], 0.f), yb = fmaxf(y1[u], 0.f);
            const int r = row[u];
            float qv[kMaxActions];
#pragma unroll
            for (int a = 0; a < kMaxActions; ++a) {
                if (a >= A) { qv[a] = 0.f; continue; }
                float part = ya * W3[a * kH + lane] + yb * W3[a * kH + lane + 32];
                for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
                qv[a] = part + b3[a];
            }
            if (lane == 0 && rb + u < p.rows) policy_choose_action(p, r, qv);
        }
    }
}

}  // namespace

#include "policy_tc.cuh"

namespace {
// bf16 (round to nearest even) of a float, on the host
inline uint16_t host_bf16(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
// weight block (out = N rows, in = K columns; torch Linear / GRUCell layout) -> canonical K-major UMMA layout
// [K/8 chunks][Npad rows][8] bf16 at `dst` (zero padded)
void pack_umma(unsigned char* dst, const float* w, int N, int K, int Npad, int Kpad) {
    uint16_t* d = reinterpret_cast<uint16_t*>(dst);
    for (int k = 0; k < Kpad; ++k)
        for (int n = 0; n < Npad; ++n)
            d[(size_t)(k / 8) * Npad * 8 + (size_t)n * 8 + (k % 8)] = (n < N && k < K) ? host_bf16(w[(size_t)n * K + k]) : (uint16_t)0;
}
// the weight block every CTA of policy_tc_kernel<P, K1> copies into shared memory
template <int K1>
std::vector<unsigned char> pack_tc(const cs_policy_weights* hw, int in_dim, int A) {
    using L = cspol::TcLayout<K1>;
    std::vector<unsigned char> tc((size_t)L::kWeightBytes, 0);
    pack_umma(tc.data() + L::kOffW1, hw->fc1_w, kH, in_dim, 64, K1);
    pack_umma(tc.data() + L::kOffWih, hw->w_ih, 3 * kH, kH, 192, 64);
    pack_umma(tc.data() + L::kOffWhh, hw->w_hh, 3 * kH, kH, 192, 64);
    pack_umma(tc.data() + L::kOffW2a, hw->fc2a_w, kH, kH, 64, 64);
    pack_umma(tc.data() + L::kOffW2b, hw->fc2b_w, A, kH, cspol::kTcNq, 64);
    float* b = reinterpret_cast<float*>(tc.data() + L::kOffBias);
    for (int j = 0; j < 64; ++j) b[j] = hw->fc1_b[j];
    for (int j = 0; j < 128; ++j) b[64 + j] = hw->b_ih[j] + hw->b_hh[j];          // r | z gates: the two biases only ever appear summed
    for (int j = 0; j < 64; ++j) { b[192 + j] = hw->b_ih[128 + j]; b[256 + j] = hw->b_hh[128 + j]; b[320 + j] = hw->fc2a_b[j]; }
    for (int a = 0; a < A; ++a) b[384 + a] = hw->fc2b_b[a];
    return tc;
}
}  // namespace

struct cs_policy {
    int device, obs_dim, n_actions, n_agents, use_last, use_id, in_dim, feat_dim;
    ConvParams conv;             // conv front end (cs_policy_set_conv), conv.w == nullptr without one
    float* d_conv_w;
    size_t w_floats;
    float* d_w;
    unsigned char* d_wtc;        // tensor-core weights, packed for the instantiation the width selects
    int wide;                    // input width > kMaxIn: the wide instantiations (policy_kernel<8>, policy_tc_kernel<P, kTcK1Wide>)
};

extern "C" {

int cs_policy_create(const cs_policy_cfg* cfg, const cs_policy_weights* hw, cs_policy** out) {
    CS_REQUIRE(cfg && hw && out, "cs_policy_create: null argument");
    CS_REQUIRE(cfg->struct_size == sizeof(cs_policy_cfg), "cs_policy_create: cfg.struct_size mismatch");
    CS_REQUIRE(cfg->hidden_dim == kH, "cs_policy_create: rnn_hidden_dim must be %d", kH);
    CS_REQUIRE(cfg->n_actions >= 1 && cfg->n_actions <= kMaxActions, "cs_policy_create: n_actions must be in 1..%d", kMaxActions);
    CS_REQUIRE(cfg->conv_out_dim >= 0 && cfg->conv_out_dim <= kMaxConvOut, "cs_policy_create: conv_out_dim must be in 0..%d", kMaxConvOut);
    const int in_dim = cfg->conv_out_dim + cfg->obs_dim + (cfg->last_action ? cfg->n_actions : 0) + (cfg->reuse_network ? cfg->n_agents : 0);
    CS_REQUIRE(cfg->obs_dim >= 1 && in_dim <= kMaxInWide, "cs_policy_create: input width %d exceeds %d", in_dim, kMaxInWide);
    CS_REQUIRE(hw->fc1_w && hw->fc1_b && hw->w_ih && hw->w_hh && hw->b_ih && hw->b_hh && hw->fc2a_w && hw->fc2a_b && hw->fc2b_w && hw->fc2b_b,
               "cs_policy_create: null weight pointer");
    const int A = cfg->n_actions;
    std::vector<float> pk;
    pk.reserve((size_t)in_dim * kH + kH + 2 * (kH * 3 * kH + 3 * kH) + kH * kH + kH + A * kH + A);
    // torch layouts: Linear.weight (out, in); GRUCell.weight_ih / weight_hh (3*hidden, hidden), gates r | z | n
    for (int k = 0; k < in_dim; ++k) for (int j = 0; j < kH; ++j) pk.push_back(hw->fc1_w[(size_t)j * in_dim + k]);
    for (int j = 0; j < kH; ++j) pk.push_back(hw->fc1_b[j]);
    for (int k = 0; k < kH; ++k) for (int j = 0; j < 3 * kH; ++j) pk.push_back(hw->w_ih[(size_t)j * kH + k]);
    for (int j = 0; j < 3 * kH; ++j) pk.push_back(hw->b_ih[j]);
    for (int k = 0; k < kH; ++k) for (int j = 0; j < 3 * kH; ++j) pk.push_back(hw->w_hh[(size_t)j * kH + k]);
    for (int j = 0; j < 3 * kH; ++j) pk.push_back(hw->b_hh[j]);
    for (int k = 0; k < kH; ++k) for (int j = 0; j < kH; ++j) pk.push_back(hw->fc2a_w[(size_t)j * kH + k]);
    for (int j = 0; j < kH; ++j) pk.push_back(hw->fc2a_b[j]);
    for (int a = 0; a < A; ++a) for (int j = 0; j < kH; ++j) pk.push_back(hw->fc2b_w[(size_t)a * kH + j]);
    for (int a = 0; a < A; ++a) pk.push_back(hw->fc2b_b[a]);

    cs_policy* h = new (std::nothrow) cs_policy();
    if (!h) { cs_set_error("out of host memory"); return CS_ERR_NOMEM; }
    h->device = cfg->device; h->obs_dim = cfg->obs_dim; h->n_actions = A; h->n_agents = cfg->n_agents;
    h->use_last = cfg->last_action; h->use_id = cfg->reuse_network; h->in_dim = in_dim; h->w_floats = pk.size(); h->d_w = nullptr;
    h->feat_dim = cfg->conv_out_dim; h->d_conv_w = nullptr; memset(&h->conv, 0, sizeof(h->conv));
    h->wide = in_dim > kMaxIn;
    cudaError_t e = cudaSetDevice(cfg->device);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_w, pk.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_w, pk.data(), pk.size() * sizeof(float), cudaMemcpyHostToDevice);
    // the largest weight block any policy can have, so that handles of different widths coexist
    constexpr size_t kMaxWeights = (size_t)kMaxIn * kH + kH + 2 * (kH * 3 * kH + 3 * kH) + kH * kH + kH + kMaxActions * kH + kMaxActions;
    if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxWeights * sizeof(float)));
    // the wide instantiation's own limit (184 KB at width 256 and 8 actions)
    constexpr size_t kMaxWeightsWide = kMaxWeights + (size_t)(kMaxInWide - kMaxIn) * kH;
    if (e == cudaSuccess && h->wide)
        e = cudaFuncSetAttribute(policy_kernel<kMaxInWide / 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxWeightsWide * sizeof(float)));
    h->d_wtc = nullptr;
    if (e == cudaSuccess) {
        using namespace cspol;
        const std::vector<unsigned char> tc = h->wide ? pack_tc<kTcK1Wide>(hw, in_dim, A) : pack_tc<kTcK1>(hw, in_dim, A);
        e = cudaMalloc(&h->d_wtc, tc.size());
        if (e == cudaSuccess) e = cudaMemcpy(h->d_wtc, tc.data(), tc.size(), cudaMemcpyHostToDevice);
        if (e == cudaSuccess && !h->wide)
            e = cudaFuncSetAttribute(policy_tc_kernel<PolicyParams, kTcK1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcLayout<kTcK1>::kSmemBytes);
        if (e == cudaSuccess && h->wide)
            e = cudaFuncSetAttribute(policy_tc_kernel<PolicyParams, kTcK1Wide>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcLayout<kTcK1Wide>::kSmemBytes);
    }
    if (e != cudaSuccess) { cudaFree(h->d_w); cudaFree(h->d_wtc); delete h; }
    CS_CUDA(e);
    *out = h;
    return CS_OK;
}

void cs_policy_destroy(cs_policy* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaFree(h->d_w);
    cudaFree(h->d_wtc);
    cudaFree(h->d_conv_w);
    delete h;
}

int cs_policy_act(cs_policy* h, const cs_policy_io* io, void* stream) {
    CS_REQUIRE(h && io && io->obs && io->hidden && io->actions && io->rows >= 0, "cs_policy_act: bad argument");
    if (io->rows == 0) return CS_OK;
    PolicyParams p;
    p.rows = io->rows; p.n_agents = h->n_agents; p.obs_dim = h->obs_dim; p.n_actions = h->n_actions; p.in_dim = h->in_dim;
    p.use_last = h->use_last; p.use_id = h->use_id; p.evaluate = io->evaluate; p.epsilon = io->epsilon; p.seed = io->seed; p.t = io->t;
    p.mode = io->mode; p.wtc = h->d_wtc; p.feat = io->feat; p.feat_dim = h->feat_dim;
    CS_REQUIRE(h->feat_dim == 0 || io->feat, "cs_policy_act: this policy has a conv front end: io.feat (cs_policy_conv_features) is required");
    CS_REQUIRE(io->mode == 0 || io->mode == 1, "cs_policy_act: mode must be 0 (argmax / epsilon-greedy) or 1 (softmax sampling)");
    CS_REQUIRE(io->precision == 0 || io->precision == 1, "cs_policy_act: precision must be 0 (fp32) or 1 (bf16 tensor cores)");
    CS_REQUIRE(io->precision == 0 || h->d_wtc, "cs_policy_act: this policy has no tensor-core weights");
    p.w = h->d_w; p.obs = io->obs; p.last_action = io->last_action; p.avail = io->avail; p.hidden = io->hidden; p.q = io->q;
    p.actions = io->actions;
    if (io->precision == 1) {
        // tensor cores: one 128-row tile per CTA iteration, two CTAs per SM (each holds its own copy of the weights); the
        // wide instantiation, one CTA per SM
        using namespace cspol;
        const int tiles = (io->rows + kTcRows - 1) / kTcRows;
        if (h->wide) {
            const int grid_tc = tiles < CS_NUM_SMS_B200 ? tiles : CS_NUM_SMS_B200;
            policy_tc_kernel<PolicyParams, kTcK1Wide><<<grid_tc, kTcThreads, TcLayout<kTcK1Wide>::kSmemBytes, (cudaStream_t)stream>>>(p);
        } else {
            const int grid_tc = tiles < 2 * CS_NUM_SMS_B200 ? tiles : 2 * CS_NUM_SMS_B200;
            policy_tc_kernel<PolicyParams, kTcK1><<<grid_tc, kTcThreads, TcLayout<kTcK1>::kSmemBytes, (cudaStream_t)stream>>>(p);
        }
        cs_count_launch(1);
        CS_CUDA(cudaGetLastError());
        return CS_OK;
    }
    const int wpc = (kPolicyThreads / 32) * kRowsPerWarp;
    int grid = (io->rows + wpc - 1) / wpc;
    if (grid > CS_NUM_SMS_B200) grid = CS_NUM_SMS_B200;                   // persistent: one CTA per SM keeps the weights resident
    if (h->wide)
        policy_kernel<kMaxInWide / 32><<<grid, kPolicyThreads, h->w_floats * sizeof(float), (cudaStream_t)stream>>>(p);
    else
        policy_kernel<1><<<grid, kPolicyThreads, h->w_floats * sizeof(float), (cudaStream_t)stream>>>(p);
    cs_count_launch(1);
    CS_CUDA(cudaGetLastError());
    return CS_OK;
}

int cs_policy_set_conv(cs_policy* h, const cs_policy_conv_cfg* cfg, const cs_policy_conv_weights* hw) {
    CS_REQUIRE(h && cfg && hw, "cs_policy_set_conv: null argument");
    CS_REQUIRE(cfg->struct_size == sizeof(cs_policy_conv_cfg), "cs_policy_set_conv: cfg.struct_size mismatch");
    CS_REQUIRE(hw->c1_w && hw->c1_b && hw->c2_w && hw->c2_b && hw->lin_w && hw->lin_b, "cs_policy_set_conv: null weight pointer");
    CS_REQUIRE(cfg->out_dim == h->feat_dim && cfg->out_dim >= 1, "cs_policy_set_conv: out_dim %d != the policy's conv_out_dim %d", cfg->out_dim, h->feat_dim);
    CS_REQUIRE(cfg->map_size >= 2 && cfg->dim_1 >= 1 && cfg->dim_1 <= 16 && cfg->dim_2 >= 1 && cfg->dim_2 <= 8 && cfg->kernel_size_1 >= 1 &&
               cfg->kernel_size_1 <= cfg->map_size && cfg->stride_1 >= 1 && cfg->kernel_size_2 >= 1 && cfg->stride_2 >= 1 && cfg->padding_2 >= 0,
               "cs_policy_set_conv: conv geometry out of range");
    ConvParams c;
    memset(&c, 0, sizeof(c));
    c.M = cfg->map_size; c.d1 = cfg->dim_1; c.k1 = cfg->kernel_size_1; c.s1 = cfg->stride_1; c.d2 = cfg->dim_2; c.k2 = cfg->kernel_size_2;
    c.s2 = cfg->stride_2; c.p2 = cfg->padding_2; c.out = cfg->out_dim;
    c.cs = (c.M - c.k1) / c.s1 + 1;                                            // network/base_net.py:11
    CS_REQUIRE((c.cs + 2 * c.p2 - c.k2) / c.s2 + 1 == c.cs, "cs_policy_set_conv: the second conv must keep the %d x %d size (base_net.py:19)", c.cs, c.cs);
    const size_t n1 = (size_t)c.d1 * c.k1 * c.k1, n2 = (size_t)c.d2 * c.d1 * c.k2 * c.k2, nl = (size_t)c.out * c.d2 * c.cs * c.cs;
    std::vector<float> pk;
    pk.insert(pk.end(), hw->c1_w, hw->c1_w + n1); pk.insert(pk.end(), hw->c1_b, hw->c1_b + c.d1);
    pk.insert(pk.end(), hw->c2_w, hw->c2_w + n2); pk.insert(pk.end(), hw->c2_b, hw->c2_b + c.d2);
    pk.insert(pk.end(), hw->lin_w, hw->lin_w + nl); pk.insert(pk.end(), hw->lin_b, hw->lin_b + c.out);
    c.w_floats = (int)pk.size();
    const size_t smem = (((size_t)c.w_floats + 3) & ~(size_t)3) * 4 + (((size_t)c.M * c.M + 3) & ~(size_t)3) * 4 + ((size_t)c.d1 + c.d2) * c.cs * c.cs * 4;
    CS_REQUIRE(smem <= 200 * 1024, "cs_policy_set_conv: conv front end needs %zu bytes of shared memory", smem);
    CS_CUDA(cudaSetDevice(h->device));
    cudaFree(h->d_conv_w);
    h->d_conv_w = nullptr;
    CS_CUDA(cudaMalloc(&h->d_conv_w, pk.size() * sizeof(float)));
    CS_CUDA(cudaMemcpy(h->d_conv_w, pk.data(), pk.size() * sizeof(float), cudaMemcpyHostToDevice));
    static size_t cur_limit = 48 * 1024;                                       // per kernel, only ever raised
    if (smem > cur_limit) {
        CS_CUDA(cudaFuncSetAttribute(flight_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cur_limit = smem;
    }
    c.w = h->d_conv_w;
    h->conv = c;
    return CS_OK;
}

int cs_policy_conv_features(cs_policy* h, const float* d_map_tiled, int32_t map_tiles, int32_t map_env_stride, int32_t num_envs,
                            float* d_feat, void* stream) {
    CS_REQUIRE(h && d_map_tiled && d_feat && num_envs >= 0, "cs_policy_conv_features: bad argument");
    CS_REQUIRE(h->conv.w, "cs_policy_conv_features: cs_policy_set_conv first");
    CS_REQUIRE(map_tiles == (h->conv.M + 3) / 4 && map_env_stride >= map_tiles * map_tiles * 16 && map_env_stride % 4 == 0,
               "cs_policy_conv_features: the map layout does not fit map_size %d", h->conv.M);
    if (num_envs == 0) return CS_OK;
    ConvParams c = h->conv;
    c.E = num_envs; c.tiles = map_tiles; c.map_stride = map_env_stride; c.map = d_map_tiled; c.feat = d_feat;
    const size_t smem = (((size_t)c.w_floats + 3) & ~(size_t)3) * 4 + (((size_t)c.M * c.M + 3) & ~(size_t)3) * 4 + ((size_t)c.d1 + c.d2) * c.cs * c.cs * 4;
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    per_sm = per_sm > 4 ? 4 : (per_sm < 1 ? 1 : per_sm);
    const int grid = num_envs < CS_NUM_SMS_B200 * per_sm ? num_envs : CS_NUM_SMS_B200 * per_sm;
    flight_conv_kernel<<<grid, kConvThreads, smem, (cudaStream_t)stream>>>(c);
    cs_count_launch(1);
    CS_CUDA(cudaGetLastError());
    return CS_OK;
}

}  // extern "C"
