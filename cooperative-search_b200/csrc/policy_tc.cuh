// Agent network on the 5th-generation tensor cores (tcgen05 + TMEM), included by policy.cu.
//
// RNN.forward (network/base_net.py:30-47) for a tile of 128 (env, agent) rows is five small GEMMs with a shared M = 128:
//   fc1   [128 x K1] x [K1 -> 64]                       -> +b, ReLU           -> x1     (input width zero padded to K1)
//   GRU   [128 x 64] x W_ih^T and [128 x 64] x W_hh^T   -> gates r | z | n    -> h'     (network/base_net.py:43, torch GRUCell)
//   fc2.0 [128 x 64] x [64 -> 64]                       -> +b, ReLU           -> f
//   fc2.2 [128 x 64] x [64 -> A (padded to 16)]         -> +b                 -> q
// One CTA of 256 threads owns a tile; threads t and t + 128 share row t -- each takes half of the columns of every
// epilogue (a warp reads the TMEM lanes 32 * (warp % 4) ..., so warps w and w + 4 see the same rows), which halves the
// dependent chain per tile and doubles the warps per SM that cover it (measured: 2.4e9 -> see DESIGN.md rows/s).  Operands are bf16 in shared memory in the canonical
// K-major, no-swizzle UMMA layout -- 16-byte chunks of 8 consecutive k, element (row, k) at
// chunk(k/8) * LBO + row * 16 + (k % 8) * 2 -- so that a thread writes its row's next operand with plain 16-byte
// stores; the weights (torch's (out, in) layout is already K-major) are packed into the same form by the host and
// stay resident in shared memory for the CTA's lifetime.  One elected thread issues the tcgen05.mma instructions
// (SASS: UTCHMMA), accumulators live in tensor memory (256 columns per CTA, two CTAs per SM), completion arrives on an
// mbarrier through tcgen05.commit, and every thread reads its row back with tcgen05.ld (SASS: LDTM) for the
// epilogue: bias, ReLU / sigmoid / tanh, the GRU blend, the bf16 operand of the next GEMM, and finally the masked
// argmax / epsilon-greedy / softmax-sampling action choice of agent/agent.py:66-97.  The r and z gates accumulate
// x1 W_ir^T + h W_hr^T in the same TMEM columns.  bf16 operands, fp32 accumulation, fp32 hidden state in HBM.
// Two instantiations: K1 = 32 for input widths <= 32 (two CTAs per SM) and K1 = 256 for widths 33..256, e.g. the
// search agents (171 obs values + 4 + n): one CTA per SM, fc1 issues only ceil(width / 16) K-steps, and the obs rows
// of a tile are staged by the whole CTA with coalesced loads (tc_wide_inputs).
#pragma once
#include <cuda_bf16.h>

namespace cspol {

constexpr int kTcThreads = 256;                    // two threads per row
constexpr int kTcRows = 128;                       // rows per tile = UMMA M
constexpr int kTcK1 = 32;                          // fc1 input width, padded (input widths <= 32)
constexpr int kTcK1Wide = 256;                     // fc1 input width, padded, of the wide instantiation (widths 33..256)
constexpr int kTcNq = 16;                          // action-value width, padded (UMMA N is a multiple of 16)
constexpr int kTcTmemCols = 256;
constexpr int kALbo = (kTcRows + 1) * 16;          // bytes between K chunks of an A operand (129 rows: bank-conflict-free transposes)
// shared-memory map (bytes) of the instantiation with padded fc1 width K1
template <int K1>
struct TcLayout {
    static constexpr int kOffW1 = 0;                                   // [K1/8 chunks][64][8] bf16
    static constexpr int kOffWih = kOffW1 + (K1 / 8) * 64 * 16;        // [8][192][8]
    static constexpr int kOffWhh = kOffWih + 8 * 192 * 16;
    static constexpr int kOffW2a = kOffWhh + 8 * 192 * 16;             // [8][64][8]
    static constexpr int kOffW2b = kOffW2a + 8 * 64 * 16;              // [8][16][8]
    static constexpr int kOffBias = kOffW2b + 8 * kTcNq * 16;          // fp32: b1[64] | b_rz[128] | b_in[64] | b_hn[64] | b2a[64] | b2b[16]
    static constexpr int kBiasFloats = 64 + 128 + 64 + 64 + 64 + kTcNq;
    static constexpr int kWeightBytes = kOffBias + kBiasFloats * 4;    // what the host packs and every CTA copies
    static constexpr int kOffA0 = (kWeightBytes + 127) & ~127;         // [K1/8][129 rows][8] bf16
    static constexpr int kOffAX = kOffA0 + (K1 / 8) * kALbo;           // [8][129][8]: x1, later f
    static constexpr int kOffAH = kOffAX + 8 * kALbo;                  // [8][129][8]: h, later h'
    static constexpr int kOffBar = kOffAH + 8 * kALbo;                 // mbarrier (8 B) + TMEM base address (4 B)
    static constexpr int kSmemBytes = kOffBar + 16;
    static constexpr int kCtasPerSm = K1 == kTcK1 ? 2 : 1;             // 2 x 104 KB, or 1 x 188 KB of the 227 KB
};
static_assert(TcLayout<kTcK1Wide>::kSmemBytes <= 227 * 1024, "the wide instantiation must fit one CTA's shared memory");

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, no-swizzle shared-memory matrix descriptor: start address, leading-dimension byte offset (between the two
// 16-byte K chunks of one MMA), stride byte offset (between 8-row groups), descriptor version 1 (Blackwell)
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, M = 128
__device__ __forceinline__ constexpr uint32_t tc_idesc(int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(kTcRows >> 4) << 24);
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[128 x N] (+)= A[128 x 16*ksteps] * B[N x 16*ksteps]^T; B is rows n0.. of a weight block with `nrows` rows per chunk
__device__ __forceinline__ void tc_gemm(uint32_t d_tmem, uint32_t a_saddr, uint32_t b_saddr, int nrows, int n0, int N, int ksteps, bool accumulate) {
    const uint32_t idesc = tc_idesc(N);
    for (int k = 0; k < ksteps; ++k) {
        const uint64_t ad = tc_desc(a_saddr + (uint32_t)k * 2u * kALbo, kALbo, 128);
        const uint64_t bd = tc_desc(b_saddr + (uint32_t)n0 * 16u + (uint32_t)k * 2u * (uint32_t)nrows * 16u, (uint32_t)nrows * 16u, 128);
        tc_mma(d_tmem, ad, bd, idesc, (accumulate || k > 0) ? 1u : 0u);
    }
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0, spins = 0;
    while (!ok) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok && ++spins > (1u << 26)) __trap();          // a lost completion must fail loudly, not hang the GPU
    }
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// 8 / 16 consecutive fp32 columns of this thread's TMEM lane (= its row of the accumulator).  The loads are asynchronous:
// several are issued back to back and tc_ld_wait() orders them before the registers are read.
__device__ __forceinline__ void tc_ld8_issue(uint32_t taddr, float* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(taddr));
}
__device__ __forceinline__ void tc_ld16_issue(uint32_t taddr, float* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
                   "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]) : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// ties 8 loaded registers to a point after tc_ld_wait(): an empty volatile asm that "rewrites" them, so that no consumer can be
// scheduled ahead of the wait (volatile asm statements keep their order)
__device__ __forceinline__ void tc_ld_tie8(float* v) {
    asm volatile("" : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]));
}
__device__ __forceinline__ float tc_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float tc_sigmoid(float x) { return fmaf(0.5f, tc_tanh(0.5f * x), 0.5f); }
__device__ __forceinline__ uint32_t tc_pack2(float a, float b) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ uint4 tc_pack8(const float* v) {
    return make_uint4(tc_pack2(v[0], v[1]), tc_pack2(v[2], v[3]), tc_pack2(v[4], v[5]), tc_pack2(v[6], v[7]));
}
// the A operands just written with ordinary stores become visible to the tensor core (async proxy), TMEM reads are ordered
// before the next MMA, and the CTA meets
__device__ __forceinline__ void tc_operands_ready() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
}

// fc1 input rows of one tile for the wide instantiation (widths 33..256), as bf16 in A0's chunks 0 .. 2 * ksteps - 1.
// A search row is 171 floats (684 B), so a thread that assembled its own row with scalar loads would touch 32 lines
// per warp load.  Instead the tile's obs rows, one contiguous block of rows * obs_dim floats, are read by the whole CTA
// with coalesced 16-byte loads and scattered element by element into A0; each thread then writes what is not obs in
// its own row (conv features, the one-hot blocks, which are generated, not loaded, and the zero padding up to the
// last K-step).  The two writers never share a 16-byte chunk except at the edges of the obs range, where both use
// 2-byte stores.
template <class L, class P>
__device__ __forceinline__ void tc_wide_inputs(const P& p, unsigned char* sm, int tile, int r, int half, int tid, int ksteps) {
    constexpr int kU = 8;                                              // 16-byte loads in flight per thread
    const int F = p.feat_dim, D = p.obs_dim, A = p.n_actions;
    unsigned char* a0 = sm + L::kOffA0;
    auto put = [&](int rw, int k, float v) {
        *reinterpret_cast<__nv_bfloat16*>(a0 + (k >> 3) * kALbo + rw * 16 + (k & 7) * 2) = __float2bfloat16_rn(v);
    };
    // this thread's row: everything but the obs elements
    {
        const int rw = tid & (kTcRows - 1);                            // (r: a dead row of a last tile repeats the last row)
        const int la = (p.use_last && p.last_action) ? (int)p.last_action[r] : 255;
        const int kla = (p.use_last && la < A) ? F + D + la : -1;
        const int kid = p.use_id ? F + D + (p.use_last ? A : 0) + r % p.n_agents : -1;
        for (int c = half; c < 2 * ksteps; c += 2) {
            const int k0 = 8 * c;
            float x[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k = k0 + i;
                x[i] = k < F ? p.feat[(size_t)(r / p.n_agents) * F + k] : ((k == kla || k == kid) ? 1.f : 0.f);
            }
            if (k0 + 8 <= F || k0 >= F + D) {
                *reinterpret_cast<uint4*>(a0 + c * kALbo + rw * 16) = tc_pack8(x);
            } else if (k0 < F || k0 + 8 > F + D) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (k0 + i < F || k0 + i >= F + D) put(rw, k0 + i, x[i]);
            }
        }
    }
    // the tile's obs block: element e is obs[row0 + e / D][e % D] -> A0 (row e / D, k = F + e % D)
    const int nrows = p.rows - tile * kTcRows < kTcRows ? p.rows - tile * kTcRows : kTcRows;
    const float* blk = p.obs + (size_t)tile * kTcRows * D;
    const int n = nrows * D;
    int head = (int)(((16u - ((uint32_t)(uintptr_t)blk & 15u)) & 15u) >> 2);   // scalar elements before the first 16-byte boundary
    head = head < n ? head : n;
    auto put_run = [&](int e, const float* v, int cnt) {
        int rw = e / D, k = e - rw * D;
        for (int j = 0; j < cnt; ++j) {
            put(rw, F + k, v[j]);
            if (++k == D) { k = 0; ++rw; }
        }
    };
    if (tid < head) { const float v = __ldcs(blk + tid); put_run(tid, &v, 1); }
    const float4* b4 = reinterpret_cast<const float4*>(blk + head);
    const int n4 = (n - head) >> 2;
    for (int i0 = tid; i0 < n4; i0 += kU * kTcThreads) {
        float4 v[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u)
            if (i0 + u * kTcThreads < n4) v[u] = __ldcs(b4 + i0 + u * kTcThreads);
#pragma unroll
        for (int u = 0; u < kU; ++u)
            if (i0 + u * kTcThreads < n4) {
                const float w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
                put_run(head + 4 * (i0 + u * kTcThreads), w, 4);
            }
    }
    const int t0 = head + 4 * n4;
    if (t0 + tid < n) { const float v = __ldcs(blk + t0 + tid); put_run(t0 + tid, &v, 1); }
}

template <class P, int K1>
__global__ void __launch_bounds__(kTcThreads, TcLayout<K1>::kCtasPerSm) policy_tc_kernel(const __grid_constant__ P p) {
    using L = TcLayout<K1>;
    extern __shared__ __align__(128) unsigned char sm[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int row = tid & (kTcRows - 1), half = tid >> 7;             // this thread's row of the tile and its half of the columns
    const uint32_t sbase = tc_smem_u32(sm);
    const uint32_t bar = sbase + L::kOffBar;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + L::kOffBar + 8);
    const float* bias = reinterpret_cast<const float*>(sm + L::kOffBias);
    const float *b1 = bias, *b_rz = bias + 64, *b_in = bias + 192, *b_hn = bias + 256, *b2a = bias + 320, *b2b = bias + 384;
    const int A = p.n_actions;

    // weights (bf16, canonical layout, packed by the host) + biases -> shared memory, once per CTA
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.wtc);
        uint4* dst = reinterpret_cast<uint4*>(sm);
        for (int i = tid; i < L::kWeightBytes / 16; i += kTcThreads) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(tmem_slot)), "r"(kTcTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_operands_ready();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);  // this warp's 32 TMEM lanes
    uint32_t phase = 0;

    unsigned char* myA0 = sm + L::kOffA0 + row * 16;
    unsigned char* myAX = sm + L::kOffAX + row * 16;
    unsigned char* myAH = sm + L::kOffAH + row * 16;

    const int ksteps1 = K1 == kTcK1 ? kTcK1 / 16 : (p.in_dim + 15) >> 4;   // fc1 K-steps: the wide form issues only those the width needs
    for (int tile = blockIdx.x; tile * kTcRows < p.rows; tile += gridDim.x) {
        const int r_raw = tile * kTcRows + row;
        const bool live = r_raw < p.rows;
        const int r = live ? r_raw : p.rows - 1;
        // ---- inputs: [conv features of the env's map ||] obs || last-action one-hot || agent-id one-hot
        //      (network/base_net.py:31-41, agent/agent.py:38-50)
        if constexpr (K1 == kTcK1) {
            const int la = (p.use_last && p.last_action) ? (int)p.last_action[r] : 255;
#pragma unroll
            for (int cc = 0; cc < kTcK1 / 16; ++cc) {
                const int c = (kTcK1 / 16) * half + cc;
                float x[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) x[i] = policy_input(p, r, la, 8 * c + i);
                *reinterpret_cast<uint4*>(myA0 + c * kALbo) = tc_pack8(x);
            }
        } else {
            tc_wide_inputs<L>(p, sm, tile, r, half, tid, ksteps1);
        }
        tc_operands_ready();
        // ---- fc1
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tc_gemm(tmem + 0, sbase + L::kOffA0, sbase + L::kOffW1, 64, 0, 64, ksteps1, false);
            tc_commit(bar);
        }
        // ... and while the tensor core works on fc1: this thread's half of the row's hidden state (units 32 * half ...), read
        // once (fp32, 8 loads in flight), kept in registers for the GRU blend, bf16 copy -> A operand of the GRU GEMMs
        float hreg[32];
        {
            const float4* hp = reinterpret_cast<const float4*>(p.hidden + (size_t)r * 64 + 32 * half);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 h4 = hp[c];
                hreg[4 * c] = h4.x; hreg[4 * c + 1] = h4.y; hreg[4 * c + 2] = h4.z; hreg[4 * c + 3] = h4.w;
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(myAH + (4 * half + c) * kALbo) = tc_pack8(hreg + 8 * c);
            // the same half row of this CTA's NEXT tile: pull it into L2 now
            const long long rn = (long long)(tile + (int)gridDim.x) * kTcRows + row;
            if (rn < p.rows) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p.hidden + (size_t)rn * 64 + 32 * half));
                if (K1 == kTcK1 && half == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.obs + (size_t)rn * p.obs_dim));
            }
            if constexpr (K1 != kTcK1) {                               // the next tile's obs block, 128-byte lines spread over the CTA
                const long long r0 = (long long)(tile + (int)gridDim.x) * kTcRows;
                if (r0 < p.rows) {
                    const long long nrows = p.rows - r0 < kTcRows ? p.rows - r0 : kTcRows;
                    const char* blk = reinterpret_cast<const char*>(p.obs + (size_t)r0 * p.obs_dim);
                    const long long bytes = nrows * p.obs_dim * 4;
                    for (long long o = 128ll * tid; o < bytes; o += 128ll * kTcThreads) asm volatile("prefetch.global.L2 [%0];" ::"l"(blk + o));
                }
            }
        }
        tc_wait(bar, phase); phase ^= 1u;
        {
            const int c = half;                                        // 32 of the 64 columns each
            float v[32];
            tc_ld16_issue(trow + 32 * c, v);
            tc_ld16_issue(trow + 32 * c + 16, v + 16);
            tc_ld_wait();
            tc_ld_tie8(v); tc_ld_tie8(v + 8); tc_ld_tie8(v + 16); tc_ld_tie8(v + 24);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + b1[32 * c + i], 0.f);
#pragma unroll
            for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(myAX + (4 * c + q) * kALbo) = tc_pack8(v + 8 * q);
        }
        tc_operands_ready();
        // ---- GRU gates: r | z accumulate x1 W_i^T + h W_h^T in columns 0..127; n keeps its two halves apart
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tc_gemm(tmem + 0, sbase + L::kOffAX, sbase + L::kOffWih, 192, 0, 128, 4, false);
            tc_gemm(tmem + 0, sbase + L::kOffAH, sbase + L::kOffWhh, 192, 0, 128, 4, true);
            tc_gemm(tmem + 128, sbase + L::kOffAX, sbase + L::kOffWih, 192, 128, 64, 4, false);
            tc_gemm(tmem + 192, sbase + L::kOffAH, sbase + L::kOffWhh, 192, 128, 64, 4, false);
            tc_commit(bar);
        }
        tc_wait(bar, phase); phase ^= 1u;
        {
            float4* ho = reinterpret_cast<float4*>(p.hidden + (size_t)r * 64 + 32 * half);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const int c = 4 * half + cc;                           // hidden units 8c .. 8c+7
                float gr[8], gz[8], gi[8], gh[8];
                tc_ld8_issue(trow + 8 * c, gr);
                tc_ld8_issue(trow + 64 + 8 * c, gz);
                tc_ld8_issue(trow + 128 + 8 * c, gi);
                tc_ld8_issue(trow + 192 + 8 * c, gh);
                tc_ld_wait();
                tc_ld_tie8(gr); tc_ld_tie8(gz); tc_ld_tie8(gi); tc_ld_tie8(gh);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int j = 8 * c + i, jl = 8 * cc + i;
                    const float rg = tc_sigmoid(gr[i] + b_rz[j]);
                    const float zg = tc_sigmoid(gz[i] + b_rz[64 + j]);
                    const float ng = tc_tanh(gi[i] + b_in[j] + rg * (gh[i] + b_hn[j]));
                    hreg[jl] = (1.f - zg) * ng + zg * hreg[jl];
                }
                if (live) {
                    ho[2 * cc] = make_float4(hreg[8 * cc], hreg[8 * cc + 1], hreg[8 * cc + 2], hreg[8 * cc + 3]);
                    ho[2 * cc + 1] = make_float4(hreg[8 * cc + 4], hreg[8 * cc + 5], hreg[8 * cc + 6], hreg[8 * cc + 7]);
                }
                *reinterpret_cast<uint4*>(myAH + c * kALbo) = tc_pack8(hreg + 8 * cc);
            }
        }
        tc_operands_ready();
        // ---- fc2.0
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tc_gemm(tmem + 0, sbase + L::kOffAH, sbase + L::kOffW2a, 64, 0, 64, 4, false);
            tc_commit(bar);
        }
        tc_wait(bar, phase); phase ^= 1u;
        {
            const int c = half;                                        // 32 of the 64 columns each
            float v[32];
            tc_ld16_issue(trow + 32 * c, v);
            tc_ld16_issue(trow + 32 * c + 16, v + 16);
            tc_ld_wait();
            tc_ld_tie8(v); tc_ld_tie8(v + 8); tc_ld_tie8(v + 16); tc_ld_tie8(v + 24);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + b2a[32 * c + i], 0.f);
#pragma unroll
            for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(myAX + (4 * c + q) * kALbo) = tc_pack8(v + 8 * q);
        }
        tc_operands_ready();
        // ---- fc2.2 -> action values
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tc_gemm(tmem + 64, sbase + L::kOffAX, sbase + L::kOffW2b, kTcNq, 0, kTcNq, 4, false);
            tc_commit(bar);
        }
        tc_wait(bar, phase); phase ^= 1u;
        if (half == 0) {                                               // (warp-uniform: warps 0..3)
            float qv[8];
            tc_ld8_issue(trow + 64, qv);
            tc_ld_wait();
            tc_ld_tie8(qv);
#pragma unroll
            for (int a = 0; a < 8; ++a) qv[a] += b2b[a];
            if (live) policy_choose_action(p, r, qv);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");     // the q read, before the next tile's first MMA
        __syncthreads();
    }
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTcTmemCols) : "memory");
}

}  // namespace cspol
