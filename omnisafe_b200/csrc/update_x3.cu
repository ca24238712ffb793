// Parity-grade tensor-core variant of the fused minibatch forward + loss + backward kernel
// (PolicyGradient._update, algorithms/on_policy/base/policy_gradient.py:L345-524; PPO._loss_pi base/ppo.py:L35-87;
// PPOLag._compute_adv_surrogate naive_lagrange/ppo_lag.py:L82-102): split-bf16 arithmetic (csrc/x3.cuh), i.e.
// every GEMM is six tcgen05 kind::f16 MMAs over the three bf16 pieces of its fp32 operands with fp32
// accumulation in TMEM -- fp32-level results on the tensor cores (the reference computes fp32 Linear layers,
// omnisafe/utils/model.py:L105-111).
//
// One CTA = one network x a strided set of 128-sample tiles (same grid / per-CTA partial-gradient contract as
// minibatch_grad_tc_kernel).  Warp-specialised: 16 epilogue warps + 1 MMA-issue warp, linked by mbarriers only.
// Each 128-sample tile is worked as two 64-sample halves a / b, each with its own activation buffers, TMEM
// columns, mbarriers and group of 8 epilogue warps; the MMA warp issues every stage for a, then b, so the tensor
// core runs one half's GEMM while the other half's epilogue works (chain GEMMs at M = 64, weight-gradient GEMMs
// with K = 64 samples per half into accumulators shared by both halves):
//
//   per half tile (activations stored ONCE as [sample][feature] bf16x3 tiles; the weight-gradient GEMMs read the
//   same tiles MN-major, so there are no transposed copies):
//     Z1   = X  W1^T            -> H1 = tanh(. + b1)
//     Z2   = H1 W2^T            -> H2 = tanh(. + b2)
//     OUT  = H2 W3^T            -> per-sample loss, dOUT
//     dZ2' = dOUT W3            -> dZ2 = dZ2' (1 - H2^2)   (stored over H2)     | dW3^T += H2^T dOUT
//     dZ1' = dZ2 W2             -> dZ1 = dZ1' (1 - H1^2)   (stored over H1)     | dW2 += dZ2^T H1, db2 += dZ2^T 1
//                                                                               | dW1 += dZ1^T X,  db1 += dZ1^T 1
//   Every epilogue writes its activation in two column halves, each announced by its own mbarrier, so the
//   next layer's MMAs start on k-steps 0-1 while the epilogue still produces k-steps 2-3; weight / bias
//   gradient MMAs run behind the dependent chain while the epilogue warps work.  The loss warps' per-sample inputs
//   are copied asynchronously into shared memory (cp.async) at the start of the tile.
//
// FUSED instantiation = the persistent cooperative kernel of one update iteration: after each minibatch the partial
// gradients are reduced slice-wise behind a software grid barrier, clipped per network, (multi-rank) exchanged over
// NVLink as 8-byte {step tag, value} words, stepped with torch-Adam arithmetic -- speculatively before the norm barrier
// on one rank -- and the weight tiles come back with one TMA bulk copy of a pre-split bf16x3 image maintained by the
// Adam owners.  Loss kinds: PPO-clip, ratio, cost surrogate (fused or stepwise), FOCOPS and P3O (stepwise, with a
// forward-only statistics pass), supplied dOUT (Fisher-vector product backward).
#include "common.cuh"
#include "mlp.cuh"
#include "optim.cuh"
#include "x3.cuh"

namespace osb {

using namespace x3;

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 512;\n" ::: "memory"); }      // epilogue warps only
__device__ __forceinline__ void half_bar_sync(int hf) { asm volatile("bar.sync %0, 256;\n" ::"r"(2 + hf) : "memory"); }   // epilogue warps of half hf

enum X3Loss { X3_PPO_CLIP = 0, X3_RATIO = 1, X3_FOCOPS = 2, X3_COST = 3, X3_FVP = 4, X3_P3O = 5 };   // X3_FVP: dOUT supplied (Fisher-vector product)

struct X3Batch {
    const float* obs; const float* act; const float* logp; const float* adv_r; const float* adv_c;
    const float* tv_r; const float* tv_c; const float* moments; const int* perm;
    long long total; unsigned perm_seed; long long mb_start; int mb_count;
    int identity_stride;     // > 0: row = (mb_start + local) * identity_stride (full-batch passes)
};
struct X3Args {
    X3Batch b;
    int kind; float clip, entropy_coef;
    const float* lagrange;
    const float* theta;
    float* gpart;            // [gridDim.x][P]
    float* stats_part;       // [gridDim.x][3][8]
    const int* stop_flag;
    int O, A, P, net_mask;
    // ---- fused optimiser (persistent mode: one launch = one pass over [mb_start, mb_start + mb_count) in
    //      minibatches of batch_size, each followed by reduce + clip + (all-reduce) + Adam inside the kernel) ----
    int batch_size;
    float* theta_rw; float* grad; float* adam_m; float* adam_v; int* adam_step;
    float critic_norm_coef, max_grad_norm, lr[3];
    float* sumsq_part;           // [3][2][gridDim.x]
    float* train_stats;          // [3][8]
    unsigned int* bar_ctr;       // [3] per-network grid barrier counters, zero at launch
    float* const* peer_buf;      // [world] receive buffers, each [2][world][P] 8-byte words {step tag, value} (pushed over NVLink), or null
    unsigned int* const* peer_flag;   // [world] flag arrays, each [2 * world + 2 * world * 160]
    int world, rank;
    unsigned int step_base;      // exchange step id of this launch's first minibatch (identical on all ranks)
    int* error_flag;
    uint8_t* wimg;               // FUSED: [3 nets][W_IMG] bf16x3 images of the weight tiles (W1 | W2 | W3), written by the Adam owners,
                                 // pulled into shared memory with one bulk copy (TMA) after every optimiser step
    // X3_FOCOPS (first_order/focops.py:L62-108; stepwise launches only): old policy per sample, the minibatch mean of the
    // KL mask from the forward-only pass 1 (null in pass 1), forward_only = statistics only
    const float* mu_old; const float* logstd_old; const float* focops_mask_mean; float focops_lam, focops_eta; int forward_only;
    const float* fvp_dmu;        // X3_FVP: tangent of mu per slab row [total][A] (fvp_tangent_x3_kernel)
    const float* fvp_vec;        // X3_FVP: direction v (its log_std block gives the log_std block of F v)
    float fvp_scale;             // X3_FVP: 1 / (rows * A)
    long long* dbg;              // optional clock64 stamps of CTA (0, 0): [0] = count, then (id, clock) pairs (tools/x3_stage_times.py)
};

constexpr int XT = 128;                      // samples per tile (the unit the tiles are dealt to the CTAs in)
constexpr int HT = 64;                       // samples per half tile: the halves a / b of a tile alternate between the tensor
                                             // core and their epilogue group, so GEMMs of one half run under the epilogue of the other
constexpr int NEPI = 512;                    // 16 epilogue warps: half hf = warp / 8, lane quarter q = warp % 4
constexpr int NGRP = NEPI / 2;               // epilogue threads of one half
constexpr int NTX3 = NEPI + 32;              // + the MMA-issue warp
constexpr uint32_t ACT_SUB = HT * 128, ACT_X3 = 3 * ACT_SUB;        // [64][64] bf16 sub-tile, x3 half tile
constexpr uint32_t D_SUB = HT * 32, D_X3 = 3 * D_SUB;               // [64][16] bf16 (SW32)
constexpr uint32_t W_SUB = 64 * 128, W_X3 = 3 * W_SUB;              // [64][64]
constexpr uint32_t W3_SUB = 16 * 128, W3_X3 = 3 * W3_SUB;           // [16][64]
constexpr uint32_t W_IMG = 2 * W_X3 + W3_X3;                         // 55 296 B: the weight tiles W1 | W2 | W3 as they sit in shared memory
// activation buffers: half a, then half b (half hf of X at OFF_X + hf * ACT_X3, of D at OFF_D + hf * D_X3)
constexpr uint32_t OFF_X = 0, OFF_H1 = OFF_X + 2 * ACT_X3, OFF_H2 = OFF_H1 + 2 * ACT_X3, OFF_D = OFF_H2 + 2 * ACT_X3,
                   OFF_W1 = OFF_D + 2 * D_X3, OFF_W2 = OFF_W1 + W_X3, OFF_W3 = OFF_W2 + W_X3, OFF_ONES = OFF_W3 + W3_X3,
                   OFF_MISC = OFF_ONES + 512;
// misc region (floats unless noted)
constexpr int MF_B1 = 0, MF_B2 = 64, MF_B3 = 128, MF_LS = 144 /* logstd[16] sigma[16] dlogstd acc[16] */, MF_STAT = 192,
              MF_RED = 200 /* [4*8 + 4*16 + 4*16] */, MF_B3ACC = 360, MF_PART = 376 /* [2][256] */, MF_SCAL = 888 /* [16] */, MF_OLD = 904 /* log sigma_old[16], 1 / sigma_old^2 [16] */, MF_END = 936;
constexpr uint32_t OFF_ROWS = OFF_MISC + MF_END * 4;                 // long long [2][128]
constexpr uint32_t OFF_BARS = OFF_ROWS + 2 * XT * 8;                 // uint64 [NBAR]
// mbarriers of one half (barrier b of half hf: index hf * NHB + b), then the weight-image barrier
enum HalfBar { RDY_X0 = 0, RDY_X1, RDY_H1_0, RDY_H1_1, RDY_H2_0, RDY_H2_1, RDY_D, RDY_DZ2_0, RDY_DZ2_1, RDY_DZ1,
               DONE_C1, DONE_C2, DONE_C3, DONE_C4A, DONE_C4B, DONE_C5A, DONE_C5B, DONE_C6, NHB };
constexpr int RDY_W = 2 * NHB, NBAR = 2 * NHB + 1;
constexpr uint32_t OFF_TMEMSLOT = OFF_BARS + NBAR * 8;
constexpr uint32_t OFF_PF = OFF_TMEMSLOT + 16;                        // float [128][12]: per-sample loss inputs (AP == 8), copied asynchronously
constexpr int PF_LD = 12;
constexpr uint32_t X3_SMEM = OFF_PF + XT * PF_LD * 4;
static_assert(XT * (5 + 2 * 16) * 4 <= 2 * ACT_X3, "per-row loss sums must fit the H2 buffers");
static_assert(1024 + X3_SMEM <= 227 * 1024, "dynamic shared memory of the bf16x3 update kernel exceeds 227 KB");
// TMEM columns: per half Z_A | Z_B | OUT (half hf at hf * T_HALF), then the weight / bias gradients shared by both halves
constexpr uint32_t T_ZA = 0, T_ZB = 64, T_OUT = 128, T_HALF = 144;
constexpr uint32_t T_DW1 = 2 * T_HALF, T_DW2 = T_DW1 + 64, T_DW3 = T_DW2 + 64, T_DB1 = T_DW3 + 16, T_DB2 = T_DB1 + 16, T_COLS = 512;
static_assert(T_DB2 + 16 <= T_COLS, "TMEM columns");

__device__ __forceinline__ unsigned long long x3_feistel(unsigned long long k, unsigned long long n, unsigned seed) {
    int bits = 2;
    while ((1ull << bits) < n) bits += 2;
    const int half = bits >> 1;
    const unsigned mask = (1u << half) - 1u;
    unsigned long long x = k;
    do {
        unsigned l = (unsigned)(x >> half) & mask, r = (unsigned)x & mask;
#pragma unroll
        for (int round = 0; round < 4; ++round) {
            const unsigned f = mix32(r ^ (seed + 0x9E3779B9u * (unsigned)(round + 1))) & mask;
            const unsigned nl = r;
            r = l ^ f;
            l = nl;
        }
        x = ((unsigned long long)l << half) | r;
    } while (x >= n);
    return x;
}

// fp32 parameters of one network -> bf16x3 weight tiles + fp32 biases in shared memory (all NEPI epilogue threads).
// All global loads are issued before the first store (one L2 round trip instead of one per loop iteration).
// O < 64 ("ones column"): column 63 of the X tile holds 1.0 and column 63 of the W1 tile holds b1, so the layer-1
// bias rides in the GEMM and db1 falls out of the dW1 accumulator (column 63) -- no bias add, no db1 MMAs.
__device__ __forceinline__ void stage_weights_x3(uint32_t sbase, float* misc, const float* __restrict__ theta,
                                                 const NetLayout& L, int net, int O, int A, int tid) {
    const bool ones_col = O < 64;
    float a1[4], b1[4], a2[4], b2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {                          // W1 / W2: [64 n][64 k], two columns per thread
        const int i = tid + j * NEPI;
        const int n = i >> 5, k = (i & 31) << 1;
        a1[j] = (k < O) ? __ldcg(theta + L.off_w1 + n * O + k) : 0.f;
        b1[j] = (k + 1 < O) ? __ldcg(theta + L.off_w1 + n * O + k + 1) : ((ones_col && k == 62) ? __ldcg(theta + L.off_b1 + n) : 0.f);
        a2[j] = __ldcg(theta + L.off_w2 + n * 64 + k); b2[j] = __ldcg(theta + L.off_w2 + n * 64 + k + 1);
    }
    const int o3 = tid >> 5, k3 = (tid & 31) << 1;         // W3: [16 o][64 k], rows >= out zero
    const float a3 = (o3 < L.out) ? __ldcg(theta + L.off_w3 + o3 * 64 + k3) : 0.f;
    const float b3 = (o3 < L.out) ? __ldcg(theta + L.off_w3 + o3 * 64 + k3 + 1) : 0.f;
    float bb1 = 0.f, bb2 = 0.f, bb3 = 0.f, ls = 0.f;
    if (tid < 64) { bb1 = ones_col ? 0.f : __ldcg(theta + L.off_b1 + tid); bb2 = __ldcg(theta + L.off_b2 + tid); }
    if (tid < 16) {
        bb3 = (tid < L.out) ? __ldcg(theta + L.off_b3 + tid) : 0.f;
        ls = (net == 0 && tid < A) ? __ldcg(theta + L.off_logstd + tid) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int i = tid + j * NEPI;
        const int n = i >> 5, k = (i & 31) << 1;
        uint32_t w0, w1, w2;
        const uint32_t off = off128(n, k);
        split2(a1[j], b1[j], w0, w1, w2);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W1 + off), "r"(w0) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W1 + W_SUB + off), "r"(w1) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W1 + 2 * W_SUB + off), "r"(w2) : "memory");
        split2(a2[j], b2[j], w0, w1, w2);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W2 + off), "r"(w0) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W2 + W_SUB + off), "r"(w1) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W2 + 2 * W_SUB + off), "r"(w2) : "memory");
    }
    {
        uint32_t w0, w1, w2;
        split2(a3, b3, w0, w1, w2);
        const uint32_t off = off128(o3, k3);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W3 + off), "r"(w0) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W3 + W3_SUB + off), "r"(w1) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sbase + OFF_W3 + 2 * W3_SUB + off), "r"(w2) : "memory");
    }
    if (tid < 64) { misc[MF_B1 + tid] = bb1; misc[MF_B2 + tid] = bb2; }
    if (tid < 16) {
        misc[MF_B3 + tid] = bb3;
        const float sd = expf(ls);
        misc[MF_LS + tid] = ls; misc[MF_LS + 16 + tid] = sd; misc[MF_LS + 32 + tid] = 1.f / (sd * sd);   // log sigma, sigma, 1 / sigma^2
    }
}

__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned int ld_acquire_sys_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u32(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

constexpr int PSTR = 9472;          // FUSED: row stride of the private partial-gradient layout [3][G][PSTR] (16 B aligned rows)

// FUSED = false: one minibatch, per-CTA partial gradients out (the contract of minibatch_grad_tc_kernel).
// FUSED = true : persistent cooperative kernel -- the CTA loops over all minibatches of one update iteration
//   (policy_gradient.py:L369-381); after each minibatch the CTAs of a network meet at a software grid barrier,
//   reduce the partial gradients slice-wise in a fixed order, clip per network (clip_grad_norm_), exchange the
//   clipped slice with the peer ranks over NVLink (clip -> average -> step, policy_gradient.py:L437-443,
//   distributed.py:L193-198), apply torch-Adam and re-stage the new weights: no relaunch, no separate
//   optimiser kernel.
// AP = padded action width of the loss epilogue (8 or 16).
// (17 warps: registers are allocated per 4 warps, so a 544-thread block is sized like 640 threads: 96 registers each;
//  __maxnreg__(120) compiles but cannot launch)
template <bool FUSED, int AP>
__global__ void __launch_bounds__(NTX3, 1) minibatch_grad_x3_kernel(X3Args p) {
    if (p.stop_flag && *p.stop_flag) return;
    const int net = (gridDim.y == 1) ? (__ffs(p.net_mask) - 1) : (int)blockIdx.y;
    if (!((p.net_mask >> net) & 1)) return;

    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
    const uint32_t sbase = smem_u32(smem_raw) + pad;
    uint8_t* gbase = smem_raw + pad;
    float* misc = reinterpret_cast<float*>(gbase + OFF_MISC);
    long long* sRowBuf = reinterpret_cast<long long*>(gbase + OFF_ROWS);
    const uint32_t bars = sbase + OFF_BARS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gbase + OFF_TMEMSLOT);
    auto bar = [&](int i) { return bars + (uint32_t)i * 8u; };

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int O = p.O, A = p.A;
    const int G = (int)gridDim.x;
    const NetLayout L = net_layout(net, O, A);
    const int noff = net_offset(net, O, A);
    const float* theta = (FUSED ? p.theta_rw : p.theta) + noff;
    // partial gradients of this CTA: FUSED -> private aligned layout, else the [CTA][P] layout optim_fused reads
    float* gout = FUSED ? p.gpart + ((size_t)((gridDim.y == 1 ? 0 : net) * G + (int)blockIdx.x)) * PSTR
                        : p.gpart + (size_t)blockIdx.x * p.P + noff;
    const bool is_mma_warp = warp == NEPI / 32;
    const int batch = FUSED ? p.batch_size : p.b.mb_count;
    const int n_mb = (p.b.mb_count + batch - 1) / batch;
    const bool ones_col = O < 64;          // bias of layer 1 / db1 ride in the GEMMs (see stage_weights_x3)

    // ---- one-time setup -------------------------------------------------------------------------------
    if (!is_mma_warp) {
        stage_weights_x3(sbase, misc, theta, L, net, O, A, tid);
        if (tid < 128) reinterpret_cast<uint32_t*>(gbase + OFF_ONES)[tid] = 0x3F803F80u;       // bf16 1.0 x 256
        if (tid < 16 && (!FUSED && p.kind == X3_FOCOPS)) {
            const float lo = (tid < A) ? __ldg(p.logstd_old + tid) : 0.f;
            const float so = expf(lo);
            misc[MF_OLD + tid] = lo; misc[MF_OLD + 16 + tid] = 1.f / (so * so);
        }
    } else {
        if (lane == 0) {
            for (int i = 0; i < NBAR; ++i) {
                const int b = i % NHB;          // producers: the 8 warps of a half, its 4 loss warps, one commit / expect_tx (RDY_W)
                const uint32_t cnt = (i == RDY_W || b >= DONE_C1) ? 1u : (b == RDY_D ? 4u : 8u);
                asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar(i)), "r"(cnt) : "memory");
            }
            mbar_init_fence();
        }
        __syncwarp();
        tmem_alloc(tmem_slot, T_COLS);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (is_mma_warp) {
        // ======================= MMA-issue warp: uniform control flow, one elected lane issues ==============
        const bool leader = elect_one_sync();
        const uint64_t dX = desc128(sbase + OFF_X), dH1 = desc128(sbase + OFF_H1), dH2 = desc128(sbase + OFF_H2);
        const uint64_t dD = desc32(sbase + OFF_D), dW1 = desc128(sbase + OFF_W1), dW2 = desc128(sbase + OFF_W2);
        const uint64_t dW3 = desc128(sbase + OFF_W3), dOnes = desc32(sbase + OFF_ONES);
        // chain GEMMs: M = 64 samples of one half; weight-gradient GEMMs: M = 64 weight rows, K = the 64 samples of one half
        const uint32_t id_fwd = idesc_bf16(64, 64, 0, 0), id_out = idesc_bf16(64, 16, 0, 0), id_bwd = idesc_bf16(64, 64, 0, 1);
        const uint32_t id_dw = idesc_bf16(64, 64, 1, 1), id_dw16 = idesc_bf16(64, 16, 1, 1);
        const bool backward = !(!FUSED && p.forward_only);       // forward-only statistics pass (FOCOPS / P3O pass 1): no backward
        auto hbar = [&](int hf, int b) { return bar(hf * NHB + b); };
        auto commit = [&](int hf, int b) { if (leader) mma_commit_a(hbar(hf, b)); __syncwarp(); };
        int it = 0;
#pragma unroll 1
        for (int mb = 0; mb < n_mb; ++mb) {
            const int count = min(batch, p.b.mb_count - mb * batch);
            const int ntiles = (count + XT - 1) / XT;
#pragma unroll 1
            for (int tile = blockIdx.x; tile < ntiles; tile += G, ++it) {
                const uint32_t par = (uint32_t)(it & 1);
                const bool first = tile == (int)blockIdx.x;         // half a of the first tile of a minibatch overwrites the accumulators
                const bool last = tile + G >= ntiles;
                // Every stage is issued for half a, then half b: while the tensor core runs one half's GEMM, the
                // epilogue group of the other half works on the previous result.
                // Z1 = X W1^T  (k-steps 0-1 after the first column half of X, 2-3 after the second)
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
#pragma unroll 1
                    for (int ph = 0; ph < 2; ++ph) {
                        mbar_wait_a(hbar(hf, RDY_X0 + ph), par);
                        tc_fence_after();
                        gemm_x3_warp(leader, tmem + hf * T_HALF + T_ZA, desc_add(dX, hf * ACT_X3 + 64u * ph), ACT_SUB, 32u, desc_add(dW1, 64u * ph), W_SUB, 32u, id_fwd, 2, ph > 0);
                    }
                    commit(hf, DONE_C1);
                }
                // db2 of the PREVIOUS tile (dZ2 still sits in the H2 buffers until this tile's E2): runs under E1,
                // completes before Z2 (in-order pipe), so DONE_C2 covers it
                if (!first && backward)
#pragma unroll 1
                    for (int hf = 0; hf < 2; ++hf)
                        gemm_x3_warp(leader, tmem + T_DB2, desc_add(dH2, hf * ACT_X3), ACT_SUB, 2048u, dOnes, 0u, 0u, id_dw16, 4, hf > 0 || tile != (int)blockIdx.x + G);
                // Z2 = H1 W2^T
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
#pragma unroll 1
                    for (int ph = 0; ph < 2; ++ph) {
                        mbar_wait_a(hbar(hf, RDY_H1_0 + ph), par);
                        tc_fence_after();
                        gemm_x3_warp(leader, tmem + hf * T_HALF + T_ZB, desc_add(dH1, hf * ACT_X3 + 64u * ph), ACT_SUB, 32u, desc_add(dW2, 64u * ph), W_SUB, 32u, id_fwd, 2, ph > 0);
                    }
                    commit(hf, DONE_C2);
                }
                // OUT = H2 W3^T
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
#pragma unroll 1
                    for (int ph = 0; ph < 2; ++ph) {
                        mbar_wait_a(hbar(hf, RDY_H2_0 + ph), par);
                        tc_fence_after();
                        gemm_x3_warp(leader, tmem + hf * T_HALF + T_OUT, desc_add(dH2, hf * ACT_X3 + 64u * ph), ACT_SUB, 32u, desc_add(dW3, 64u * ph), W3_SUB, 32u, id_out, 2, ph > 0);
                    }
                    commit(hf, DONE_C3);
                }
                if (!backward) continue;
                // dZ2' = dOUT W3 ; dW3^T += H2^T dOUT
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
                    mbar_wait_a(hbar(hf, RDY_D), par);
                    tc_fence_after();
                    gemm_x3_warp(leader, tmem + hf * T_HALF + T_ZA, desc_add(dD, hf * D_X3), D_SUB, 32u, dW3, W3_SUB, 2048u, id_bwd, 1, false);
                    commit(hf, DONE_C4A);
                    gemm_x3_warp(leader, tmem + T_DW3, desc_add(dH2, hf * ACT_X3), ACT_SUB, 2048u, desc_add(dD, hf * D_X3), D_SUB, 512u, id_dw16, 4, !first || hf > 0);
                    commit(hf, DONE_C4B);
                }
                // dZ1' = dZ2 W2 ; dW2 += dZ2^T H1
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
#pragma unroll 1
                    for (int ph = 0; ph < 2; ++ph) {
                        mbar_wait_a(hbar(hf, RDY_DZ2_0 + ph), par);
                        tc_fence_after();
                        gemm_x3_warp(leader, tmem + hf * T_HALF + T_ZB, desc_add(dH2, hf * ACT_X3 + 64u * ph), ACT_SUB, 32u, desc_add(dW2, 4096u * ph), W_SUB, 2048u, id_bwd, 2, ph > 0);
                    }
                    commit(hf, DONE_C5A);
                    gemm_x3_warp(leader, tmem + T_DW2, desc_add(dH2, hf * ACT_X3), ACT_SUB, 2048u, desc_add(dH1, hf * ACT_X3), ACT_SUB, 2048u, id_dw, 4, !first || hf > 0);
                    commit(hf, DONE_C5B);
                }
                // dW1 += dZ1^T X (column 63 = db1 with the ones column) ; last tile of the minibatch: its own db2
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
                    mbar_wait_a(hbar(hf, RDY_DZ1), par);
                    tc_fence_after();
                    const bool acc = !first || hf > 0;
                    gemm_x3_warp(leader, tmem + T_DW1, desc_add(dH1, hf * ACT_X3), ACT_SUB, 2048u, desc_add(dX, hf * ACT_X3), ACT_SUB, 2048u, id_dw, 4, acc);
                    if (!ones_col) gemm_x3_warp(leader, tmem + T_DB1, desc_add(dH1, hf * ACT_X3), ACT_SUB, 2048u, dOnes, 0u, 0u, id_dw16, 4, acc);
                    if (last) gemm_x3_warp(leader, tmem + T_DB2, desc_add(dH2, hf * ACT_X3), ACT_SUB, 2048u, dOnes, 0u, 0u, id_dw16, 4, acc);
                    commit(hf, DONE_C6);
                }
            }
        }
    } else {
        // ======================= epilogue warps ===============================================================
        const int q = warp & 3, h = warp >> 2;          // lane quarter, column group of the gradient read-out
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        // tile loop: the 8 warps of half hf = warp / 8 own its 64 samples; the M = 64 accumulators hold sample row
        // 16 q + l in lane l < 16 of quarter q.  Warps with h2 == 0 (the loss warps) also run the loss, one lane l < 16 per sample.
        const int hf = warp >> 3, h2 = h & 1, gtid = tid & (NGRP - 1);
        const int s_row = 16 * q + (lane & 15);          // sample row of this thread in its half
        const bool loss_warp = h2 == 0, loss_lane = loss_warp && lane < 16;
        const uint32_t sX = sbase + OFF_X + hf * ACT_X3, sH1 = sbase + OFF_H1 + hf * ACT_X3, sH2 = sbase + OFF_H2 + hf * ACT_X3;
        const uint32_t sD = sbase + OFF_D + hf * D_X3;
        const uint32_t tHalf = tmem + lane_base + hf * T_HALF;
        // column of this thread in column half ph: 32 ph + 16 h2 + 8 (lane / 16) .. + 7 (see tmem_ld8_m64)
        const int ccol = 16 * h2 + 8 * (lane >> 4);
        auto hbar = [&](int b) { return bar(hf * NHB + b); };
        const float lam = (p.lagrange != nullptr) ? __ldg(p.lagrange) : 0.f;
        float m_r = 0.f, s_r = 1.f, m_c = 0.f;
        if (p.b.moments) { m_r = __ldg(p.b.moments + 0); s_r = __ldg(p.b.moments + 1); m_c = __ldg(p.b.moments + 2); }
        const float inv_sr = 1.f / s_r, inv_1lam = 1.f / (1.f + lam);
        float* sB1 = misc + MF_B1; float* sB2 = misc + MF_B2; float* sB3 = misc + MF_B3; float* sLs = misc + MF_LS;
        float* sRed = misc + MF_RED; float* sPart = misc + MF_PART; float* sScal = misc + MF_SCAL;

        // X gather: thread -> row xm = gtid / 4 of its half, columns 32 ph + 8 (gtid % 4) .. + 7 in column half ph
        const int xm = gtid >> 2, xc = (gtid & 3) << 3;
        const bool vec = (O & 3) == 0;
        float xpre[16];
        auto prefetch_x = [&](const long long* rows) {
            const long long row = rows[hf * HT + xm];
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const int c0 = 32 * ph + xc;
                if (vec) {
#pragma unroll
                    for (int v4 = 0; v4 < 2; ++v4) {
                        const int c = c0 + 4 * v4;
                        const float4 v = (row >= 0 && c < O) ? __ldg(reinterpret_cast<const float4*>(p.b.obs + row * O + c))
                                                             : make_float4(0.f, 0.f, 0.f, 0.f);
                        xpre[8 * ph + 4 * v4] = v.x; xpre[8 * ph + 4 * v4 + 1] = v.y; xpre[8 * ph + 4 * v4 + 2] = v.z; xpre[8 * ph + 4 * v4 + 3] = v.w;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) xpre[8 * ph + i] = (row >= 0 && c0 + i < O) ? __ldg(p.b.obs + row * O + c0 + i) : 0.f;
                }
            }
            if (ones_col && xc == 24) xpre[15] = 1.0f;     // column 63: the ones column (every row: padding rows have dZ1 = 0)
        };
        auto announce = [&](int b) {        // this warp's stores of one column half are visible to the tensor core
            fence_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(hbar(b));
        };
        const bool dbg_on = p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && (tid == 0 || tid == 256);
        int dbg_n = 0;
        auto stamp = [&](int id) {
            if (dbg_on && dbg_n < 400) {
                long long* d = p.dbg + (tid == 0 ? 0 : 1024);
                d[1 + 2 * dbg_n] = id; d[2 + 2 * dbg_n] = clock64(); ++dbg_n; d[0] = dbg_n;
            }
        };
        unsigned int nbar = 0;              // software grid barriers passed so far (FUSED)
        auto net_barrier = [&]() {          // all CTAs of this network: writes before it are visible after it (via L2)
            epi_bar_sync();                  // the CTA's writes happen-before thread 0's release (cumulative at gpu scope)
            if (tid == 0) {
                asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p.bar_ctr + net), "r"(1u) : "memory");
                const unsigned int target = (unsigned int)G * (nbar + 1u);
                while (ld_acquire_gpu_u32(p.bar_ctr + net) < target) {}
            }
            ++nbar;
            epi_bar_sync();
        };
        auto mb_geom = [&](int mb, long long& start, int& count) {
            start = p.b.mb_start + (long long)mb * batch;
            count = min(batch, p.b.mb_count - mb * batch);
        };
        auto tile_rows = [&](int mb, int tile, long long* dst) {      // the loss lane of a sample writes its row
            if (loss_lane) {
                long long start; int count;
                mb_geom(mb, start, count);
                const int local = tile * XT + hf * HT + s_row;
                long long row = -1;
                if (local < count) {
                    const long long k = start + local;
                    if (p.b.identity_stride > 0) row = k * p.b.identity_stride;
                    else row = p.b.perm ? (long long)p.b.perm[k] : (long long)x3_feistel((unsigned long long)k, (unsigned long long)p.b.total, p.b.perm_seed);
                }
                dst[hf * HT + s_row] = row;
            }
        };
        int step_t0 = 0;
        if (FUSED) step_t0 = p.adam_step[net];
        // FUSED: where this thread's parameter (the first of its slice chunk) lives inside the weight-tile image, or -1
        // (log_std, b2, b3, and b1 when it is not folded into W1): byte offset of the hi piece, stride between pieces
        int img_off = -1; uint32_t img_sub = 0;
        if (FUSED) {
            const int Sx = (L.size + G - 1) / G, px = (int)blockIdx.x * Sx + tid;
            if (tid < Sx && px < L.size) {
                if (px >= L.off_w1 && px < L.off_b1) { const int e = px - L.off_w1; img_off = (int)off128(e / O, e % O); img_sub = W_SUB; }
                else if (px >= L.off_b1 && px < L.off_w2) { if (ones_col) { img_off = (int)off128(px - L.off_b1, 63); img_sub = W_SUB; } }
                else if (px >= L.off_w2 && px < L.off_b2) { const int e = px - L.off_w2; img_off = (int)(W_X3 + off128(e >> 6, e & 63)); img_sub = W_SUB; }
                else if (px >= L.off_w3 && px < L.off_b3) { const int e = px - L.off_w3; img_off = (int)(2 * W_X3 + off128(e >> 6, e & 63)); img_sub = W3_SUB; }
            }
        }
        uint8_t* wimg = FUSED ? p.wimg + (size_t)net * W_IMG : nullptr;
        // per-thread partial sums of the loss warps over the tiles of one minibatch (reduced once per minibatch)
        float acc_st[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, acc_dls[AP], acc_db[AP];      // loss, ratio, kl, count, FOCOPS mask
#pragma unroll
        for (int a = 0; a < AP; ++a) { acc_dls[a] = 0.f; acc_db[a] = 0.f; }

        int rpar = 0, it = 0;
        if ((int)blockIdx.x < (min(batch, p.b.mb_count) + XT - 1) / XT) {     // rows + X of the first tile
            tile_rows(0, blockIdx.x, sRowBuf);
            half_bar_sync(hf);
            prefetch_x(sRowBuf);
        }
#pragma unroll 1
        for (int mb = 0; mb < n_mb; ++mb) {
            long long mb_start; int count;
            mb_geom(mb, mb_start, count);
            const int ntiles = (count + XT - 1) / XT;
            const float inv_b = 1.0f / (float)count;
            const bool have_tiles = (int)blockIdx.x < ntiles;
            if (FUSED && tid == NEPI - 1) {        // Adam bias corrections of this minibatch's step, off the critical path
                const AdamBias b = adam_bias(p.lr[net], step_t0 + mb + 1);
                sScal[8] = b.step_size;
                sScal[9] = b.bc2_sqrt;
            }
#pragma unroll 1
            for (int tile = blockIdx.x; tile < ntiles; tile += G, ++it) {
                const uint32_t par = (uint32_t)(it & 1);
                long long* sRow = sRowBuf + rpar * XT;
                long long* sRowNext = sRowBuf + (rpar ^ 1) * XT;
                const bool has_next = tile + G < ntiles;
                // ---- E0: X tile (prefetched registers -> bf16x3) ------------------------------------------------
                stamp(0);
                if (has_next) tile_rows(mb, tile + G, sRowNext);
                if (it > 0 && !(!FUSED && p.forward_only)) mbar_wait_a(hbar(DONE_C6), par ^ 1u);   // previous tile's dW1 / db1 read X and dZ1
                stamp(1);
                tc_fence_after();
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = xpre[8 * ph + i];
                    store8_x3(sX, ACT_SUB, xm, 32 * ph + xc, v);
                    announce(RDY_X0 + ph);
                }
                half_bar_sync(hf);                                         // next tile's row list is complete
                stamp(2);
                // loss warps: this tile's per-sample inputs (used in E3) fly under the forward phases -- asynchronously into
                // shared memory when they fit (AP == 8), so that no register has to wait for them
                float pf_act[AP], pf_logp = 0.f, pf_advr = 0.f, pf_advc = 0.f, pf_tv = 0.f;
                long long prow = -1;
                if (loss_warp) {
                    if (loss_lane) prow = sRow[hf * HT + s_row];
#pragma unroll
                    for (int a = 0; a < AP; ++a) pf_act[a] = 0.f;
                    if (prow >= 0) {
                        const float* asrc = (p.kind == X3_FVP) ? p.fvp_dmu : p.b.act;
                        if (AP == 8) {
                            const uint32_t dst = sbase + OFF_PF + (uint32_t)((hf * HT + s_row) * PF_LD) * 4u;
                            auto cp4 = [&](uint32_t d, const float* src) {
                                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(src) : "memory");
                            };
                            if (net == 0) {
#pragma unroll
                                for (int a = 0; a < AP; ++a)
                                    if (a < A) cp4(dst + 4u * a, asrc + prow * A + a);
                                if (p.kind != X3_FVP) { cp4(dst + 32u, p.b.logp + prow); cp4(dst + 36u, p.b.adv_r + prow); cp4(dst + 40u, p.b.adv_c + prow); }
                            } else {
                                cp4(dst + 32u, (net == 1 ? p.b.tv_r : p.b.tv_c) + prow);
                            }
                        } else if (net == 0) {
#pragma unroll
                            for (int a = 0; a < AP; ++a)
                                if (a < A) pf_act[a] = __ldg(asrc + prow * A + a);
                            if (p.kind != X3_FVP) { pf_logp = __ldg(p.b.logp + prow); pf_advr = __ldg(p.b.adv_r + prow); pf_advc = __ldg(p.b.adv_c + prow); }
                        } else {
                            pf_tv = __ldg((net == 1 ? p.b.tv_r : p.b.tv_c) + prow);
                        }
                    }
                }
                // ---- E1: H1 = tanh(Z1 + b1) -------------------------------------------------------------------
                mbar_wait_a(hbar(DONE_C1), par);
                tc_fence_after();
                stamp(3);
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    const int c0 = 32 * ph + ccol;
                    float v[8];
                    tmem_ld8_m64(tHalf + T_ZA + (uint32_t)(32 * ph + 16 * h2), v);
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = tanh_acc(v[i] + sB1[c0 + i]);
                    store8_x3(sH1, ACT_SUB, s_row, c0, v);
                    announce(RDY_H1_0 + ph);
                }
                // ---- E2: H2 = tanh(Z2 + b2) -------------------------------------------------------------------
                stamp(4);
                mbar_wait_a(hbar(DONE_C2), par);
                tc_fence_after();
                stamp(5);
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    const int c0 = 32 * ph + ccol;
                    float v[8];
                    tmem_ld8_m64(tHalf + T_ZB + (uint32_t)(32 * ph + 16 * h2), v);
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = tanh_acc(v[i] + sB2[c0 + i]);
                    store8_x3(sH2, ACT_SUB, s_row, c0, v);
                    announce(RDY_H2_0 + ph);
                }
                stamp(6);
                // ---- E3: OUT -> loss -> dOUT (loss warps: one lane l < 16 per sample) --------------------------------
                if (loss_warp) {
                    if (AP == 8) {
                        asm volatile("cp.async.wait_all;\n" ::: "memory");
                        const float* pf = reinterpret_cast<const float*>(gbase + OFF_PF) + (hf * HT + s_row) * PF_LD;
                        if (prow >= 0) {
                            if (net == 0) {
#pragma unroll
                                for (int a = 0; a < AP; ++a)
                                    if (a < A) pf_act[a] = pf[a];
                                pf_logp = pf[8]; pf_advr = pf[9]; pf_advc = pf[10];
                            } else {
                                pf_tv = pf[8];
                            }
                        }
                    }
                    mbar_wait_a(hbar(DONE_C3), par);
                    tc_fence_after();
                    stamp(7);
                    float o[AP], d16[16];
#pragma unroll
                    for (int a = 0; a < 16; ++a) d16[a] = 0.f;
                    if (AP == 8) {
                        float t8[8];
                        tmem_ld8(tHalf + T_OUT, t8);
#pragma unroll
                        for (int a = 0; a < AP; ++a) o[a] = t8[a];
                    } else {
                        float t16[16];
                        tmem_ld16(tHalf + T_OUT, t16);
#pragma unroll
                        for (int a = 0; a < AP; ++a) o[a] = t16[a];
                    }
                    if (prow >= 0) {
                        if (net != 0) {
                            const float d = o[0] + sB3[0] - pf_tv;
                            acc_st[0] += d * d; acc_st[3] += 1.f;
                            d16[0] = 2.f * d * inv_b;
                            acc_db[0] += d16[0];
                        } else if (p.kind == X3_FVP) {
                            // J^T diag(sigma^-2) dmu / (B A): the supplied tangent is the output gradient
                            acc_st[3] += 1.f;
#pragma unroll
                            for (int a = 0; a < AP; ++a)
                                if (a < A) {
                                    const float dm = pf_act[a] * sLs[32 + a] * p.fvp_scale;
                                    d16[a] = dm;
                                    acc_db[a] += dm;
                                }
                        } else {
                            float logp_new = 0.f, diff[AP];
#pragma unroll
                            for (int a = 0; a < AP; ++a) {
                                diff[a] = 0.f;
                                if (a < A) {
                                    const float d = pf_act[a] - (o[a] + sB3[a]);
                                    diff[a] = d;
                                    logp_new += -(d * d) * (0.5f * sLs[32 + a]) - sLs[a] - 0.9189385332046727f;
                                }
                            }
                            const float ratio = expf(logp_new - pf_logp);
                            const float adv_r = (pf_advr - m_r) * inv_sr;
                            const float adv_c = pf_advc - m_c;
                            const float adv = (adv_r - lam * adv_c) * inv_1lam;
                            float dlogp, loss;
                            if (p.kind == X3_PPO_CLIP || (!FUSED && p.kind == X3_P3O)) {
                                const float rc = fminf(fmaxf(ratio, 1.f - p.clip), 1.f + p.clip);
                                const float s1 = ratio * adv, s2 = rc * adv;
                                loss = -fminf(s1, s2);
                                dlogp = (s1 <= s2) ? -adv * ratio * inv_b : 0.f;
                                if (!FUSED && p.kind == X3_P3O) {
                                    // P3O (penalty_function/p3o.py:L48-91): + kappa * relu(mean_j(ratio_j adv_c_j) + Jc - limit); the gate
                                    // (kappa when the minibatch mean makes the relu active) comes from the forward-only pass 1.
                                    // Statistic slot 2: pass 1 -> ratio * adv_c; pass 2 -> the penalty term (Loss/Loss_pi_cost).
                                    const bool pass2 = p.focops_mask_mean != nullptr;
                                    const float gate = pass2 ? __ldg(p.focops_mask_mean) : 0.f;
                                    dlogp += gate * adv_c * ratio * inv_b;
                                    acc_st[2] += pass2 ? gate * (ratio * adv_c + p.focops_eta) : ratio * adv_c;
                                }
                            } else if (p.kind == X3_RATIO) {
                                loss = -ratio * adv; dlogp = -adv * ratio * inv_b;
                            } else if (p.kind == X3_COST) {
                                loss = ratio * adv_c; dlogp = adv_c * ratio * inv_b;
                            }
                            float dmask = 0.f, dmo[AP];
#pragma unroll
                            for (int a = 0; a < AP; ++a) dmo[a] = 0.f;
                            if ((!FUSED && p.kind == X3_FOCOPS)) {
                                // The reference forms (kl[b,1] - ratio[b] adv[b] / lam) * mask[b,1] and takes the mean of the
                                // [b,b] matrix (first_order/focops.py:L85-89):  loss = mean_i(mask_i kl_i) - mean_i(mask_i)
                                // mean_j(ratio_j adv_j) / lam;  mean_i(mask_i) of this minibatch comes from the forward-only pass 1.
                                const float* sOld = misc + MF_OLD;
                                float kl = 0.f;
#pragma unroll
                                for (int a = 0; a < AP; ++a)
                                    if (a < A) {
                                        const float sn = sLs[16 + a];
                                        dmo[a] = (o[a] + sB3[a]) - __ldg(p.mu_old + prow * A + a);
                                        kl += (sOld[a] - sLs[a]) + (sn * sn + dmo[a] * dmo[a]) * (0.5f * sOld[16 + a]) - 0.5f;
                                    }
                                dmask = (kl <= p.focops_eta) ? 1.f : 0.f;
                                const float mbar = p.focops_mask_mean ? __ldg(p.focops_mask_mean) : dmask;
                                loss = kl * dmask - mbar * ratio * adv / p.focops_lam;
                                dlogp = -mbar * adv * ratio / p.focops_lam * inv_b;
                                acc_st[2] += kl; acc_st[4] += dmask;
                            }
                            acc_st[0] += loss; acc_st[1] += ratio; acc_st[3] += 1.f;
#pragma unroll
                            for (int a = 0; a < AP; ++a)
                                if (a < A) {
                                    const float iv = sLs[32 + a];
                                    float dm = dlogp * diff[a] * iv;
                                    float dl = dlogp * (diff[a] * diff[a] * iv - 1.f);
                                    if ((!FUSED && p.kind == X3_FOCOPS)) {
                                        const float sn = sLs[16 + a];
                                        dm += dmask * inv_b * dmo[a] * (misc + MF_OLD)[16 + a];
                                        dl += dmask * inv_b * (sn * sn * (misc + MF_OLD)[16 + a] - 1.f);
                                    }
                                    d16[a] = dm;
                                    acc_db[a] += dm;
                                    acc_dls[a] += dl;
                                }
                        }
                    }
                    if (lane < 16) store16_x3_sw32(sD, D_SUB, s_row, d16);
                    announce(RDY_D);
                    stamp(8);
                }
                stamp(9);
                if (!FUSED && p.forward_only) {                                      // statistics pass: no backward; H2 is free once OUT is done
                    if (has_next) prefetch_x(sRowNext);
                    if (!loss_warp) { mbar_wait_a(hbar(DONE_C3), par); tc_fence_after(); }
                    rpar ^= 1;
                    continue;
                }
                // ---- E4: dZ2 = (dOUT W3) (1 - H2^2), stored over H2 once dW3 has read it --------------------------
                if (has_next) prefetch_x(sRowNext);                        // next tile's rows fly during the backward half
                mbar_wait_a(hbar(DONE_C4A), par);
                tc_fence_after();
                stamp(10);
                float dz[16];
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    const int c0 = 32 * ph + ccol;
                    float v[8], hh[8];
                    tmem_ld8_m64(tHalf + T_ZA + (uint32_t)(32 * ph + 16 * h2), v);
                    load8_x3(sH2, ACT_SUB, s_row, c0, hh);
#pragma unroll
                    for (int i = 0; i < 8; ++i) dz[8 * ph + i] = v[i] * (1.f - hh[i] * hh[i]);
                }
                stamp(11);
                mbar_wait_a(hbar(DONE_C4B), par);
                stamp(12);
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = dz[8 * ph + i];
                    store8_x3(sH2, ACT_SUB, s_row, 32 * ph + ccol, v);
                    announce(RDY_DZ2_0 + ph);
                }
                // ---- E5: dZ1 = (dZ2 W2) (1 - H1^2), stored over H1 once dW2 has read it --------------------------
                stamp(13);
                mbar_wait_a(hbar(DONE_C5A), par);
                tc_fence_after();
                stamp(14);
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    const int c0 = 32 * ph + ccol;
                    float v[8], hh[8];
                    tmem_ld8_m64(tHalf + T_ZB + (uint32_t)(32 * ph + 16 * h2), v);
                    load8_x3(sH1, ACT_SUB, s_row, c0, hh);
#pragma unroll
                    for (int i = 0; i < 8; ++i) dz[8 * ph + i] = v[i] * (1.f - hh[i] * hh[i]);
                }
                stamp(15);
                mbar_wait_a(hbar(DONE_C5B), par);
                stamp(16);
#pragma unroll
                for (int ph = 0; ph < 2; ++ph) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = dz[8 * ph + i];
                    store8_x3(sH1, ACT_SUB, s_row, 32 * ph + ccol, v);
                }
                announce(RDY_DZ1);
                stamp(17);
                rpar ^= 1;
            }
            stamp(20);
            // ---- rows + X of the first tile of the NEXT minibatch: the gather flies under the optimiser phases ------
            if (FUSED && mb + 1 < n_mb) {
                long long s2; int c2;
                mb_geom(mb + 1, s2, c2);
                if ((int)blockIdx.x < (c2 + XT - 1) / XT) {
                    tile_rows(mb + 1, blockIdx.x, sRowBuf + rpar * XT);
                    half_bar_sync(hf);
                    prefetch_x(sRowBuf + rpar * XT);
                }
            }
            // ---- this CTA's partial gradient of the minibatch: TMEM accumulators -> global ------------------------
            if (have_tiles) {
                // Loss-lane partial sums, reduced exactly as with whole 128-sample tiles: each loss lane owns one tile row
                // (hf * 64 + s_row) across the tiles; the rows go through shared memory (the H2 buffers, idle once the last MMA
                // of the minibatch has completed) to threads 0-127, one row each, so warp q sums rows 32 q .. 32 q + 31
                // (butterfly), then the four warps in a fixed order.
                mbar_wait_a(bar(NHB + ((!FUSED && p.forward_only) ? DONE_C3 : DONE_C6)), (uint32_t)((it - 1) & 1));   // half b's last commit
                tc_fence_after();
                stamp(21);
                constexpr int RLD = 5 + 2 * AP;
                float* sLoss = reinterpret_cast<float*>(gbase + OFF_H2);
                if (loss_lane) {
                    float* r = sLoss + (hf * HT + s_row) * RLD;
#pragma unroll
                    for (int i = 0; i < 5; ++i) { r[i] = acc_st[i]; acc_st[i] = 0.f; }
#pragma unroll
                    for (int a = 0; a < AP; ++a) { r[5 + a] = acc_dls[a]; r[5 + AP + a] = acc_db[a]; acc_dls[a] = 0.f; acc_db[a] = 0.f; }
                }
                epi_bar_sync();
                if (tid < XT) {
                    const float* r = sLoss + tid * RLD;
#pragma unroll
                    for (int i = 0; i < 5; ++i) {
                        const float v = warp_sum(r[i]);
                        if (lane == 0) sRed[q * 8 + i] = v;
                    }
#pragma unroll
                    for (int a = 0; a < AP; ++a) {
                        const float dl = warp_sum(r[5 + a]), db = warp_sum(r[5 + AP + a]);
                        if (lane == 0) { sRed[32 + q * 16 + a] = dl; sRed[96 + q * 16 + a] = db; }
                    }
                }
                if (!FUSED && p.forward_only) {
                    epi_bar_sync();                    // sRed of the four reducing warps
                    if (tid >= 64 && tid < 72) {
                        const int i = tid - 64;
                        __stcg(p.stats_part + ((size_t)blockIdx.x * 3 + net) * 8 + i, (i < 5) ? (sRed[i] + sRed[8 + i]) + (sRed[16 + i] + sRed[24 + i]) : 0.f);
                    }
                    break;
                }
                const int t_row = 16 * q + lane;       // row (lane < 16) of the M = 64 accumulators
                const int c16 = 16 * h;
                float v[16];
                tmem_ld16(tmem + lane_base + T_DW2 + (uint32_t)c16, v);
                if (lane < 16) {
                    float* dst = gout + L.off_w2 + t_row * 64 + c16;
                    if (FUSED && (L.off_w2 & 3) == 0) {
#pragma unroll
                        for (int i = 0; i < 16; i += 4) __stcg(reinterpret_cast<float4*>(dst + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) __stcg(dst + i, v[i]);
                    }
                }
                tmem_ld16(tmem + lane_base + T_DW1 + (uint32_t)c16, v);
                if (lane < 16) {
                    float* dst = gout + L.off_w1 + t_row * O + c16;
                    if (FUSED && ((L.off_w1 | O) & 3) == 0) {
#pragma unroll
                        for (int i = 0; i < 16; i += 4)
                            if (c16 + i < O) __stcg(reinterpret_cast<float4*>(dst + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (c16 + i < O) __stcg(dst + i, v[i]);
                    }
                    if (ones_col && h == 3) __stcg(gout + L.off_b1 + t_row, v[15]);        // column 63 of dW1 = db1
                }
                if (h == 0) {      // dW3^T [k][o]
                    tmem_ld16(tmem + lane_base + T_DW3, v);
                    if (lane < 16)
#pragma unroll
                        for (int o = 0; o < 16; ++o)
                            if (o < L.out) __stcg(gout + L.off_w3 + o * 64 + t_row, v[o]);
                } else if (h == 1) {
                    if (!ones_col) {
                        tmem_ld16(tmem + lane_base + T_DB1, v);
                        if (lane < 16) __stcg(gout + L.off_b1 + t_row, v[0]);
                    }
                } else if (h == 2) {
                    tmem_ld16(tmem + lane_base + T_DB2, v);
                    if (lane < 16) __stcg(gout + L.off_b2 + t_row, v[0]);
                }
                tc_fence_before();
                epi_bar_sync();                        // sRed of the four reducing warps
                if (tid < L.out) __stcg(gout + L.off_b3 + tid, (sRed[96 + tid] + sRed[112 + tid]) + (sRed[128 + tid] + sRed[144 + tid]));
                if (net == 0 && tid >= 32 && tid < 32 + A) {
                    const int a = tid - 32;
                    float g = (sRed[32 + a] + sRed[48 + a]) + (sRed[64 + a] + sRed[80 + a]);
                    if (blockIdx.x == 0 && (p.kind == X3_PPO_CLIP || (!FUSED && (p.kind == X3_FOCOPS || p.kind == X3_P3O)))) g -= p.entropy_coef / (float)A;
                    if (p.kind == X3_FVP) g = (blockIdx.x == 0) ? 2.f / (float)A * __ldg(p.fvp_vec + L.off_logstd + a) : 0.f;
                    __stcg(gout + L.off_logstd + a, g);
                }
                if (tid >= 64 && tid < 72) {
                    const int i = tid - 64;
                    __stcg(p.stats_part + ((size_t)blockIdx.x * 3 + net) * 8 + i, (i < 5) ? (sRed[i] + sRed[8 + i]) + (sRed[16 + i] + sRed[24 + i]) : 0.f);
                }
            } else {
                for (int i = tid; i < L.size; i += NEPI) __stcg(gout + i, 0.f);      // no tile of this (short) minibatch
                if (tid < 8) __stcg(p.stats_part + ((size_t)blockIdx.x * 3 + net) * 8 + tid, 0.f);
            }
            stamp(22);
            if (!FUSED) break;

            // ================= in-kernel optimiser step =========================================================
            net_barrier();                                             // every partial gradient of this network is in L2
            stamp(23);
            const int S = (L.size + G - 1) / G;                        // parameters owned by this CTA: [p0, p0 + S)
            const int p0 = (int)blockIdx.x * S;
            const int Gh = (G + 1) >> 1;
            const float* gnet = p.gpart + (size_t)((gridDim.y == 1 ? 0 : net) * G) * PSTR;
            float ssq = 0.f, st2 = 0.f;
            for (int base = 0; base < S; base += 256) {
                const int pi = base + (tid & 255), part = tid >> 8;
                const bool valid = pi < S && p0 + pi < L.size;
                float sacc = 0.f;
                if (valid) {
                    const float* src = gnet + p0 + pi;
                    const int b1 = min(G, (part + 1) * Gh);
                    for (int b = part * Gh; b < b1; b += 32) {       // 32 partial rows in flight per thread
                        float t[32];
#pragma unroll
                        for (int u = 0; u < 32; ++u) t[u] = (b + u < b1) ? __ldcg(src + (size_t)(b + u) * PSTR) : 0.f;
#pragma unroll
                        for (int w = 16; w > 0; w >>= 1)
#pragma unroll
                            for (int u = 0; u < w; ++u) t[u] += t[u + w];
                        sacc += t[0];
                    }
                }
                sPart[tid] = sacc;
                epi_bar_sync();
                if (part == 0 && valid) {
                    const int qg = noff + p0 + pi;
                    float g = sPart[tid] + sPart[256 + tid];
                    if (net != 0 && p.critic_norm_coef > 0.f) {
                        const float th = __ldcg(p.theta_rw + qg);
                        g += 2.f * p.critic_norm_coef * th; st2 += th * th;
                    }
                    __stcg(p.grad + qg, g);
                    ssq += g * g;
                }
                epi_bar_sync();
            }
            ssq = warp_sum(ssq); st2 = warp_sum(st2);
            if (lane == 0) { sPart[warp] = ssq; sPart[16 + warp] = st2; }
            epi_bar_sync();
            if (tid == 0) {
                float a = 0.f, b = 0.f;
                for (int w = 0; w < 16; ++w) { a += sPart[w]; b += sPart[16 + w]; }
                __stcg(p.sumsq_part + (net * 2 + 0) * G + blockIdx.x, a);
                __stcg(p.sumsq_part + (net * 2 + 1) * G + blockIdx.x, b);
            }
            // Adam state of this thread's parameter: loaded before the barrier, consumed after it
            const bool own = tid < S && p0 + tid < L.size;
            float pre_th = 0.f, pre_m = 0.f, pre_v = 0.f;
            if (own) { pre_th = __ldcg(p.theta_rw + noff + p0 + tid); pre_m = __ldcg(p.adam_m + noff + p0 + tid); pre_v = __ldcg(p.adam_v + noff + p0 + tid); }
            // torch-Adam step of one parameter (+ its three bf16 pieces in the weight-tile image)
            auto adam_store = [&](int qg, float g, float th, float m, float v, bool img) {
                const float th_new = adam_update(g, th, m, v, {sScal[8], sScal[9]});
                __stcg(p.theta_rw + qg, th_new);
                __stcg(p.adam_m + qg, m); __stcg(p.adam_v + qg, v);
                if (img && img_off >= 0) {           // where the weight tiles expect them
                    uint32_t w0, w1, w2;
                    split2(th_new, 0.f, w0, w1, w2);
                    __stcg(reinterpret_cast<unsigned short*>(wimg + img_off), (unsigned short)w0);
                    __stcg(reinterpret_cast<unsigned short*>(wimg + img_off + img_sub), (unsigned short)w1);
                    __stcg(reinterpret_cast<unsigned short*>(wimg + img_off + 2 * img_sub), (unsigned short)w2);
                }
            };
            // One rank: clip_grad_norm_ almost never clips (max_grad_norm 40), so Adam runs SPECULATIVELY with coefficient 1
            // before the slice norms are known; the barrier that publishes the norms is then also the one that publishes the
            // new parameters, and only a step that does clip redoes Adam from the saved state (one more barrier).
            const bool spec = p.world == 1 && S <= NEPI;
            float g_raw = 0.f;
            if (spec && own) { g_raw = __ldcg(p.grad + noff + p0 + tid); adam_store(noff + p0 + tid, g_raw, pre_th, pre_m, pre_v, true); }
            stamp(24);
            net_barrier();                                             // every slice norm of this network is in L2
            stamp(25);
            if (warp == 0) {
                float tot = 0.f, t2 = 0.f;
                for (int b = lane; b < G; b += 32) { tot += __ldcg(p.sumsq_part + (net * 2 + 0) * G + b); t2 += __ldcg(p.sumsq_part + (net * 2 + 1) * G + b); }
                tot = warp_sum(tot); t2 = warp_sum(t2);
                if (lane == 0) {
                    sScal[0] = clip_coef(p.max_grad_norm, tot);
                    sScal[3] = t2;
                }
            } else if (warp == 1 && blockIdx.x == 0) {               // loss statistics of this minibatch (logger means)
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                for (int b = lane; b < G; b += 32)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[i] += __ldcg(p.stats_part + ((size_t)b * 3 + net) * 8 + i);
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i] = warp_sum(acc[i]);
                if (lane == 0) { sScal[4] = acc[0]; sScal[5] = acc[1]; sScal[6] = acc[2]; sScal[7] = acc[3]; }
            }
            epi_bar_sync();
            if (blockIdx.x == 0 && tid == 0)
                fold_train_stats(p.train_stats + net * 8, sScal + 4, net != 0, p.critic_norm_coef, sScal + 3);
            const float clipc = sScal[0];
            const unsigned int xstep = p.step_base + (unsigned int)mb;
            const int xpar = (int)(xstep & 1u);
            if (spec) {
                if (clipc != 1.0f) {                                   // (uniform over the network: same partial norms, same order)
                    if (own) {
                        const float g = g_raw * clipc;
                        __stcg(p.grad + noff + p0 + tid, g);
                        adam_store(noff + p0 + tid, g, pre_th, pre_m, pre_v, true);
                    }
                    stamp(26);
                    net_barrier();
                }
            } else {
                    // clip -> average over ranks -> Adam (policy_gradient.py:L437-443, distributed.py:L193-198).  world > 1: every
            // parameter of the slice travels as ONE 8-byte word {step tag, clipped gradient} stored straight into every peer's
            // receive buffer [parity][source rank][P] over NVLink; the receiver spins on the tag of each word -- data and
            // flag arrive together, so there is no fence, no flag round and no barrier in the exchange.
            for (int base = 0; base < S; base += NEPI) {
                const int pi = base + tid;
                if (pi < S && p0 + pi < L.size) {
                    const int qg = noff + p0 + pi;
                    float g = __ldcg(p.grad + qg) * clipc;
                    bool fail = false;
                    if (p.world > 1) {
                        const unsigned long long word = ((unsigned long long)xstep << 32) | (unsigned long long)__float_as_uint(g);
                        const size_t slot = ((size_t)(xpar * p.world + p.rank)) * p.P + qg;
                        for (int r = 0; r < p.world; ++r)
                            if (r != p.rank)
                                asm volatile("st.relaxed.sys.global.b64 [%0], %1;" ::"l"(reinterpret_cast<unsigned long long*>(p.peer_buf[r]) + slot), "l"(word) : "memory");
                        const unsigned long long* mine = reinterpret_cast<const unsigned long long*>(p.peer_buf[p.rank]);
                        float sum = 0.f;
                        const long long t0 = clock64();
                        for (int r = 0; r < p.world; ++r) {
                            float v = g;
                            if (r != p.rank) {
                                const unsigned long long* src = mine + ((size_t)(xpar * p.world + r)) * p.P + qg;
                                unsigned long long w64;
                                for (;;) {
                                    asm volatile("ld.relaxed.sys.global.b64 %0, [%1];" : "=l"(w64) : "l"(src) : "memory");
                                    if ((unsigned int)(w64 >> 32) == xstep) break;
                                    if (clock64() - t0 > 20000000000LL) { *p.error_flag = 1; fail = true; break; }   // ~10 s: fail loudly, never hang the GPU
                                }
                                v = __uint_as_float((unsigned int)w64);
                            }
                            sum += v;
                        }
                        g = sum / (float)p.world;
                    }
                    if (!fail) {
                        __stcg(p.grad + qg, g);
                        const bool pre = base == 0;                     // first chunk: state prefetched before the barrier
                        adam_store(qg, g, pre ? pre_th : __ldcg(p.theta_rw + qg), pre ? pre_m : __ldcg(p.adam_m + qg),
                                   pre ? pre_v : __ldcg(p.adam_v + qg), pre);
                    }
                }
            }
            stamp(26);
            net_barrier();                                             // the new parameters of this network are in L2
            }
            stamp(27);
            if (S <= NEPI) {
                // weights: ONE bulk copy (TMA) of the image the Adam owners just wrote; biases / log_std: a few scalar loads
                if (tid == 0) {
                    asm volatile("fence.proxy.async.global;\n" ::: "memory");       // generic-proxy writes (other SMs, acquired above) -> async-proxy read
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar(RDY_W)), "r"(W_IMG) : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                                 ::"r"(sbase + OFF_W1), "l"(wimg), "r"(W_IMG), "r"(bar(RDY_W)) : "memory");
                }
                if (tid >= 64 && tid < 128) { const int i = tid - 64; if (!ones_col) misc[MF_B1 + i] = __ldcg(theta + L.off_b1 + i); misc[MF_B2 + i] = __ldcg(theta + L.off_b2 + i); }
                if (tid >= 128 && tid < 144) {
                    const int i = tid - 128;
                    misc[MF_B3 + i] = (i < L.out) ? __ldcg(theta + L.off_b3 + i) : 0.f;
                    const float ls = (net == 0 && i < A) ? __ldcg(theta + L.off_logstd + i) : 0.f;
                    const float sd = expf(ls);
                    misc[MF_LS + i] = ls; misc[MF_LS + 16 + i] = sd; misc[MF_LS + 32 + i] = 1.f / (sd * sd);
                }
                mbar_wait_a(bar(RDY_W), (uint32_t)(mb & 1));
            } else {
                stage_weights_x3(sbase, misc, theta, L, net, O, A, tid);   // slices longer than the block: the image is incomplete
            }
            epi_bar_sync();
            stamp(28);
        }
        if (FUSED && blockIdx.x == 0 && tid == 0) p.adam_step[net] = step_t0 + n_mb;     // every CTA read it before the first barrier
    }
    tc_fence_before();
    __syncthreads();
    if (is_mma_warp) tmem_dealloc(tmem, T_COLS);
}

// mean_i 1{KL_i <= eta} of a minibatch from the forward-only pass (statistic slot 4 / slot 3 of the actor rows)
__global__ void x3_mask_mean_kernel(const float* __restrict__ stats_part, int nblocks, float* __restrict__ out,
                                    const int* __restrict__ stop_flag, int kind, float kappa, float jc_minus_limit) {
    if (threadIdx.x != 0 || (stop_flag && *stop_flag)) return;
    const int slot = (kind == X3_P3O) ? 2 : 4;
    float m = 0.f, n = 0.f;
    for (int b = 0; b < nblocks; ++b) { m += stats_part[((size_t)b * 3) * 8 + slot]; n += stats_part[((size_t)b * 3) * 8 + 3]; }
    const float mean = n > 0.f ? m / n : 0.f;
    out[0] = (kind == X3_P3O) ? ((mean + jc_minus_limit > 0.f) ? kappa : 0.f) : mean;
}

}  // namespace osb

using namespace osb;

extern "C" {

static long long* g_x3_dbg = nullptr;
// development aid: clock64 stamps of CTA (0, 0) of the next launches go to buf (2048 long long), NULL turns it off
int osb_x3_debug_buffer(long long* buf) { g_x3_dbg = buf; return OSB_OK; }

static int x3_set_attr() {
    static bool attr = false;
    if (!attr) {
        const size_t smem = 1024 + X3_SMEM;
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_x3_kernel<false, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_x3_kernel<false, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_x3_kernel<true, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_x3_kernel<true, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    return OSB_OK;
}

// Split-bf16 (parity-grade tensor-core) variant of osb_minibatch_grad: same arguments, O <= 64, A <= 16,
// loss kinds PPO-clip / ratio / cost surrogate.  gpart holds osb_tc_grid_blocks(mb_count, net_mask) rows of P floats.
int osb_minibatch_grad_x3(const float* theta, int O, int A, const float* obs, const float* act,
                          const float* logp, const float* adv_r, const float* adv_c,
                          const float* tv_r, const float* tv_c, const float* mu_old,
                          const float* moments, const int* perm, long long total, unsigned perm_seed,
                          long long mb_start, int mb_count, int loss_kind, float clip,
                          float entropy_coef, float focops_lam, float focops_eta,
                          const float* lagrange, const float* logstd_old, int net_mask, float* gpart,
                          float* stats_part, const int* stop_flag, void* stream) {
    OSB_CHECK_ARG(theta && obs && act && logp && adv_r && adv_c && tv_r && tv_c && moments, "null input");
    OSB_CHECK_ARG(O > 0 && O <= 64 && A > 0 && A <= 16 && mb_count > 0 && total > 0, "bf16x3 path needs O <= 64, A <= 16");
    OSB_CHECK_ARG(mb_start >= 0 && mb_start + mb_count <= total, "minibatch window out of range");
    OSB_CHECK_ARG(loss_kind == X3_PPO_CLIP || loss_kind == X3_RATIO || loss_kind == X3_COST || loss_kind == X3_FOCOPS || loss_kind == X3_P3O, "loss kind not on the bf16x3 path");
    OSB_CHECK_ARG(loss_kind != X3_FOCOPS || (mu_old && logstd_old), "FOCOPS needs mu_old / logstd_old");
    OSB_CHECK_ARG(net_mask > 0 && net_mask < 8, "net_mask");
    X3Args p = {};
    p.b = X3Batch{obs, act, logp, adv_r, adv_c, tv_r, tv_c, moments, perm, total, perm_seed, mb_start, mb_count, 0};
    p.mu_old = mu_old; p.logstd_old = logstd_old; p.focops_lam = focops_lam; p.focops_eta = focops_eta;
    p.kind = loss_kind; p.clip = clip; p.entropy_coef = entropy_coef; p.lagrange = lagrange;
    p.theta = theta; p.gpart = gpart; p.stats_part = stats_part; p.stop_flag = stop_flag;
    p.O = O; p.A = A; p.P = actor_layout(O, A).size + 2 * critic_layout(O, A).size; p.net_mask = net_mask;
    p.batch_size = mb_count; p.world = 1; p.dbg = g_x3_dbg;
    const int nb = osb_tc_grid_blocks(mb_count, net_mask);
    int rc = x3_set_attr();
    if (rc) return rc;
    const bool single = (net_mask & (net_mask - 1)) == 0;
    if ((loss_kind == X3_FOCOPS || loss_kind == X3_P3O) && (net_mask & 1)) {
        // pass 1: actor forward only -> mean of the KL mask over the minibatch (FOCOPS: the reference's [b,1] x [b] broadcast) or
        // the relu gate of the minibatch-mean cost surrogate (P3O: focops_lam carries kappa, focops_eta carries Jc - limit)
        static float* d_mask_mean = nullptr;
        if (!d_mask_mean) OSB_CUDA(cudaMalloc(&d_mask_mean, sizeof(float)));
        X3Args q = p;
        q.forward_only = 1; q.net_mask = 1;
        const int nb1 = osb_tc_grid_blocks(mb_count, 1);
        if (A <= 8) minibatch_grad_x3_kernel<false, 8><<<dim3(nb1, 1), NTX3, 1024 + X3_SMEM, (cudaStream_t)stream>>>(q);
        else minibatch_grad_x3_kernel<false, 16><<<dim3(nb1, 1), NTX3, 1024 + X3_SMEM, (cudaStream_t)stream>>>(q);
        OSB_LAUNCH_CHECK();
        x3_mask_mean_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(stats_part, nb1, d_mask_mean, stop_flag, loss_kind, focops_lam, focops_eta);
        OSB_LAUNCH_CHECK();
        p.focops_mask_mean = d_mask_mean;
    }
    if (A <= 8) minibatch_grad_x3_kernel<false, 8><<<dim3(nb, single ? 1 : 3), NTX3, 1024 + X3_SMEM, (cudaStream_t)stream>>>(p);
    else minibatch_grad_x3_kernel<false, 16><<<dim3(nb, single ? 1 : 3), NTX3, 1024 + X3_SMEM, (cudaStream_t)stream>>>(p);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

// backward half of the bf16x3 Fisher-vector product (called by osb_fvp_partials_x3, csrc/fvp_x3.cu)
int osb_x3_fvp_backward(const float* theta_actor, const float* vec, int O, int A, const float* obs, long long total, int stride,
                        const float* dmu, float* gpart, float* stats_scratch, void* stream) {
    const long long nrows = (total + stride - 1) / stride;
    X3Args p = {};
    p.b = X3Batch{obs, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, total, 0u, 0, (int)nrows, stride};
    p.kind = X3_FVP; p.theta = theta_actor; p.gpart = gpart; p.stats_part = stats_scratch;
    p.O = O; p.A = A; p.P = actor_layout(O, A).size; p.net_mask = 1;
    p.batch_size = (int)nrows; p.world = 1; p.dbg = nullptr;
    p.fvp_dmu = dmu; p.fvp_vec = vec; p.fvp_scale = 1.0f / ((float)nrows * (float)A);
    const int nb = osb_tc_grid_blocks(nrows, 1);
    int rc = x3_set_attr();
    if (rc) return rc;
    if (A <= 8) minibatch_grad_x3_kernel<false, 8><<<dim3(nb, 1), NTX3, 1024 + X3_SMEM, (cudaStream_t)stream>>>(p);
    else minibatch_grad_x3_kernel<false, 16><<<dim3(nb, 1), NTX3, 1024 + X3_SMEM, (cudaStream_t)stream>>>(p);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

// One update iteration of PolicyGradient._update (policy_gradient.py:L369-381) as ONE persistent cooperative
// kernel on bf16x3 tiles: all minibatches of [0, total) in steps of batch_size, each = fused forward + loss +
// backward, fixed-order partial reduction, per-network clip_grad_norm_, (world > 1: clipped-gradient exchange
// over NVLink peer memory, policy_gradient.py:L437-443 / distributed.py:L193-198) and torch-Adam, with the
// parameters re-staged in shared memory between minibatches.  perm: [total] slab rows of this iteration or NULL
// (Feistel order keyed by perm_seed).  gpart: osb_tc_grid_blocks(batch_size, net_mask) rows of P floats.
// peer_buf / peer_flag: device arrays of `world` pointers ([2][world][P] floats, [2*world + 2*world*160] flags)
// or NULL for one rank.
int osb_ppo_update_iter_x3(float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step, int O, int A,
                           const float* obs, const float* act, const float* logp, const float* adv_r,
                           const float* adv_c, const float* tv_r, const float* tv_c, const float* moments,
                           const int* perm, long long total, unsigned perm_seed, int batch_size, int loss_kind,
                           float clip, float entropy_coef, const float* lagrange, int net_mask,
                           float critic_norm_coef, float max_grad_norm, float lr_actor, float lr_critic_r,
                           float lr_critic_c, float* gpart, float* stats_part, float* train_stats,
                           const int* stop_flag, void* peer_buf, void* peer_flag, int world, int rank,
                           int* p2p_error, void* stream) {
    OSB_CHECK_ARG(theta && grad && adam_m && adam_v && adam_step && obs && act && logp && adv_r && adv_c && tv_r && tv_c && moments, "null input");
    OSB_CHECK_ARG(O > 0 && O <= 64 && A > 0 && A <= 16 && batch_size > 0 && total > 0 && total < (1ll << 31), "bf16x3 path needs O <= 64, A <= 16");
    OSB_CHECK_ARG(loss_kind == X3_PPO_CLIP || loss_kind == X3_RATIO || loss_kind == X3_COST, "loss kind not on the bf16x3 path");
    OSB_CHECK_ARG(net_mask > 0 && net_mask < 8 && gpart && stats_part && train_stats, "bad argument");
    OSB_CHECK_ARG(world >= 1 && (world == 1 || (peer_buf && peer_flag && p2p_error && rank >= 0 && rank < world && world <= 64)), "bad p2p argument");
    static float* d_ws = nullptr;            // [0, 4): barrier counters (u32); [64, 64 + 6 * 148): slice norms
    static unsigned int step_base = 0;       // identical on every rank: same call sequence
    cudaStream_t s = (cudaStream_t)stream;
    if (!d_ws) OSB_CUDA(cudaMalloc(&d_ws, (64 + 6 * 148) * sizeof(float)));
    OSB_CUDA(cudaMemsetAsync(d_ws, 0, 4 * sizeof(unsigned int), s));
    X3Args p = {};
    p.b = X3Batch{obs, act, logp, adv_r, adv_c, tv_r, tv_c, moments, perm, total, perm_seed, 0, (int)total, 0};
    p.kind = loss_kind; p.clip = clip; p.entropy_coef = entropy_coef; p.lagrange = lagrange;
    p.theta = theta; p.gpart = gpart; p.stats_part = stats_part; p.stop_flag = stop_flag;
    p.O = O; p.A = A; p.P = actor_layout(O, A).size + 2 * critic_layout(O, A).size; p.net_mask = net_mask;
    p.batch_size = batch_size; p.theta_rw = theta; p.grad = grad; p.adam_m = adam_m; p.adam_v = adam_v; p.adam_step = adam_step;
    p.critic_norm_coef = critic_norm_coef; p.max_grad_norm = max_grad_norm;
    p.lr[0] = lr_actor; p.lr[1] = lr_critic_r; p.lr[2] = lr_critic_c;
    p.sumsq_part = d_ws + 64; p.train_stats = train_stats; p.bar_ctr = reinterpret_cast<unsigned int*>(d_ws);
    p.peer_buf = (float* const*)peer_buf; p.peer_flag = (unsigned int* const*)peer_flag;
    p.world = world; p.rank = rank; p.error_flag = p2p_error; p.dbg = g_x3_dbg;
    {   // weight-tile images: padding positions stay zero, so a change of the layout clears them
        static uint8_t* d_wimg = nullptr;
        static int img_O = -1, img_A = -1;
        if (!d_wimg) OSB_CUDA(cudaMalloc(&d_wimg, 3 * W_IMG));
        if (img_O != O || img_A != A) { OSB_CUDA(cudaMemsetAsync(d_wimg, 0, 3 * W_IMG, s)); img_O = O; img_A = A; }
        p.wimg = d_wimg;
    }
    const int n_mb = (int)((total + batch_size - 1) / batch_size);
    p.step_base = step_base + 1u;
    step_base += (unsigned int)n_mb;
    const int first = (int)(total < batch_size ? total : batch_size);
    const int nb = osb_tc_grid_blocks(first, net_mask);
    int rc = x3_set_attr();
    if (rc) return rc;
    const bool single = (net_mask & (net_mask - 1)) == 0;
    void* args[] = {&p};
    osb_count_launch();
    OSB_CUDA(cudaLaunchCooperativeKernel(A <= 8 ? (void*)minibatch_grad_x3_kernel<true, 8> : (void*)minibatch_grad_x3_kernel<true, 16>,
                                         dim3(nb, single ? 1 : 3), dim3(NTX3), args, 1024 + X3_SMEM, s));
    return OSB_OK;
}

}  // extern "C"
