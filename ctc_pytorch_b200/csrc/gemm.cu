// K1 — dense "TN" GEMM on the 5th-generation tensor cores:  C[M,N] (+)= A[M,K] * B[N,K]^T
// with A and B bf16, K contiguous (K-major), fp32 accumulation in TMEM, fp32 or bf16 output.
//
// This one kernel carries every dense contraction of the acoustic model that is not inside the
// time recurrence (the reference reaches them through nn.LSTM / nn.Linear library calls,
// timit/models/model_ctc.py:23-26,33,136-139,165-166):
//   gate pre-activations   Gx[T*N, 8H]  = X[T*N, I]       * Wih_packed[8H, I]^T
//   input gradient         dX[T*N, I]   = dG[T*N, 8H]     * WihT_packed[I, 8H]^T
//   weight gradients       dWih[8H, I]  = dG^T[8H, T*N]   * X^T[I, T*N]^T        (K = T*N)
//                          dWhh[4H, H]  = dG^T[4H, T*N]   * Hprev^T[H, T*N]^T    (K = T*N, shifted)
//   output layer           logits, dXfc, dWfc likewise.
//
// Structure (one CTA per SM, persistent over 128 x BN output tiles):
//   warp 0    TMA producer: cp.async.bulk.tensor 2-D boxes (128 x 64 of A, BN x 64 of B) into a
//             STAGES-deep SWIZZLE_128B shared-memory ring, completion on mbarriers.
//   warp 1    one elected thread issues tcgen05.mma (M=128, N=BN, K=16) from shared-memory
//             descriptors into one of two TMEM accumulator buffers; tcgen05.commit releases ring
//             slots back to the producer and hands finished accumulators to the epilogue.
//   warp 2    TMEM allocation / deallocation (2*BN columns).
//   warps 4-7 epilogue: tcgen05.ld 32 lanes x 32 columns per warp, convert, store to global; the
//             second accumulator buffer lets the next tile's MMAs run under the stores.
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"
#include "ctcb200.h"

namespace ctcb200 {
namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle row

template <int BN>
struct GemmCfg {
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = (BN == 256) ? 4 : (BN == 128 ? 6 : 8);
    static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
    static constexpr int STAGING_BYTES = 4 * 2 * 4096;  // per epilogue warp: two 32x32 fp32 boxes for the TMA store
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + 256 + 1024;  // + barriers + alignment
};

template <int BN>
__global__ void __launch_bounds__(256, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, void* __restrict__ Cout, long long ldc, int M, int N, int K,
               int a_koff, int b_koff, int out_bf16, int accumulate, int tma_store, int split_k, int mn_major,
               unsigned int* __restrict__ split_turn, unsigned int ticket_base) {
    using Cfg = GemmCfg<BN>;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* staging = smem + STAGES * Cfg::STAGE_BYTES;  // 1024-byte aligned (stage sizes are multiples of 1024)
    uint64_t* full = reinterpret_cast<uint64_t*>(staging + Cfg::STAGING_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tiles = (M + BM - 1) / BM, n_tiles = (N + BN - 1) / BN;
    const int out_tiles = m_tiles * n_tiles;
    const int tiles = out_tiles * split_k;  // work items: (output tile, K split); splits add into C through the TMA unit
    const int kblocks_total = (K + BK - 1) / BK;
    const int kb_per_split = (kblocks_total + split_k - 1) / split_k;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if (tma_store) tma_prefetch_desc(&tmC);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], 4);
        }
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    // split_k > 1: every CTA owns one work item, handed out in the order the CTAs start (a ticket counter in
    // split_turn[0] that keeps counting across the launches of a stream; ticket_base is where this launch began).
    // A split then only ever waits for splits whose CTAs are already running, whatever order blocks are dispatched in.
    uint32_t* first_tile = tmem_slot + 1;
    if (threadIdx.x == 0) *first_tile = split_k > 1 ? atomicAdd(split_turn, 1u) - ticket_base : blockIdx.x;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int tile0 = static_cast<int>(*first_tile);

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = tile0; tile < tiles; tile += gridDim.x) {
                const int ot = tile % out_tiles, sp = tile / out_tiles;
                const int m_blk = ot % m_tiles, n_blk = ot / m_tiles;
                const int kb0 = sp * kb_per_split, kb1 = min(kblocks_total, kb0 + kb_per_split);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], Cfg::STAGE_BYTES);
                    uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                    if (mn_major) {
                        // operands stored [K rows, M (N) columns]: boxes of 64 K rows x 64 columns (8 KB, SWIZZLE_128B), one per
                        // 64-wide column group of the tile; the K offsets are ROW coordinates here (no alignment constraint)
#pragma unroll
                        for (int g = 0; g < BM / 64; ++g)
                            tma_load_2d(sa + g * 8192, &tmA, &full[stage], m_blk * BM + g * 64, a_koff + kb * BK);
#pragma unroll
                        for (int g = 0; g < BN / 64; ++g)
                            tma_load_2d(sa + Cfg::A_BYTES + g * 8192, &tmB, &full[stage], n_blk * BN + g * 64, b_koff + kb * BK);
                    } else {
                        tma_load_2d(sa, &tmA, &full[stage], a_koff + kb * BK, m_blk * BM);
                        tma_load_2d(sa + Cfg::A_BYTES, &tmB, &full[stage], b_koff + kb * BK, n_blk * BN);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // the whole warp runs the (warp-uniform) pipeline bookkeeping so descriptors stay in uniform registers;
        // one elected lane issues the tcgen05 instructions
        constexpr uint32_t idesc_k = umma_idesc_bf16(BM, BN);
        // MN-major operands (both): bits 15 / 16 of the instruction descriptor select the transposed shared-memory layout
        const uint32_t idesc = mn_major ? (idesc_k | (1u << 15) | (1u << 16)) : idesc_k;
        const bool leader = elect_one();
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        for (int tile = tile0; tile < tiles; tile += gridDim.x, ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait(&tempty[acc], acc_phase ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + acc * BN;
            const int sp = tile / out_tiles;
            const int kb0 = sp * kb_per_split, kb1 = min(kblocks_total, kb0 + kb_per_split);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
                // K-major: a K=16 slice is 32 bytes along a 128-byte row; MN-major: 16 K rows = two 8-row groups of 1 KB
                const uint64_t ad = mn_major ? umma_desc_mn_sw128(a_addr) : umma_desc_sw128(a_addr);
                const uint64_t bd = mn_major ? umma_desc_mn_sw128(a_addr + Cfg::A_BYTES) : umma_desc_sw128(a_addr + Cfg::A_BYTES);
                const uint64_t ks = mn_major ? (2048 >> 4) : 2;
                if (leader) {
                    umma_bf16(d_tmem, ad, bd, idesc, kb != kb0 ? 1u : 0u);
                    umma_bf16(d_tmem, ad + ks, bd + ks, idesc, 1u);
                    umma_bf16(d_tmem, ad + 2 * ks, bd + 2 * ks, idesc, 1u);
                    umma_bf16(d_tmem, ad + 3 * ks, bd + 3 * ks, idesc, 1u);
                    umma_commit(&empty[stage]);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (leader) umma_commit(&tfull[acc]);
            __syncwarp();
        }
    } else if (warp >= 4) {
        const int ew = warp - 4;
        int it = 0;
        float* Cf = reinterpret_cast<float*>(Cout);
        __nv_bfloat16* Cb = reinterpret_cast<__nv_bfloat16*>(Cout);
        const bool vec_f32 = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(Cout) & 15) == 0);
        const bool vec_b16 = (ldc % 8 == 0) && ((reinterpret_cast<uintptr_t>(Cout) & 15) == 0);
        for (int tile = tile0; tile < tiles; tile += gridDim.x, ++it) {
            const int ot = tile % out_tiles;
            const int m_blk = ot % m_tiles, n_blk = ot / m_tiles;
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const int row = m_blk * BM + ew * 32 + lane;
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BN;
            if (tma_store) {
                // registers -> 128B-swizzled shared box -> TMA store: full 128-byte lines leave the SM, bounds are
                // clipped by the hardware; two boxes per warp so the next tcgen05.ld overlaps the previous store
                uint8_t* wbuf = staging + ew * 8192;
                const int sp = tile / out_tiles;
                const bool has_work = sp * kb_per_split < kblocks_total;  // an empty K split contributes nothing
                // K splits add their partial tiles into C one after another in split order (a turn counter per output
                // tile and epilogue warp), so the float sums, and with them the result, are the same on every run.
                // Split sp waits only for splits that took lower tickets, i.e. CTAs that are already running.
                unsigned int* turn = split_k > 1 ? split_turn + 1 + ot * 4 + ew : nullptr;
                if (turn) {
                    if (lane == 0) {
                        while (ld_acquire(turn) != static_cast<unsigned int>(sp)) {
                        }
                        fence_proxy_async_all();
                    }
                    __syncwarp();
                }
#pragma unroll 1
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    const int col0 = n_blk * BN + c0;
                    if (col0 >= N || !has_work) break;
                    uint32_t r[32];
                    tmem_ld_32x32(t_row + c0, r);
                    tmem_ld_wait();
                    uint8_t* box = wbuf + ((c0 >> 5) & 1) * 4096;
                    if (lane == 0) bulk_group_wait_read<1>();  // the store issued two chunks ago has left this box
                    __syncwarp();
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<uint4*>(box + lane * 128 + ((q ^ (lane & 7)) << 4)) =
                            make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (split_k > 1 || accumulate) tma_reduce_add_2d(&tmC, box, col0, m_blk * BM + ew * 32);
                        else tma_store_2d(&tmC, box, col0, m_blk * BM + ew * 32);
                        bulk_group_commit();
                    }
                }
                if (turn && lane == 0) {   // this split's additions are complete in global memory: pass the turn on
                    bulk_group_wait_all();
                    fence_proxy_async_all();
                    if (sp == split_k - 1) *turn = 0u;   // the last split leaves the counter zeroed for the next launch
                    else red_release_add(turn, 1u);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[acc]);
                continue;
            }
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(t_row + c0, r);
                tmem_ld_wait();
                const int col0 = n_blk * BN + c0;
                if (row < M && col0 < N) {
                    const bool fullchunk = col0 + 32 <= N;
                    if (!out_bf16) {
                        float* dst = Cf + static_cast<long long>(row) * ldc + col0;
                        if (fullchunk && vec_f32) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                float4 v = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]),
                                                       __uint_as_float(r[4 * q + 2]), __uint_as_float(r[4 * q + 3]));
                                float4* p = reinterpret_cast<float4*>(dst) + q;
                                if (accumulate) {
                                    float4 o = *p;
                                    v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                                }
                                *p = v;
                            }
                        } else {
#pragma unroll
                            for (int q = 0; q < 32; ++q) {
                                if (col0 + q < N) {
                                    float v = __uint_as_float(r[q]);
                                    if (accumulate) v += dst[q];
                                    dst[q] = v;
                                }
                            }
                        }
                    } else {
                        __nv_bfloat16* dst = Cb + static_cast<long long>(row) * ldc + col0;
                        if (fullchunk && vec_b16) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                uint32_t w[4];
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(r[8 * q + 2 * e]),
                                                                             __uint_as_float(r[8 * q + 2 * e + 1]));
                                    w[e] = *reinterpret_cast<uint32_t*>(&h);
                                }
                                reinterpret_cast<uint4*>(dst)[q] = make_uint4(w[0], w[1], w[2], w[3]);
                            }
                        } else {
#pragma unroll
                            for (int q = 0; q < 32; ++q)
                                if (col0 + q < N) dst[q] = __float2bfloat16(__uint_as_float(r[q]));
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
        if (tma_store && lane == 0) bulk_group_wait_all();  // all stores of this warp are complete before the CTA exits
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// First use of a tile width on a device: opt in to its shared memory AND make sure the kernel is loaded. CUDA loads kernels
// lazily, at their first launch, and that load may have to wait for everything running on the device: a GEMM whose first
// launch is a chunk of a streamed input projection (side stream, see ctcb200_lstm_fwd_streamed) would then wait for the
// recurrent kernel, which itself spins on that chunk — observed as a device-wait timeout in the very first step of a fresh
// process, whenever the capped launch picked a tile width the uncapped first chunk had not used. gemm_preload() therefore
// touches every tile width before a kernel that waits on GEMM output is launched (cudaFuncGetAttributes forces the load).
template <int BN>
int gemm_prepare() {
    static bool ready[MAX_DEVICES] = {false};   // function attributes and loaded modules are per device (context)
    const int dev = current_device();
    if (!ready[dev]) {
        CTCB_CUDA(cudaFuncSetAttribute(gemm_tn_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       GemmCfg<BN>::SMEM_BYTES));
        cudaFuncAttributes fa;
        CTCB_CUDA(cudaFuncGetAttributes(&fa, gemm_tn_kernel<BN>));
        ready[dev] = true;
    }
    return OK;
}

template <int BN>
int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, int tma_store, int split_k,
                void* C, long long ldc, int M, int N, int K, int a_koff, int b_koff, int out_bf16, int accumulate,
                int max_ctas, cudaStream_t stream, int mn_major, unsigned int* split_turn, unsigned int ticket_base) {
    using Cfg = GemmCfg<BN>;
    const int rc_attr = gemm_prepare<BN>();
    if (rc_attr != OK) return rc_attr;
    int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN) * split_k;
    // max_ctas: 0 = persistent over all SMs; > 0 = cap (leave SMs to a concurrent kernel); < 0 = one tile per CTA
    // (short-lived CTAs, so a kernel launched later on another stream gets SMs quickly)
    int limit = max_ctas > 0 ? max_ctas : device_sm_count();
    int grid = (max_ctas < 0 || tiles < limit) ? tiles : limit;
    CTCB_REQUIRE(split_k == 1 || grid == tiles, "gemm: a split-K launch needs one CTA per work item (%d tiles, grid %d)", tiles, grid);
    gemm_tn_kernel<BN><<<grid, 256, Cfg::SMEM_BYTES, stream>>>(tmA, tmB, tmC, C, ldc, M, N, K, a_koff, b_koff, out_bf16,
                                                              accumulate, tma_store, split_k, mn_major, split_turn,
                                                              ticket_base);
    CTCB_LAUNCH_CHECK();
    return OK;
}

}  // namespace

// Ordered split-K additions, one state per (device, stream): a buffer of 1 + device_sm_count() * 4 words (the ticket
// counter, then the turn counters: a split launch has at most sms / 2 output tiles, 4 epilogue warps each), zeroed once
// when the stream first runs a split launch, and the ticket count the stream's launches have taken so far. Every launch
// leaves its turn counters at zero, so the launches of one stream reuse the buffer; launches in different streams, which
// may run concurrently, never share one.
struct SplitState {
    unsigned int* buf = nullptr;
    unsigned int tickets = 0;
};
static std::mutex split_mu;
static std::map<std::pair<int, cudaStream_t>, SplitState> split_states;

static int split_state(cudaStream_t stream, SplitState** out) {
    std::lock_guard<std::mutex> lock(split_mu);
    SplitState& st = split_states[std::make_pair(current_device(), stream)];
    if (!st.buf) {
        const size_t bytes = (1 + static_cast<size_t>(device_sm_count()) * 4) * sizeof(unsigned int);
        CTCB_CUDA(cudaMalloc(reinterpret_cast<void**>(&st.buf), bytes));
        CTCB_CUDA(cudaMemsetAsync(st.buf, 0, bytes, stream));
    }
    *out = &st;
    return OK;
}

// Internal entry used by the other translation units as well as the C ABI below.
static int gemm_impl(const void* A, long long lda, const void* B, long long ldb, void* C, long long ldc, int M, int N,
                     int K, int a_koff, int b_koff, int out_bf16, int accumulate, int force_bn, int max_ctas,
                     cudaStream_t stream, int mn_major) {
    CTCB_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: empty problem M=%d N=%d K=%d", M, N, K);
    CTCB_REQUIRE(a_koff >= 0 && b_koff >= 0 && (mn_major || (a_koff % 8 == 0 && b_koff % 8 == 0)),
                 "gemm: K offsets (%d, %d) must be non-negative (multiples of 8 for K-major operands: TMA box start is 16-byte "
                 "aligned)", a_koff, b_koff);
    int bn = force_bn;
    // SMs this launch may use: a positive max_ctas leaves the rest of the device to a concurrent kernel
    const int sms = (max_ctas > 0 && max_ctas < device_sm_count()) ? max_ctas : device_sm_count();
    const int m_tiles = (M + BM - 1) / BM;
    if (bn == 0) {
        // waves x measured relative cost of one tile (B200: 256-wide tiles run the tensor pipe ~65 % busy, 128-wide
        // ones are shared-memory bound at ~0.62 of that per tile, 64-wide ~0.45): pick the cheapest estimate
        const struct { int bn; double cost; } cand[3] = {{256, 1.0}, {128, 0.62}, {64, 0.45}};
        double best = 1e30;
        for (const auto& c : cand) {
            if (c.bn > 64 && N <= c.bn / 2) continue;  // more than half of the tile would be padding
            const long long t = static_cast<long long>(m_tiles) * ((N + c.bn - 1) / c.bn);
            const double est = static_cast<double>((t + sms - 1) / sms) * c.cost;
            if (est < best - 1e-9) { best = est; bn = c.bn; }
        }
    }
    CTCB_REQUIRE(bn == 64 || bn == 128 || bn == 256, "gemm: tile width %d not in {64,128,256}", bn);
    CUtensorMap tmA, tmB;
    int rc;
    if (mn_major) {   // operands stored [K rows, M (N) columns]; out-of-range rows / columns of a box read as zero
        rc = make_tmap_bf16_2d(&tmA, A, static_cast<uint64_t>(a_koff) + K, M, lda, BK, 64);
        if (rc != OK) return rc;
        rc = make_tmap_bf16_2d(&tmB, B, static_cast<uint64_t>(b_koff) + K, N, ldb, BK, 64);
    } else {
        rc = make_tmap_bf16_2d(&tmA, A, M, static_cast<uint64_t>(a_koff) + K, lda, BM, BK);
        if (rc != OK) return rc;
        rc = make_tmap_bf16_2d(&tmB, B, N, static_cast<uint64_t>(b_koff) + K, ldb, bn, BK);
    }
    if (rc != OK) return rc;
    // fp32 results leave through TMA stores when the row pitch allows a tensor map (16-byte multiples)
    CUtensorMap tmC = tmA;
    int tma_store = 0;
    static const bool allow_tma_store = getenv("CTCB200_GEMM_EPILOGUE") == nullptr || getenv("CTCB200_GEMM_EPILOGUE")[0] != 'd';
    // accumulate = 1 rides the same path: the tile is ADDED to C by the TMA unit (cp.reduce.async.bulk ... .add)
    if (allow_tma_store && !out_bf16 && ldc % 4 == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0) {
        rc = make_tmap_f32_2d(&tmC, C, M, N, ldc, 32, 32);
        if (rc != OK) return rc;
        tma_store = 1;
    }
    // split K when the output has too few tiles to fill the machine and K is long (weight gradients: K = T*N);
    // partial tiles are added into a zeroed C by the TMA unit
    int split_k = 1;
    if (tma_store && max_ctas >= 0 && ldc == N) {
        const long long t = static_cast<long long>(m_tiles) * ((N + bn - 1) / bn);
        const int kblocks = (K + BK - 1) / BK;
        while (split_k < 8 && t * (split_k * 2) <= sms && kblocks / (split_k * 2) >= 16) split_k *= 2;
        if (split_k > 1 && !accumulate) CTCB_CUDA(cudaMemsetAsync(C, 0, static_cast<size_t>(M) * ldc * sizeof(float), stream));
    }
    SplitState* st = nullptr;
    if (split_k > 1) {
        rc = split_state(stream, &st);
        if (rc != OK) return rc;
    }
    unsigned int* split_turn = st ? st->buf : nullptr;
    const unsigned int base = st ? st->tickets : 0u;
    switch (bn) {
        case 64: rc = launch_gemm<64>(tmA, tmB, tmC, tma_store, split_k, C, ldc, M, N, K, a_koff, b_koff, out_bf16, accumulate, max_ctas, stream, mn_major, split_turn, base); break;
        case 128: rc = launch_gemm<128>(tmA, tmB, tmC, tma_store, split_k, C, ldc, M, N, K, a_koff, b_koff, out_bf16, accumulate, max_ctas, stream, mn_major, split_turn, base); break;
        default: rc = launch_gemm<256>(tmA, tmB, tmC, tma_store, split_k, C, ldc, M, N, K, a_koff, b_koff, out_bf16, accumulate, max_ctas, stream, mn_major, split_turn, base); break;
    }
    if (rc == OK && st) {   // the launch's CTAs take exactly its tile count of tickets (one work item per CTA)
        std::lock_guard<std::mutex> lock(split_mu);
        st->tickets = base + static_cast<unsigned int>(m_tiles * ((N + bn - 1) / bn) * split_k);
    }
    return rc;
}

int gemm_preload() {
    int rc = gemm_prepare<64>();
    if (rc == OK) rc = gemm_prepare<128>();
    if (rc == OK) rc = gemm_prepare<256>();
    return rc;
}

int gemm_tn_bf16(const void* A, long long lda, const void* B, long long ldb, void* C, long long ldc, int M, int N,
                 int K, int a_koff, int b_koff, int out_bf16, int accumulate, int force_bn, int max_ctas,
                 cudaStream_t stream) {
    return gemm_impl(A, lda, B, ldb, C, ldc, M, N, K, a_koff, b_koff, out_bf16, accumulate, force_bn, max_ctas, stream, 0);
}

}  // namespace ctcb200

// C[M,N] (+)= A[a_roff : a_roff+K, 0:M]^T * B[b_roff : b_roff+K, 0:N]: both operands stored with the CONTRACTED index as the row
// index (MN-major for the tensor core). This is the shape of every weight gradient (dW = dG^T X over the T*N rows of a batch):
// the gate gradients and the activations are consumed as the recurrent kernels / the forward pass left them, no transposed
// copies (round 1 spent 1.1 ms per cfg2 step on transpose_dg / cast_transpose kernels for the K-major form).
extern "C" CTCB200_API int ctcb200_gemm_atb_bf16(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
                                                 int M, int N, int K, int a_roff, int b_roff, int accumulate, int tile_n,
                                                 int max_ctas, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    return ctcb200::gemm_impl(A, lda, B, ldb, C, ldc, M, N, K, a_roff, b_roff, 0, accumulate, tile_n, max_ctas, stream, 1);
}

extern "C" CTCB200_API int ctcb200_gemm_preload(void) { return ctcb200::gemm_preload(); }

extern "C" CTCB200_API int ctcb200_gemm_tn_bf16(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
                                    int M, int N, int K, int a_koff, int b_koff, int out_bf16, int accumulate,
                                    int tile_n, int max_ctas, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    return ctcb200::gemm_tn_bf16(A, lda, B, ldb, C, ldc, M, N, K, a_koff, b_koff, out_bf16, accumulate, tile_n,
                                 max_ctas, stream);
}
