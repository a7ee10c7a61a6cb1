// K2 / K3 — persistent recurrent LSTM kernels (forward scan and BPTT) for one bidirectional layer.
//
// Replaces the time loop inside nn.LSTM(bias=False, bidirectional=True) that the reference calls at
// timit/models/model_ctc.py:23-26,33 (forward) and back-propagates through at
// timit/steps/train_ctc.py:63. Semantics reproduced exactly: h0 = c0 = 0, gate order i,f,g,o,
// c_t = sig(f) c_{t-1} + sig(i) tanh(g), h_t = sig(o) tanh(c_t), the reverse direction scans
// t = T-1 .. 0 over *all* padded frames (the reference does not pack sequences).
//
// Decomposition. The input projection x_t W_ih^T for all t is one big tensor-core GEMM (gemm.cu)
// done beforehand; what remains per step is the thin product W_hh h_{t-1} ([4H x H] x [H x N]).
// W_hh never leaves the chip: each CTA owns 32 hidden units = 128 gate rows of one direction and keeps that
// [128 x H] bf16 slice resident in TENSOR MEMORY (tcgen05.mma with the A operand in TMEM); per step it issues the
// K = H MMA chain from four warps into four TMEM accumulators. The H/32 CTAs of a (direction, batch group) form
// one thread-block cluster; the only per-step traffic is the all-gather of h_t (H x NB bf16), one bulk DSMEM copy
// per peer with complete_tx on the peer's mbarrier, landing directly in the next step's K-major SWIZZLE_64B
// B-operand image. Gate non-linearities, the cell update and the hadamard products are fused in registers.
//
// Kernels in this file (DESIGN.md §3.2 has the measurements):
//   lstm_fwd_pipe_kernel   default forward for H <= 512: two 8-column halves software-pipelined over element,
//                          tensor-core and copy warps; gx arrives as TMA boxes
//   lstm_fwd_kernel<NB,EX,X3,CELL> un-pipelined forward; EX selects the exchange (3 = bulk DSMEM copies inside one cluster,
//                          0 = global image + counter, cooperative launch: the fallback when no cluster fits)
//   lstm_bwd_kernel<NB,EX,X3,CELL> BPTT: CTA (q, mb) of a (4, H/128) cluster holds gate q's transposed slice for 128 units; the
//                          four gate partials are reduce-scattered (fp16 on the wire), the dG blocks all-gathered
//   X3 = split-operand mode (precision "x3"): every product is W_hi h_hi + W_hi h_lo + W_lo h_hi on bf16 hi/lo halves,
//                          fp32 hand-offs and fp32 saved gates: the path whose gradients meet the reference's fp32 numbers to 1e-3;
//                          its three-times-longer MMA chain starts on the first K block that lands (one mbarrier per K block,
//                          rotated exchange order: exchange_peer / arrival_kblock)
//   CELL = LSTM / GRU / vanilla RNN on one four-gate-slot layout (train_ctc.py:20's rnn_type choices)
//   lstm_fwd2/bwd2_kernel  two gate tiles per CTA for H in (512, 640]
#include <cuda_fp16.h>

#include <cstdlib>

#include "common.cuh"
#include "ctcb200.h"

namespace ctcb200 {
namespace {

constexpr int LSTM_THREADS = 256;

__device__ __forceinline__ void wait_counter(const unsigned int* flag, unsigned int target) {
    if (ld_acquire(flag) >= target) return;
    const long long t0 = clock64();
    while (ld_acquire(flag) < target) {
        if (clock64() - t0 > SPIN_LIMIT_CYCLES) spin_timeout_trap(2);
    }
}

__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }
// single-MUFU hyperbolic tangent (max relative error ~2^-11): experiment switch CTCB200_LSTM_ACT=approx
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Pack the bf16 of 8 consecutive lanes (this lane = lowest) into a uint4; valid on lanes % 8 == 0.
__device__ __forceinline__ uint4 pack8_bf16(float v) {
    __nv_bfloat16 b = __float2bfloat16(v);
    uint32_t x = static_cast<uint32_t>(*reinterpret_cast<unsigned short*>(&b));
    uint32_t p1 = x | (__shfl_down_sync(0xffffffffu, x, 1) << 16);
    uint32_t p2 = __shfl_down_sync(0xffffffffu, p1, 2);
    uint32_t p3 = __shfl_down_sync(0xffffffffu, p1, 4);
    uint32_t p4 = __shfl_down_sync(0xffffffffu, p2, 4);
    return make_uint4(p1, p2, p3, p4);
}

// Element offset (bf16 units) of the 16-byte chunk holding unit `u` (u % 8 == 0), batch row `n`, inside a [H x NB]
// K-major SWIZZLE_64B operand image: K blocks of 32 units = [NB rows x 64 bytes], 16-byte chunk c of row n stored at
// position c ^ ((n >> 1) & 3). The 32 units a CTA produces are therefore one contiguous NB*64-byte block.
// With PARTS = 2 (split-operand mode) every 32-unit block is [hi part | lo part]; this is the offset of the hi part.
template <int NB, int PARTS = 1>
__device__ __forceinline__ int image_chunk_offset(int u, int n) {
    const int kb = u >> 5, c = (u & 31) >> 3;
    return kb * (NB * 32 * PARTS) + n * 32 + ((c ^ ((n >> 1) & 3)) << 3);
}

// ---- thread-block-cluster primitives (distributed shared memory exchange) ------------------------------
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_v4(uint32_t addr, uint4 v) {
    asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive (release at cluster scope) on an mbarrier that lives in CTA `cta_rank` of this cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* local_bar, uint32_t cta_rank) {
    const uint32_t raddr = mapa_shared(smem_u32(local_bar), cta_rank);
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory");
}
// bulk (TMA-engine) copy of `bytes` from this CTA's shared memory into a peer CTA's shared memory; the peer's
// mbarrier receives complete_tx(bytes) when the data has landed — no separate arrive, no release fence
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes,
                                                  uint32_t mbar_cluster_addr) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     dst_cluster_addr),
                 "r"(src_cta_addr), "r"(bytes), "r"(mbar_cluster_addr)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait_cluster(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait_cluster(bar, parity)) {
        if (clock64() - t0 > SPIN_LIMIT_CYCLES) spin_timeout_trap(3);
    }
}

// Load this CTA's [128 x H] bf16 weight slice into TMEM columns [col0, col0 + H/2): row r -> lane r, K elements
// (2c, 2c+1) packed into 32-bit column c — the A-operand layout of tcgen05.mma with A in tensor memory.
// Executed by warps 0-3 (warp w owns lanes 32w..32w+31).
__device__ __forceinline__ void load_weights_to_tmem(const __nv_bfloat16* __restrict__ w_rows, int K, uint32_t tmem_base,
                                                     uint32_t col0, int warp, int lane, int row_pitch = 0) {
    if (row_pitch == 0) row_pitch = K;  // K = number of K elements to load per row
    const uint4* src = reinterpret_cast<const uint4*>(w_rows + static_cast<size_t>(warp * 32 + lane) * row_pitch);
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + col0;
    for (int kb = 0; kb < K / 16; ++kb) {
        const uint4 a = __ldg(src + 2 * kb), b = __ldg(src + 2 * kb + 1);
        const uint32_t r[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        tmem_st_32x8(taddr + kb * 8, r);
    }
    tmem_st_wait();
}

// Accumulator columns of up to four issuing warps -> registers, all loads in flight before the single wait, summed.
template <int CPT>
__device__ __forceinline__ void tmem_ld_cpt(uint32_t taddr, uint32_t (&r)[CPT]) {
    if constexpr (CPT == 16) tmem_ld_32x16(taddr, r);
    else if constexpr (CPT == 8) tmem_ld_32x8(taddr, r);
    else tmem_ld_32x4(taddr, r);
}
template <int CPT>
__device__ __forceinline__ void load_partial_sums(uint32_t taddr, int acc_stride, int parts, uint32_t (&acc)[CPT]) {
    uint32_t a1[CPT], a2[CPT], a3[CPT];
    tmem_ld_cpt<CPT>(taddr, acc);
    if (parts > 1) tmem_ld_cpt<CPT>(taddr + acc_stride, a1);
    if (parts > 2) {
        tmem_ld_cpt<CPT>(taddr + 2 * acc_stride, a2);
        tmem_ld_cpt<CPT>(taddr + 3 * acc_stride, a3);
    }
    tmem_ld_wait();
    if (parts > 1) {
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
            float v = __uint_as_float(acc[c]) + __uint_as_float(a1[c]);
            if (parts > 2) v += __uint_as_float(a2[c]) + __uint_as_float(a3[c]);
            acc[c] = __float_as_uint(v);
        }
    }
}
// Cell type of a recurrent layer (train_ctc.py:20 supported_rnn = nn.LSTM / nn.GRU / nn.RNN). All cells use the SAME operand
// layout — four gate slots per hidden unit, 128 gate rows per CTA — so that packing, the input-projection GEMM, the exchange
// and the weight-gradient GEMMs are shared: LSTM fills the slots with (i, f, g, o), GRU with (r, z, n, -), the vanilla RNN with
// (g, -, -, -); unused slots carry zero weights (some idle tensor-core work for a configuration option, no extra code paths).
enum { CELL_LSTM = 0, CELL_GRU = 1, CELL_RNN = 2 };

// ------------------------------------------------------------------------------------------------
// Split-operand (X3) kernels only: order of the per-step all-gather inside a cluster, and one mbarrier per K block.
// A bulk DSMEM copy costs ~33 cycles of the SM's copy engine on top of a ~315-cycle hand-off (tools/dsmem_bench.cu). The x3
// MMA chain is three times as long as the bf16 one (96 tcgen05.mma per step), so it pays to start it on the first K block that
// lands: the CTAs are paired (pair a = CTAs 2a, 2a+1 = the two 32-unit blocks of K block a), sender (a, b) serves receiver pair
// (a + i) mod P in slot i, every receiver gets one K block (two copies) per slot, and the issuing warps wait per K block.
// Measured (cfg2 layer shape, ms per launch): x3 forward 2.39 -> 2.14, x3 BPTT 2.61 -> 2.45. The bf16 kernels keep ONE barrier
// per operand image: with their short chain the extra waits cost more than the overlap returns (measured: BPTT 1.48 -> 1.7).
// ------------------------------------------------------------------------------------------------
constexpr int MAX_KB = 8;   // K blocks of 64 units in a one-cluster kernel (H <= 512)
// K elements of a [128 x H] weight slice that fit tensor memory next to the accumulators: columns [64, 64 + 896/2) of 512. The
// bf16 global-exchange kernels (EX = 0) take H up to 1024; the K blocks past 896 sit in shared memory (TMA, SWIZZLE_128B) and
// go through the SS-form MMA, as the x3 kernels' W_lo slice does.
constexpr int TMEM_K_MAX = 896;
constexpr int MAX_HIDDEN = 1024;     // largest (device) hidden size of the recurrent kernels
constexpr int MAX_HIDDEN_X3 = 640;   // split-operand mode: the W_lo slice and the hi/lo operand image must fit shared memory
__device__ __forceinline__ uint32_t exchange_peer(int me, int pos, int ctas) {   // pos-th destination of CTA `me`
    const int pairs = ctas >> 1;
    int c = (me >> 1) + (pos >> 1);
    if (c >= pairs) c -= pairs;
    return static_cast<uint32_t>(2 * c + ((me ^ pos) & 1));
}
__device__ __forceinline__ int arrival_kblock(int me, int it, int kblocks) {     // K block that lands it-th at CTA `me`
    int kb = (me >> 1) - it;
    if (kb < 0) kb += kblocks;
    return kb;
}
// Values prefetched from global memory at the top of a step go through an empty volatile asm where they are first used:
// volatile asms keep their order, so no arithmetic on them can be scheduled above the mbarrier waits in between (ptxas otherwise
// hoists e.g. the tanh of c_t in front of the MMA issue, and the issuing warps then stall on the global load every step).
__device__ __forceinline__ void pin_reg(float& x) { asm volatile("" : "+f"(x)); }
__device__ __forceinline__ void pin_reg(uint32_t& x) { asm volatile("" : "+r"(x)); }

struct FwdParams {
    const float* gx;          // [T*N, 8H] gate pre-activations from the input projection (packed column order)
    float* hout;              // [T*N, 2H] layer output (fwd | reverse)
    float* c_save;            // [T*N, 2H] cell states, or null (inference)
    uint2* gates_save;        // [T*N, 2H] activated gates as 4 x fp16 (i,f,g,o), or null
    float4* gates_save32;     // split-operand mode: the same as 4 x fp32 (BPTT then sees the gates at full precision)
    __nv_bfloat16* himg;      // EX = 0: [2 dirs][groups][2 parities][H*NB*PARTS] operand images in global memory
    unsigned int* flags;      // EX = 0: [2 dirs][groups] step counters, 32 uints apart
    int T, N, H, groups, n0;  // n0 = first batch row of this launch's group 0
    long long* trace;         // debug: per-step clock64 stamps of CTA (0,0,0), or null
    const __nv_bfloat16* w;   // packed recurrent weights [8H, H] (hi part): source of the TMEM-resident A operand
    int mma_split;            // number of warps (1, 2 or 4) that issue slices of the K chain into their own accumulator
    int act_approx;           // 1: gate non-linearities through tanh.approx (one MUFU op each)
    int rnn_relu;             // CELL_RNN: 1 = nonlinearity='relu', 0 = 'tanh'
    unsigned int* resident;   // optional uint32[2]: [0] += 1 once every CTA of this launch is running ([1] = arrivals)
    // Streamed input projection (all optional, gx_ready = null: gx is complete at launch). The rows of gx are produced chunk by
    // chunk by GEMM launches on ANOTHER stream while this kernel runs: chunk c holds the time steps each direction visits in
    // its scan steps [c * chunk_T, (c + 1) * chunk_T) (forward scan: rows t, reverse scan: rows T - 1 - t). Chunk 0 is complete
    // at launch (stream order); a stream memory operation publishes *gx_ready = gx_base + c once chunks 1..c are complete.
    const unsigned int* gx_ready;
    unsigned int gx_base;
    int chunk_T;
};

// Tell the host-side scheduler that the whole grid of this launch is resident: from then on the SMs this kernel does
// not use can be handed to independent work on another stream (the weight-gradient GEMMs of the layer above under a BPTT
// kernel, the later time chunks of the input projection under a forward kernel) without delaying the cluster launch. The last
// CTA to arrive publishes; the arrival word is reset for the next launch.
__device__ __forceinline__ void announce_resident(unsigned int* resident) {
    if (resident != nullptr && threadIdx.x == 0) {
        const unsigned int total = gridDim.x * gridDim.y * gridDim.z;
        if (atomicAdd(resident + 1, 1u) == total - 1) {
            atomicExch(resident + 1, 0u);
            __threadfence();
            atomicAdd(resident, 1u);
        }
    }
}

// Streamed input projection: block until the chunk that scan step t opens has been published (called by one lane; the data
// were written by TMA stores of a kernel that completed before the stream memory operation that published the counter).
__device__ __forceinline__ void wait_gx_chunk(const unsigned int* ready, unsigned int need) {
    if (static_cast<int>(ld_acquire_sys(ready) - need) >= 0) return;
    const long long t0 = clock64();
    bool reported = false;
    while (static_cast<int>(ld_acquire_sys(ready) - need) < 0) {
        __nanosleep(100);
        const long long dt = clock64() - t0;
        if (dt > SPIN_LIMIT_CYCLES / 2 && !reported) {   // (earlier than the mbarrier waits that pile up behind this one)
            printf("ctcb200: streamed input projection late: chunk counter %u, needed %u (block %d,%d,%d)\n",
                   ld_acquire_sys(ready), need, blockIdx.x, blockIdx.y, blockIdx.z);
            reported = true;
        }
        if (dt > SPIN_LIMIT_CYCLES + SPIN_LIMIT_CYCLES / 2) spin_timeout_trap(3);
    }
}
// gx element: coherent (L2) load while the projection is being streamed in by another kernel, read-only path otherwise
__device__ __forceinline__ float load_gx(const FwdParams& p, const float* a) {
    return p.gx_ready != nullptr ? ld_cg_f32(a) : __ldg(a);
}

// Split a float into bf16 hi + bf16 lo (hi + lo carries 16 mantissa bits of the value).
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16(v);
    lo = __float2bfloat16(v - __bfloat162float(hi));
}

// Un-pipelined forward recurrence (one element phase per step over all NB columns of the group).
//   EX = 3: the H/32 CTAs of one (direction, batch group) form one thread-block cluster and all-gather h_t with one bulk
//           (TMA-engine) DSMEM copy per peer, complete_tx on the peer's mbarrier.
//   EX = 0: exchange through a global operand image + release/acquire counter (any H, needs a cooperative launch).
//   X3    : split-operand ("bf16x3") mode for fp32-grade results: W = W_hi + W_lo, h = h_hi + h_lo (all bf16) and the product
//           is accumulated as W_hi h_hi + W_hi h_lo + W_lo h_hi in the fp32 TMEM accumulator (the dropped W_lo h_lo term is
//           2^-18 relative). W_hi stays resident in TMEM, W_lo in shared memory (TMA-loaded once, SWIZZLE_128B); every
//           32-unit block of the operand image carries [hi | lo], so the exchange is still one copy per peer.
template <int NB, int EX, bool X3, int CELL = CELL_LSTM>
__global__ void __launch_bounds__(LSTM_THREADS, 1)
lstm_fwd_kernel(const __grid_constant__ CUtensorMap tmWlo, FwdParams p) {
    constexpr bool CL = EX != 0, BULK = EX == 3;
    constexpr int PARTS = X3 ? 2 : 1;
    constexpr uint32_t BLK_BYTES = NB * 64;             // 32 units x NB batch rows of one operand part
    constexpr uint32_t BLK_STRIDE = PARTS * BLK_BYTES;  // what one CTA contributes to the operand image per step
    constexpr int CPT = NB / 2;        // accumulator columns per thread
    constexpr int EPT = NB / 8;        // (unit, batch) elements per thread in the cell update
    constexpr int S_STRIDE = NB * 4 + 4;
    constexpr int OUT_CHUNKS = NB * 4; // 16-byte chunks of one part of h_t this CTA produces per step (32 units x NB)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int H = p.H, T = p.T, N = p.N;
    const int himg_bytes = H * NB * 2 * PARTS;
    constexpr bool SPILL = EX == 0 && !X3;                           // H > TMEM_K_MAX possible (see TMEM_K_MAX)
    const int k_tmem = (SPILL && H > TMEM_K_MAX) ? TMEM_K_MAX : H;   // K elements of the W slice resident in TMEM
    const int kb_tmem = k_tmem / 64;
    uint8_t* sW = smem;                                              // X3: the W_lo slice [128 x H] bf16; SPILL: K >= k_tmem
    uint8_t* sH = sW + (X3 ? 128 * H * 2 : (SPILL ? 128 * (H - k_tmem) * 2 : 0));   // BULK: two parities, else one buffer
    float* sS = reinterpret_cast<float*>(sH + (BULK ? 2 : 1) * himg_bytes);
    uint4* sOut = reinterpret_cast<uint4*>(sS + 32 * S_STRIDE);      // BULK only: staging of this CTA's block [hi | lo]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + (BULK ? PARTS * OUT_CHUNKS : 0));
    uint64_t* w_full = bars;
    uint64_t* acc_full = bars + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
    // h_full[parity * HB_STRIDE + kb]: BULK -> the peers' blocks of a parity have landed (X3: one barrier per K block kb, see
    // exchange_peer; bf16: kb = 0 only); EX=0 -> [0] counts the local image copy
    constexpr bool KBB = BULK && X3;
    constexpr int HB_STRIDE = KBB ? MAX_KB : 1;
    uint64_t* h_full = bars + 4;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int j = blockIdx.x, dir = blockIdx.y, grp = blockIdx.z;
    const int ctas = gridDim.x;
    const int kblocks = H / 64;
    announce_resident(p.resident);

    if (tid == 0) {
        if constexpr (X3) tma_prefetch_desc(&tmWlo);
        mbar_init(w_full, 1);
        for (int i = 0; i < 2 * HB_STRIDE; ++i) mbar_init(&h_full[i], BULK ? 1 : LSTM_THREADS);
        mbar_init(acc_full, p.mma_split);
        fence_mbar_init();
        if constexpr (BULK) {  // arm both parities: each expects one block from every CTA of the cluster (two per K block)
            for (int i = 0; i < 2 * HB_STRIDE; ++i) mbar_expect_tx(&h_full[i], (KBB ? 2 : ctas) * BLK_STRIDE);
        }
    }
    // TMEM: up to four accumulators in columns [0, 64), the W_hi slice (A operand) in columns [64, 64 + k_tmem/2)
    uint32_t tmem_cols = 64;
    while (tmem_cols < 64u + k_tmem / 2) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    if constexpr (BULK) {
        // h_{-1} = 0: the first operand buffer starts zeroed
        for (int i = tid; i < himg_bytes / 16; i += LSTM_THREADS) reinterpret_cast<uint4*>(sH)[i] = make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if constexpr (CL) cluster_sync_all();  // peers' barriers are initialised before anyone arrives on them

    if (warp < 4)
        load_weights_to_tmem(p.w + (static_cast<size_t>(dir) * 4 * H + j * 128) * H, k_tmem, tmem_base, 64, warp, lane,
                             SPILL ? H : 0);
    if constexpr (X3) {
        if (tid == 0) {
            mbar_expect_tx(w_full, 128 * H * 2);
            for (int kb = 0; kb < kblocks; ++kb) tma_load_2d(sW + kb * 16384, &tmWlo, w_full, kb * 64, dir * 4 * H + j * 128);
        }
    }
    if constexpr (SPILL) {   // (tmWlo maps the W_hi image here)
        if (tid == 0 && k_tmem < H) {
            mbar_expect_tx(w_full, 128 * (H - k_tmem) * 2);
            for (int kb = kb_tmem; kb < kblocks; ++kb)
                tma_load_2d(sW + (kb - kb_tmem) * 16384, &tmWlo, w_full, kb * 64, dir * 4 * H + j * 128);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int lq = warp & 3, ch = warp >> 2;
    const bool warp_leader = elect_one();      // the lane of each warp that issues / tracks its bulk copies
    const int row = lq * 32 + lane;            // gate row inside this CTA's 128
    const int u_loc = row >> 2, q = row & 3;   // hidden unit (0..31) and gate (i,f,g,o)
    const float act_s = (q == 2) ? 2.0f : 1.0f;
    const float act_h = (q == 2) ? 1.0f : 0.5f;
    const size_t gx_col = static_cast<size_t>(dir) * 4 * H + j * 128 + row;
    const size_t G8 = static_cast<size_t>(8) * H, H2 = static_cast<size_t>(2) * H;
    __nv_bfloat16* img = BULK ? nullptr : p.himg + (static_cast<size_t>(dir) * p.groups + grp) * 2 * H * NB * PARTS;
    unsigned int* flag = CL ? nullptr : p.flags + (dir * p.groups + grp) * 32;
    const int chunks = H * NB / 8 * PARTS;
    constexpr uint32_t idesc = umma_idesc_bf16(128, NB);

    float c_state[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) c_state[e] = 0.0f;

#define TRACE(k) do { if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && tid == (k >= 8 ? 255 : 0)) p.trace[t * 16 + (k)] = clock64(); } while (0)
    int gx_gate = p.chunk_T;   // first scan step of the next chunk of a streamed input projection
    for (int t = 0; t < T; ++t) {
        const int tt = dir ? (T - 1 - t) : t;
        TRACE(0);
        // (1) this step's input-projection terms: independent of the recurrence, issued first
        if (p.gx_ready != nullptr && t == gx_gate) {   // streamed projection: the chunk this step opens must have landed
            if (lane == 0) wait_gx_chunk(p.gx_ready, p.gx_base + static_cast<unsigned int>(t / p.chunk_T));
            __syncwarp();
            gx_gate += p.chunk_T;
        }
        float gx[CPT];
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
            const int gn = p.n0 + grp * NB + ch * CPT + c;
            gx[c] = (gn < N) ? load_gx(p, p.gx + (static_cast<size_t>(tt) * N + gn) * G8 + gx_col) : 0.0f;
        }
        if constexpr (!BULK) {
            // (2) all CTAs of this (direction, group) have published h_{t-1}
            if (lane == 0) wait_counter(flag, static_cast<unsigned int>(ctas) * t);
            __syncwarp();
            // (3) operand image -> shared memory
            const uint4* src = reinterpret_cast<const uint4*>(img + static_cast<size_t>(t & 1) * H * NB * PARTS);
            uint4* dst = reinterpret_cast<uint4*>(sH);
            for (int i = tid; i < chunks; i += LSTM_THREADS) dst[i] = ld_cg_v4(src + i);
            fence_proxy_async_smem();
            mbar_arrive(&h_full[0]);
        }
        // (4) up to four warps issue interleaved K blocks of the chain into their own accumulator (the issue rate of one
        // warp, ~40 cycles per tcgen05.mma, would bound the chain); the whole warp runs the warp-uniform address
        // arithmetic so the descriptors live in uniform registers, one elected lane issues each tcgen05.mma
        if (warp < p.mma_split) {
            if constexpr (X3) { if (t == 0) mbar_wait(w_full, 0); }
            if constexpr (SPILL) { if (t == 0 && k_tmem < H) mbar_wait(w_full, 0); }
            if constexpr (KBB) {
                // per-K-block waits inside the loop; the issuing warps took part in last step's CTA barriers themselves
            } else if constexpr (BULK) {
                if (t > 0) {
                    mbar_wait(&h_full[t & 1], ((t - 1) >> 1) & 1);                // every peer's block has landed
                    if (lane == 0 && warp == 0) mbar_expect_tx(&h_full[t & 1], ctas * BLK_STRIDE);  // re-arm for step t+2
                }
            } else {
                mbar_wait(&h_full[0], t & 1);
            }
            tc_fence_after();
            TRACE(1);
            const uint32_t a0 = smem_u32(sW), b0 = smem_u32(sH) + (BULK ? (t & 1) * himg_bytes : 0);
            const bool leader = elect_one();
            const int kstep = p.mma_split, kfirst = warp;
            const uint32_t dacc = tmem_base + warp * NB;
            constexpr uint32_t B2 = BLK_STRIDE / 16;   // descriptor step to the second 32-unit block of a 64-wide K block
            constexpr uint32_t LO = BLK_BYTES / 16;    // descriptor step from a block's hi part to its lo part
#pragma unroll 1
            for (int it = kfirst; it < kblocks; it += kstep) {
                const int kb = KBB ? arrival_kblock(j, it, kblocks) : it;   // X3: K blocks in their arrival order
                if constexpr (KBB) {
                    if (t > 0) {
                        uint64_t* kf = &h_full[(t & 1) * HB_STRIDE + kb];
                        mbar_wait(kf, ((t - 1) >> 1) & 1);                    // both source blocks of this K block have landed
                        if (lane == 0) mbar_expect_tx(kf, 2 * BLK_STRIDE);    // re-arm for step t + 2 (this warp owns kb)
                    }
                }
                // 64 K elements = two SWIZZLE_64B blocks of the B image, two K=16 slices (32 bytes apart) in each
                const uint64_t bd = umma_desc_sw64(b0 + kb * (2 * BLK_STRIDE));
                const uint32_t ta = tmem_base + 64 + kb * 32;
                if (SPILL && kb >= kb_tmem) {   // this K block of W sits in shared memory
                    const uint64_t ad = umma_desc_sw128(a0 + (kb - kb_tmem) * 16384);
                    if (leader) {
                        umma_bf16(dacc, ad, bd, idesc, it != kfirst ? 1u : 0u);
                        umma_bf16(dacc, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(dacc, ad + 4, bd + B2, idesc, 1u);
                        umma_bf16(dacc, ad + 6, bd + B2 + 2, idesc, 1u);
                    }
                } else if (leader) {
                    umma_bf16_ts(dacc, ta, bd, idesc, it != kfirst ? 1u : 0u);
                    umma_bf16_ts(dacc, ta + 8, bd + 2, idesc, 1u);
                    umma_bf16_ts(dacc, ta + 16, bd + B2, idesc, 1u);
                    umma_bf16_ts(dacc, ta + 24, bd + B2 + 2, idesc, 1u);
                }
                if constexpr (X3) {
                    const uint64_t ad = umma_desc_sw128(a0 + kb * 16384);
                    if (leader) {
                        // W_hi x h_lo
                        umma_bf16_ts(dacc, ta, bd + LO, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 8, bd + LO + 2, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 16, bd + B2 + LO, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 24, bd + B2 + LO + 2, idesc, 1u);
                        // W_lo x h_hi
                        umma_bf16(dacc, ad, bd, idesc, 1u);
                        umma_bf16(dacc, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(dacc, ad + 4, bd + B2, idesc, 1u);
                        umma_bf16(dacc, ad + 6, bd + B2 + 2, idesc, 1u);
                    }
                }
            }
            if (leader) umma_commit(acc_full);
            TRACE(2);
        }
        __syncwarp();
        // (5) accumulator -> registers
        mbar_wait(acc_full, t & 1);
        tc_fence_after();
        TRACE(3); TRACE(8);
        uint32_t acc[CPT];
        load_partial_sums<CPT>(tmem_base + (static_cast<uint32_t>(lq * 32) << 16) + ch * CPT, NB, p.mma_split, acc);
        tc_fence_before();
        TRACE(4); TRACE(9);
        // (6) gate non-linearity, then regroup the four gates of a unit through shared memory
        if constexpr (CELL == CELL_LSTM) {
#pragma unroll
            for (int c = 0; c < CPT; ++c) {
                const float pre = __uint_as_float(acc[c]) + gx[c];
                float a;
                if (p.act_approx) a = act_h * tanh_approx(act_h * pre) + (1.0f - act_h);   // sigmoid(x) = (tanh(x/2) + 1) / 2
                else a = act_s * fast_sigmoid(act_s * pre) - (act_s - 1.0f);              // sigmoid, or tanh for gate g
                sS[u_loc * S_STRIDE + (ch * CPT + c) * 4 + q] = a;
            }
        } else if constexpr (CELL == CELL_GRU) {
            // slots (r, z, n, -): r, z = sigmoid(W_h. h + gx); the n gate needs r first, so its recurrent part W_hn h and its
            // input part gx_n travel separately (slot 2 and the unused slot 3) to the thread that finishes the unit
#pragma unroll
            for (int c = 0; c < CPT; ++c) {
                const float rec = __uint_as_float(acc[c]);
                float* dst = sS + u_loc * S_STRIDE + (ch * CPT + c) * 4;
                if (q < 2) dst[q] = fast_sigmoid(rec + gx[c]);
                else if (q == 2) { dst[2] = rec; dst[3] = gx[c]; }
            }
        } else {
#pragma unroll
            for (int c = 0; c < CPT; ++c)
                if (q == 0) sS[u_loc * S_STRIDE + (ch * CPT + c) * 4] = __uint_as_float(acc[c]) + gx[c];
        }
        TRACE(10);
        if constexpr (BULK) { if (warp_leader) bulk_wait_read_all(); }  // last step's copies have finished reading sOut
        __syncthreads();
        TRACE(5); TRACE(11);
        // (7) cell update for (unit = lane, batch n = warp + 8e); publish h_t as the next step's B operand
        float hv[EPT];
        float4 gv[EPT];
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int n = warp + 8 * e;
            float4 g4 = *reinterpret_cast<const float4*>(&sS[lane * S_STRIDE + n * 4]);
            float h;
            if constexpr (CELL == CELL_LSTM) {
                const float cn = g4.y * c_state[e] + g4.x * g4.z;
                c_state[e] = cn;
                h = g4.w * (p.act_approx ? tanh_approx(cn) : fast_tanh(cn));
            } else if constexpr (CELL == CELL_GRU) {
                // n = tanh(gx_n + r (W_hn h)), h' = (1 - z) n + z h  (torch's GRU, bias-free); saved slots: (r, z, n, W_hn h)
                const float nn_ = fast_tanh(g4.w + g4.x * g4.z);
                h = (1.0f - g4.y) * nn_ + g4.y * c_state[e];
                c_state[e] = h;                       // the recurrent state is h itself; c_save then holds h_t for BPTT
                g4 = make_float4(g4.x, g4.y, nn_, g4.z);
            } else {
                h = p.rnn_relu ? fmaxf(g4.x, 0.0f) : fast_tanh(g4.x);
                c_state[e] = h;
                g4 = make_float4(h, 0.0f, 0.0f, 0.0f);
            }
            hv[e] = h;
            gv[e] = g4;
            __nv_bfloat16 h_hi, h_lo;
            split_bf16(h, h_hi, h_lo);
            if constexpr (BULK) {
                // staging in destination order: chunk `oct` of row n sits at slot oct ^ ((n >> 1) & 3) of the 64-byte
                // row; every lane drops its own bf16 (no shuffle chain on the critical path)
                const int so = n * 32 + (((lane >> 3) ^ ((n >> 1) & 3)) << 3) + (lane & 7);
                reinterpret_cast<__nv_bfloat16*>(sOut)[so] = h_hi;
                if constexpr (X3) reinterpret_cast<__nv_bfloat16*>(sOut)[OUT_CHUNKS * 8 + so] = h_lo;
            } else {
                __nv_bfloat16* nxt = img + static_cast<size_t>((t + 1) & 1) * H * NB * PARTS + image_chunk_offset<NB, PARTS>(j * 32 + lane, n);
                const uint4 pk = pack8_bf16(__bfloat162float(h_hi));
                if ((lane & 7) == 0) *reinterpret_cast<uint4*>(nxt) = pk;
                if constexpr (X3) {
                    const uint4 pl = pack8_bf16(__bfloat162float(h_lo));
                    if ((lane & 7) == 0) *reinterpret_cast<uint4*>(nxt + NB * 32) = pl;
                }
            }
        }
        TRACE(12);
        if constexpr (BULK) {
            fence_proxy_async_smem();   // staging writes (generic proxy) -> bulk-copy engine (async proxy)
            __syncthreads();
            TRACE(6);
            if (t + 1 < T) {
                // one bulk copy per peer (our contiguous block -> slot j of the peer's next operand buffer); warp w
                // serves peers w and w + 8 so the copies are issued in parallel with warp-uniform operands
                const uint32_t dst = smem_u32(sH) + ((t + 1) & 1) * himg_bytes + j * BLK_STRIDE;
                const uint32_t bar = smem_u32(&h_full[((t + 1) & 1) * HB_STRIDE + (KBB ? (j >> 1) : 0)]);
#pragma unroll
                for (int pos = warp; pos < 16; pos += 8) {
                    if (pos < ctas && warp_leader) {
                        const uint32_t d = KBB ? exchange_peer(j, pos, ctas) : static_cast<uint32_t>(pos);
                        bulk_copy_to_peer(mapa_shared(dst, d), smem_u32(sOut), BLK_STRIDE, mapa_shared(bar, d));
                    }
                }
                if (warp_leader) bulk_commit();
            }
            TRACE(13); TRACE(7);
        } else {
            __threadfence();
            __syncthreads();
            if (tid == 0) red_release_add(flag, 1u);
        }
        // (8) off the critical path: layer output and the activations BPTT needs
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int gn = p.n0 + grp * NB + warp + 8 * e;
            if (gn < N) {
                const size_t o = (static_cast<size_t>(tt) * N + gn) * H2 + static_cast<size_t>(dir) * H + j * 32 + lane;
                p.hout[o] = hv[e];
                if (p.c_save) p.c_save[o] = c_state[e];
                if (p.gates_save32) {
                    p.gates_save32[o] = gv[e];
                } else if (p.gates_save) {
                    __half2 lo = __floats2half2_rn(gv[e].x, gv[e].y), hi = __floats2half2_rn(gv[e].z, gv[e].w);
                    p.gates_save[o] = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CL) cluster_sync_all();  // no CTA exits while a peer may still address its shared memory
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// forward, software-pipelined: the 16 batch columns of a group are two independent recurrences (columns 0-7 = half A,
// 8-15 = half B). Warps 0-7 run the element phase (TMEM -> gates -> cell -> h_t -> bulk copies to the peers) of A and B
// alternately; warps 8-11 only issue tensor-core work. While half A's h_t is in flight to the cluster and its next
// W_hh h product is being issued, the element warps are busy with half B, and vice versa — the DSMEM hand-off and the
// MMA chain disappear from the per-step critical path of the CTA. Each half has its own mbarriers, accumulators and
// staging block; both halves share the operand image (half A = rows 0-7 of every 16-row block, half B = rows 8-15:
// the 1 KB block a CTA contributes per step is the two halves back to back). An MMA (N = 16) of one half also
// multiplies the other half's rows, possibly mid-update: those accumulator columns are never read.
// ------------------------------------------------------------------------------------------------
constexpr int PIPE_THREADS = 512;   // 8 element warps + 4 tensor-core warps + 4 copy warps


__global__ void __launch_bounds__(PIPE_THREADS, 1)
lstm_fwd_pipe_kernel(const __grid_constant__ CUtensorMap tmGx, FwdParams p) {
    constexpr int NB = 16, HB = 8;              // batch columns per group / per half
    constexpr uint32_t BLK_BYTES = NB * 64;     // block of one CTA inside the operand image (both halves)
    constexpr uint32_t HALF_BYTES = HB * 64;
    constexpr uint32_t ACC_COLS = 128;          // 2 halves x 4 issuing warps x 16 accumulator columns
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int H = p.H, T = p.T, N = p.N;
    const int himg_bytes = H * NB * 2;
    uint8_t* sH = smem;                                                     // two parities
    uint8_t* sOut = sH + 2 * himg_bytes;                                    // [2 halves][2 parities][HALF_BYTES] staging
    float* sGx = reinterpret_cast<float*>(sOut + 4 * HALF_BYTES);           // [4 stages][8 batch rows][128 gate rows] (TMA boxes)
    uint64_t* bars = reinterpret_cast<uint64_t*>(sGx + 4 * HB * 128);
    uint64_t* h_full = bars;          // [half][parity]: every peer's half block of h_{t-1} has landed
    uint64_t* acc_full = bars + 4;    // [half]: the four partial accumulators of a half-step are complete
    // [half][parity of t]: all element warps have staged their part of h_t. One barrier per step parity: a copy warp that is
    // late by more than a step (it polls the chunk counter of a streamed input projection) must not find its barrier a full
    // parity cycle ahead — the cluster stalls before the element warps can arrive for step t + 2, so with two barriers per half
    // a late waiter always still sees "its" phase
    uint64_t* so_ready = bars + 6;
    uint64_t* gx_full = bars + 10;    // [4 stages]: the input-projection box of a half-step has landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int j = blockIdx.x, dir = blockIdx.y, grp = blockIdx.z;
    const int ctas = gridDim.x;
    const int kblocks = H / 64;
    announce_resident(p.resident);

    if (tid == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(&h_full[i], 1);
        mbar_init(&acc_full[0], 4);
        mbar_init(&acc_full[1], 4);
        for (int i = 0; i < 4; ++i) mbar_init(&so_ready[i], 8);
        for (int i = 0; i < 4; ++i) mbar_init(&gx_full[i], 1);
        tma_prefetch_desc(&tmGx);
        fence_mbar_init();
        for (int i = 0; i < 4; ++i) mbar_expect_tx(&h_full[i], ctas * HALF_BYTES);
    }
    uint32_t tmem_cols = 256;
    while (tmem_cols < ACC_COLS + H / 2) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    for (int i = tid; i < 2 * himg_bytes / 16; i += PIPE_THREADS)
        reinterpret_cast<uint4*>(sH)[i] = make_uint4(0u, 0u, 0u, 0u);   // h_{-1} = 0
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();
    if (warp < 4) load_weights_to_tmem(p.w + (static_cast<size_t>(dir) * 4 * H + j * 128) * H, H, tmem_base, ACC_COLS, warp, lane);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    constexpr uint32_t idesc = umma_idesc_bf16(128, NB);
#ifdef CTCB200_TRACE   // phase stamps: compiled in only for the trace build (python -m ctc_pytorch_b200._build --trace)
#define PTRACE(k) do { if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && lane == 0) p.trace[t * 16 + (k)] = clock64(); } while (0)
#else
#define PTRACE(k) do { } while (0)
#endif

    if (warp >= 12) {
        // ---------------- copy warps: warp 12 + w ships this CTA's staged half block to peers 4w .. 4w+3 (issuing a bulk
        // copy costs ~60 cycles of its scheduler, so the sixteen copies are spread over the four schedulers);
        // the element warps never wait for the copy engine. A staging block (half, parity of t) is reused two steps later,
        // by which time the element phase has consumed h_{t+1} of every peer, which they could only produce after this
        // block had landed everywhere — no wait_group needed.
        // Warp 12 also keeps a 4-deep ring of input-projection boxes (gx rows of the 8 batch columns of a half-step x this
        // CTA's 128 gate rows, one TMA tensor load each) four half-steps ahead of the element phase.
        // Streamed input projection (FwdParams::gx_ready): a box of a chunk that has not been published yet is NOT waited for
        // here — the copy duties of this warp must never fall behind (the hand-off barriers are parity-tracked: a copy warp that
        // blocks for a while finds its so_ready barrier two phases ahead and waits forever; observed). The fetch is deferred
        // instead and retried while this lane waits for the next so_ready, which is exactly where the element warps end up
        // waiting when they run out of boxes.
        int gx_gate = p.chunk_T;               // first scan step of the next unpublished chunk ...
        unsigned int gate_need = p.gx_base + 1u;   // ... and the counter value that publishes it
        int next_k = 0;                        // next half-step (k = 2 t + half) whose box has not been requested yet
        auto try_fetch = [&]() -> bool {
            const int k = next_k;
            const int t_ = k >> 1, half_ = k & 1;
            const int tt_ = dir ? (T - 1 - t_) : t_;
            if (p.gx_ready != nullptr && t_ >= gx_gate) {
                if (static_cast<int>(ld_acquire_sys(p.gx_ready) - gate_need) < 0) return false;
                fence_proxy_async_all();   // the flag was read through the generic proxy, the box is fetched by the TMA unit
                gx_gate += p.chunk_T;
                ++gate_need;
            }
            mbar_expect_tx(&gx_full[k & 3], HB * 128 * 4);
            tma_load_2d(sGx + (k & 3) * HB * 128, &tmGx, &gx_full[k & 3], dir * 4 * H + j * 128, tt_ * N + grp * NB + half_ * HB);
            ++next_k;
            return true;
        };
        if (warp == 12 && lane == 0)
            while (next_k < 4 && next_k < 2 * T && try_fetch()) {}   // (chunk_T >= 2: steps 0 and 1 are in chunk 0)
        for (int t = 0; t + 1 < T; ++t) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int k_cur = 2 * t + half;
                // Normally every box up to k_cur + 3 has been requested and all lanes simply wait for the element warps. Only
                // when a box was deferred (its chunk of a streamed projection had not been published) lane 0 polls alone and
                // retries the request while it waits: box k uses ring stage k & 3, free once half-step k - 4 has been observed.
                const bool deferred = warp == 12 && __shfl_sync(0xffffffffu, next_k <= k_cur + 3 && next_k < 2 * T ? 1 : 0, 0) != 0;
                if (deferred) {
                    if (lane == 0) {
                        uint64_t* sr = &so_ready[half * 2 + (t & 1)];
                        const long long t0 = clock64();
                        while (!mbar_try_wait(sr, (t >> 1) & 1)) {
                            if (next_k <= k_cur + 3 && next_k < 2 * T) try_fetch();
                            if (clock64() - t0 > SPIN_LIMIT_CYCLES) { spin_timeout_report(10 + half, t); spin_timeout_trap(4); }
                        }
                    }
                    __syncwarp();
                } else {
                    mbar_wait_tag(&so_ready[half * 2 + (t & 1)], (t >> 1) & 1, 10 + half, t);
                }
                if (warp == 12 && half == 0) PTRACE(10);
                const int d = (warp - 12) * 4 + lane;
                if (lane < 4 && d < ctas) {
                    const uint32_t src = smem_u32(sOut + (half * 2 + (t & 1)) * HALF_BYTES);
                    const uint32_t dst = smem_u32(sH) + ((t + 1) & 1) * himg_bytes + j * BLK_BYTES + half * HALF_BYTES;
                    const uint32_t bar = smem_u32(&h_full[half * 2 + ((t + 1) & 1)]);
                    bulk_copy_to_peer(mapa_shared(dst, static_cast<uint32_t>(d)), src, HALF_BYTES,
                                      mapa_shared(bar, static_cast<uint32_t>(d)));
                }
                __syncwarp();
                // the hand-off first, then the prefetch: this half-step's stage is free now as well (k <= k_cur + 4)
                if (warp == 12 && lane == 0)
                    while (next_k <= k_cur + 4 && next_k < 2 * T && try_fetch()) {}
                if (warp == 12 && half == 0) PTRACE(11);
            }
        }
        if (warp == 12 && lane == 0) {
            // deferred boxes of the last steps: their stages are free (half-steps <= 2T - 5 were observed above) and this warp
            // has no other duty left, so it may block on the chunk counter now
            while (next_k < 2 * T) {
                if (!try_fetch()) wait_gx_chunk(p.gx_ready, gate_need);
            }
        }
    } else if (warp >= 8) {
        // ---------------- tensor-core warps: K blocks m, m+4, ... of every half-step into accumulator (half, m) ----------
        const int m = warp - 8;
        const bool leader = elect_one();
        for (int t = 0; t < T; ++t) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                uint64_t* hf = &h_full[half * 2 + (t & 1)];
                if (t > 0) {
                    mbar_wait_tag(hf, ((t - 1) >> 1) & 1, 20 + half, t);   // every peer's half block has landed
                    if (m == 0 && lane == 0) mbar_expect_tx(hf, ctas * HALF_BYTES);   // re-arm for step t + 2
                }
                tc_fence_after();
                if (m == 0) PTRACE(12 + 2 * half);
                const uint32_t b0 = smem_u32(sH) + (t & 1) * himg_bytes;
                const uint32_t dacc = tmem_base + half * 64 + m * NB;
#pragma unroll 1
                for (int kb = m; kb < kblocks; kb += 4) {
                    const uint64_t bd = umma_desc_sw64(b0 + kb * (NB * 128));
                    const uint32_t ta = tmem_base + ACC_COLS + kb * 32;
                    if (leader) {
                        umma_bf16_ts(dacc, ta, bd, idesc, kb != m ? 1u : 0u);
                        umma_bf16_ts(dacc, ta + 8, bd + 2, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 16, bd + (NB * 64 / 16), idesc, 1u);
                        umma_bf16_ts(dacc, ta + 24, bd + (NB * 64 / 16) + 2, idesc, 1u);
                    }
                }
                if (leader) umma_commit(&acc_full[half]);
                __syncwarp();
                if (m == 0) PTRACE(13 + 2 * half);
            }
        }
    } else {
        // ---------------- element warps ---------------------------------------------------------------------------------
        // Thread (lq, ch, lane): TMEM lane = gate row lq*32 + lane = (unit lq*8 + lane/4, gate lane%4), accumulator columns
        // ch*4 .. ch*4+3 of the half. After the non-linearity a 4x4 transpose inside each lane quad (two shuffle rounds)
        // gives every lane the four gates of ONE batch column, so the cell update needs no shared-memory regrouping.
        const int lq = warp & 3, ch = warp >> 2;
        const int row = lq * 32 + lane;
        const int q = lane & 3, u = lq * 8 + (lane >> 2);       // gate of the accumulator row; hidden unit inside this CTA
        const bool b0 = (q & 1) != 0, b1 = (q & 2) != 0;
        const int n = ch * 4 + q;                               // batch column (inside the half) this lane finishes
        const float act_s = (q == 2) ? 2.0f : 1.0f;
        const float act_h = (q == 2) ? 1.0f : 0.5f;
        const size_t gx_col = static_cast<size_t>(dir) * 4 * H + j * 128 + row;
        const size_t G8 = static_cast<size_t>(8) * H, H2 = static_cast<size_t>(2) * H;
        const int parts = (kblocks < 4) ? kblocks : 4;   // accumulators that received MMAs (H = 128: two K blocks)
        const int so_off = n * 32 + ((lq ^ ((n >> 1) & 3)) << 3) + (lane >> 2);   // bf16 slot of (row n, unit u) in a half block
        float c_state[2] = {0.0f, 0.0f};
        for (int t = 0; t < T; ++t) {
            const int tt = dir ? (T - 1 - t) : t;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                if (warp == 0) PTRACE(6 * half + 0);
                mbar_wait_tag(&acc_full[half], t & 1, 30 + half, t);
                tc_fence_after();
                if (warp == 0) PTRACE(6 * half + 1);
                uint32_t acc[4];
                // accumulator column = image row: half B's batch columns are columns 8-15 of its accumulators
                load_partial_sums<4>(tmem_base + (static_cast<uint32_t>(lq * 32) << 16) + half * 64 + half * HB + ch * 4, NB, parts,
                                     acc);
                tc_fence_before();
                if (warp == 0) PTRACE(6 * half + 2);
                mbar_wait_tag(&gx_full[((t & 1) << 1) | half], (t >> 1) & 1, 40 + half, t);   // box of half-step k = 2t + half: stage k & 3, phase k >> 2
                const float* gxs = sGx + ((((t & 1) << 1) | half) * HB + ch * 4) * 128 + row;
                float a[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float pre = __uint_as_float(acc[c]) + gxs[c * 128];
                    if (p.act_approx) a[c] = act_h * tanh_approx(act_h * pre) + (1.0f - act_h);
                    else a[c] = act_s * fast_sigmoid(act_s * pre) - (act_s - 1.0f);   // sigmoid, or tanh for gate g
                }
                // quad transpose: round 1 swaps the odd/even column of each column pair with lane q^1, round 2 swaps
                // column pairs with lane q^2; afterwards r0..r3 = gates q, q^1, q^2, q^3 of column n
                const float k0 = b0 ? a[1] : a[0], s0 = b0 ? a[0] : a[1];
                const float k1 = b0 ? a[3] : a[2], s1 = b0 ? a[2] : a[3];
                const float x0 = __shfl_xor_sync(0xffffffffu, s0, 1), x1 = __shfl_xor_sync(0xffffffffu, s1, 1);
                const float r0 = b1 ? k1 : k0, r1 = b1 ? x1 : x0;
                const float y0 = b1 ? k0 : k1, y1 = b1 ? x0 : x1;
                const float r2 = __shfl_xor_sync(0xffffffffu, y0, 2), r3 = __shfl_xor_sync(0xffffffffu, y1, 2);
                const float e0 = b0 ? r1 : r0, e1 = b0 ? r0 : r1, e2 = b0 ? r3 : r2, e3 = b0 ? r2 : r3;
                const float gi = b1 ? e2 : e0, gf = b1 ? e3 : e1, gg = b1 ? e0 : e2, go = b1 ? e1 : e3;
                if (warp == 0) PTRACE(6 * half + 3);
                const float cn = gf * c_state[half] + gi * gg;
                c_state[half] = cn;
                const float h = go * (p.act_approx ? tanh_approx(cn) : fast_tanh(cn));
                // staging blocks are double-buffered per half (parity of t); see the copy warp for why reuse is safe
                uint8_t* so = sOut + (half * 2 + (t & 1)) * HALF_BYTES;
                reinterpret_cast<__nv_bfloat16*>(so)[so_off] = __float2bfloat16(h);
                fence_proxy_async_smem();   // staging writes (generic proxy) -> bulk-copy engine (async proxy)
                __syncwarp();
                if (lane == 0) mbar_arrive(&so_ready[half * 2 + (t & 1)]);
                if (warp == 0) PTRACE(6 * half + 4);
                // off the critical path: layer output and what BPTT needs
                const int gn = grp * NB + half * HB + n;
                if (gn < N) {
                    const size_t o = (static_cast<size_t>(tt) * N + gn) * H2 + static_cast<size_t>(dir) * H + j * 32 + u;
                    p.hout[o] = h;
                    if (p.c_save) p.c_save[o] = cn;
                    if (p.gates_save) {
                        __half2 lo = __floats2half2_rn(gi, gf), hi = __floats2half2_rn(gg, go);
                        p.gates_save[o] = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
                    }
                }
                if (warp == 0 && half == 0) PTRACE(5);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// backward (BPTT)
// ------------------------------------------------------------------------------------------------
struct BwdParams {
    const float* dhout;        // [T*N, 2H] gradient w.r.t. the layer output
    const float* c_save;       // [T*N, 2H]
    const uint2* gates_save;   // [T*N, 2H] 4 x fp16
    const float4* gates_save32;  // split-operand mode: 4 x fp32 instead
    __nv_bfloat16* dg;         // [T*N, 8H] gate gradients, packed column order (A operand of the dX GEMM); hi part in X3 mode
    __nv_bfloat16* dg_lo;      // X3: the lo part of the same
    __nv_bfloat16* dg_rec;     // GRU: gate gradients as the RECURRENT weights see them (n slot = dn_pre * r), for dW_hh; hi part
    __nv_bfloat16* dg_rec_lo;  // GRU + X3: lo part
    int rnn_relu;              // CELL_RNN: 1 = relu, 0 = tanh
    __nv_bfloat16* dgimg;      // EX = 0: [2 dirs][groups][4 gates][2][H*NB*PARTS] operand images
    unsigned int* flags;       // EX = 0: [2 dirs][groups]
    int T, N, H, groups, n0;
    const __nv_bfloat16* w;    // packed transposed recurrent weights [8H, H] (hi part)
    int mma_split;
    long long* trace;          // optional [T][16] clock64 stamps of CTA 0 / thread 0 (CTCB200_LSTM_TRACE)
    unsigned int* resident;    // optional uint32[2]: [0] += 1 once every CTA of this launch is running ([1] = arrivals)
    // Streamed gate gradients (optional): every CTA adds 1 to *progress once its dG rows of the scan steps [c*chunk_T,
    // (c+1)*chunk_T) are written and visible (c = 0, 1, ...; also after the last, possibly shorter, chunk), so another stream can
    // run the input-gradient / weight-gradient GEMMs of a chunk (stream memory-operation wait on the counter) while the
    // recurrence is still going: forward scan of BPTT = rows T-1-s, reverse scan = rows s.
    unsigned int* progress;
    int chunk_T;
    const float* bn_x;         // optional: layer output [T*N, 2H]; the BatchNorm backward of the layer above is applied to
    const float* bn_coef;      // dhout on the fly: dh = coef[0][c]*dhout + coef[1][c]*bn_x + coef[2][c], coef f32 [3][2H]
};


// Streamed gate gradients: called by every thread at the end of scan step t, after its dG stores of that step.
__device__ __forceinline__ void publish_dg_chunk(const BwdParams& p, int t, int T, int& next_pub) {
    if (p.progress != nullptr && (t + 1 == next_pub || t + 1 == T)) {
        __threadfence();          // this thread's dG rows are visible device-wide ...
        __syncthreads();          // ... for every thread of the CTA ...
        if (threadIdx.x == 0) red_release_add(p.progress, 1u);   // ... before the chunk is counted
        next_pub += p.chunk_T;
    }
}

// BatchNorm-backward coefficients of column c (identity when the fusion is off)
struct BnCoef { float a, b, d; };
__device__ __forceinline__ BnCoef load_bn_coef(const BwdParams& p, int c) {
    BnCoef k{1.0f, 0.0f, 0.0f};
    if (p.bn_x != nullptr) {
        k.a = __ldg(p.bn_coef + c);
        k.b = __ldg(p.bn_coef + 2 * p.H + c);
        k.d = __ldg(p.bn_coef + 4 * p.H + c);
    }
    return k;
}

// CTA (mb, q) keeps the [128 units x H] slice of gate q's transposed recurrent block. Per BPTT step:
//   partial dh[128, NB] = slice * dG_q  ->  reduce-scatter of the 4 gate partials inside the (4,*) cluster row
//   -> 32 finished units per CTA -> LSTM cell backward -> the four dG chunks go to the next step's operands.
// EX = 3: the whole (direction, group) = 4 x H/128 CTAs is one cluster; partial rows and dG blocks travel as bulk DSMEM
//         copies with complete_tx on the receiver's mbarrier (partials as fp16, or fp32 in X3 mode).
// EX = 0: cluster of the 4 gate CTAs only; dG images + release/acquire counter in global memory (any H).
// X3    : split-operand mode as in the forward kernel: W^T = hi (TMEM) + lo (shared memory), dG = hi + lo blocks.
template <int NB, int EX, bool X3, int CELL = CELL_LSTM>
__global__ void __launch_bounds__(LSTM_THREADS, 1)
lstm_bwd_kernel(const __grid_constant__ CUtensorMap tmWTlo, BwdParams p) {
    constexpr bool CL = EX != 0, BULK = EX == 3;
    constexpr int PARTS = X3 ? 2 : 1;
    constexpr uint32_t BLK_BYTES = NB * 64;
    constexpr uint32_t BLK_STRIDE = PARTS * BLK_BYTES;
    constexpr int CPT = NB / 2;
    constexpr int EPT = NB / 8;
    constexpr int OUT_CHUNKS = NB * 4;
    constexpr uint32_t PART_BYTES = X3 ? 4 : 2;   // width of one partial-dh element on the wire (BULK)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int H = p.H, T = p.T, N = p.N;
    const int img_bytes = H * NB * 2 * PARTS;
    constexpr bool SPILL = EX == 0 && !X3;                            // H > TMEM_K_MAX possible (see TMEM_K_MAX)
    const int k_tmem = (SPILL && H > TMEM_K_MAX) ? TMEM_K_MAX : H;    // K elements of the W^T slice resident in TMEM
    const int kb_tmem = k_tmem / 64;
    uint8_t* sW = smem;                                               // X3: the W^T_lo slice [128 x H] bf16; SPILL: K >= k_tmem
    uint8_t* sB = sW + (X3 ? 128 * H * 2 : (SPILL ? 128 * (H - k_tmem) * 2 : 0));   // BULK: two parities, else one buffer
    float* sR = reinterpret_cast<float*>(sB + (BULK ? 2 : 1) * img_bytes);  // [4 src][NB][32] partial dh blocks
    uint4* sOut = reinterpret_cast<uint4*>(sR + 4 * NB * 32);         // BULK only: [4 gates][PARTS][OUT_CHUNKS]
    float* sP = reinterpret_cast<float*>(sOut + (BULK ? 4 * PARTS * OUT_CHUNKS : 0));  // BULK only: [4 dst][NB][32] partial staging
    uint64_t* bars = reinterpret_cast<uint64_t*>(sP + (BULK ? 4 * NB * 32 : 0));
    uint64_t* w_full = bars;
    uint64_t* acc_full = bars + 1;
    uint64_t* r_full = bars + 2;   // BULK: the 4 partial blocks of a step have landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
    constexpr bool KBB = BULK && X3;               // X3: one barrier per K block of the dG image (see exchange_peer)
    constexpr bool PRE = BULK && CELL == CELL_LSTM; // cell-backward factors that do not need the recurrent dh are computed early
    constexpr int HB_STRIDE = KBB ? MAX_KB : 1;
    uint64_t* b_full = bars + 4;   // [parity * HB_STRIDE + kb]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    announce_resident(p.resident);
    const int q = blockIdx.x;   // gate handled by this CTA
    const int mb = blockIdx.y;  // block of 128 hidden units
    const int MB = gridDim.y;
    const int dir = blockIdx.z / p.groups, grp = blockIdx.z % p.groups;
    const int ctas = 4 * MB;
    const int kblocks = H / 64;
    // rank inside the cluster: CL -> x + 4*y (cluster spans the whole (4, MB) plane), else x
    auto rank_of = [&](int qq, int mm) -> uint32_t { return static_cast<uint32_t>(CL ? qq + 4 * mm : qq); };

    if (tid == 0) {
        if constexpr (X3) tma_prefetch_desc(&tmWTlo);
        mbar_init(w_full, 1);
        for (int i = 0; i < 2 * HB_STRIDE; ++i) mbar_init(&b_full[i], BULK ? 1 : LSTM_THREADS);
        mbar_init(acc_full, p.mma_split);
        mbar_init(r_full, 1);
        fence_mbar_init();
        if constexpr (BULK) {
            for (int i = 0; i < 2 * HB_STRIDE; ++i) mbar_expect_tx(&b_full[i], (KBB ? 2 : ctas) * BLK_STRIDE);
            mbar_expect_tx(r_full, 4 * NB * 32 * PART_BYTES);  // four gate partials of [NB][32] values per step
        }
    }
    uint32_t tmem_cols = 64;
    while (tmem_cols < 64u + k_tmem / 2) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    if constexpr (BULK) {
        for (int i = tid; i < img_bytes / 16; i += LSTM_THREADS) reinterpret_cast<uint4*>(sB)[i] = make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();  // every CTA of the cluster has its barriers / receive buffers ready

    // rows of the transposed gate block: (dir, q, unit); this CTA takes units [128 mb, +128)
    if (warp < 4)
        load_weights_to_tmem(p.w + (static_cast<size_t>(dir * 4 + q) * H + mb * 128) * H, k_tmem, tmem_base, 64, warp, lane,
                             SPILL ? H : 0);
    if constexpr (X3) {
        if (tid == 0) {
            mbar_expect_tx(w_full, 128 * H * 2);
            for (int kb = 0; kb < kblocks; ++kb)
                tma_load_2d(sW + kb * 16384, &tmWTlo, w_full, kb * 64, (dir * 4 + q) * H + mb * 128);
        }
    }
    if constexpr (SPILL) {   // (tmWTlo maps the W^T_hi image here)
        if (tid == 0 && k_tmem < H) {
            mbar_expect_tx(w_full, 128 * (H - k_tmem) * 2);
            for (int kb = kb_tmem; kb < kblocks; ++kb)
                tma_load_2d(sW + (kb - kb_tmem) * 16384, &tmWTlo, w_full, kb * 64, (dir * 4 + q) * H + mb * 128);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int lq = warp & 3, ch = warp >> 2;
    const bool warp_leader = elect_one();
    const int unit = mb * 128 + q * 32 + lane;  // the unit this thread finishes in the element phase
    const BnCoef bnk = load_bn_coef(p, dir * H + unit);
    const size_t H2 = static_cast<size_t>(2) * H, G8 = static_cast<size_t>(8) * H;
    const size_t dg_col = static_cast<size_t>(dir) * 4 * H + static_cast<size_t>(unit >> 5) * 128 + (unit & 31) * 4;
    __nv_bfloat16* imgs = BULK ? nullptr : p.dgimg + (static_cast<size_t>(dir) * p.groups + grp) * 4 * 2 * H * NB * PARTS;
    unsigned int* flag = CL ? nullptr : p.flags + (dir * p.groups + grp) * 32;
    const int chunks = H * NB / 8 * PARTS;
    constexpr uint32_t idesc = umma_idesc_bf16(128, NB);
    // remote receive slot: partial block from source gate q lands in the CTA that owns rows 32 lq.. of this unit block
    const uint32_t remote_base = mapa_shared(smem_u32(sR + (q * NB + ch * CPT) * 32 + lane), rank_of(lq, mb));

    float dc_carry[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) dc_carry[e] = 0.0f;

#define BTRACE(k) do { if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && tid == 0) p.trace[t * 16 + (k)] = clock64(); } while (0)
    int next_pub = p.chunk_T;   // streamed gate gradients: scan step count that completes the next chunk
    for (int t = 0; t < T; ++t) {
        const int tt = dir ? t : (T - 1 - t);          // reverse of the forward scan order
        BTRACE(0);
        const int tprev = dir ? tt + 1 : tt - 1;       // time index that held c_{prev} in the forward scan
        const bool has_prev = dir ? (tt + 1 < T) : (tt >= 1);
        // (1) saved activations and the incoming gradient for this thread's elements
        // NOTHING loaded here may be touched before phase (6): these loads are issued ahead of the MMA chain so that their
        // latency hides behind it (a conversion at the load site would stall the issuing warps on the load every step)
        float dh_in[EPT], bx_in[EPT], c_t[EPT], c_p[EPT];
        float pre_dh[PRE ? EPT : 1], k_o[PRE ? EPT : 1], k_c[PRE ? EPT : 1], k_i[PRE ? EPT : 1], k_f[PRE ? EPT : 1], k_g[PRE ? EPT : 1],
            k_carry[PRE ? EPT : 1];   // LSTM cluster kernels: cell-backward factors computed while the partials are in flight
        float4 gts32[X3 ? EPT : 1];
        uint2 gts16[X3 ? 1 : EPT];
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int gn = p.n0 + grp * NB + warp + 8 * e;
            const bool ok = gn < N;
            const size_t o = (static_cast<size_t>(tt) * N + (ok ? gn : 0)) * H2 + static_cast<size_t>(dir) * H + unit;
            dh_in[e] = ok ? __ldg(p.dhout + o) : 0.0f;
            bx_in[e] = (p.bn_x != nullptr && ok) ? __ldg(p.bn_x + o) : 0.0f;   // combined with dh_in where it is consumed
            c_t[e] = ok ? __ldg(p.c_save + o) : 0.0f;
            if constexpr (X3) gts32[e] = ok ? __ldg(p.gates_save32 + o) : make_float4(0.f, 0.f, 0.f, 0.f);
            else gts16[e] = ok ? __ldg(p.gates_save + o) : make_uint2(0u, 0u);
            const size_t op = (static_cast<size_t>(has_prev ? tprev : tt) * N + (ok ? gn : 0)) * H2 +
                              static_cast<size_t>(dir) * H + unit;
            c_p[e] = (ok && has_prev) ? __ldg(p.c_save + op) : 0.0f;
        }
        if constexpr (!BULK) {
            // (2) gate gradients of the previous BPTT step are published
            if (lane == 0) wait_counter(flag, static_cast<unsigned int>(ctas) * t);
            __syncwarp();
            // (3) dG image of gate q -> shared memory
            const uint4* src = reinterpret_cast<const uint4*>(imgs + (static_cast<size_t>(q) * 2 + (t & 1)) * H * NB * PARTS);
            uint4* dst = reinterpret_cast<uint4*>(sB);
            for (int i = tid; i < chunks; i += LSTM_THREADS) dst[i] = ld_cg_v4(src + i);
            fence_proxy_async_smem();
            mbar_arrive(&b_full[0]);
        }
        // (4) partial dh[128 units, NB] = W_q^T slice * dG_q (issued like the forward kernel's chain)
        if (warp < p.mma_split) {
            if constexpr (X3) { if (t == 0) mbar_wait(w_full, 0); }
            if constexpr (SPILL) { if (t == 0 && k_tmem < H) mbar_wait(w_full, 0); }
            if constexpr (KBB) {
                // per-K-block waits inside the loop; the issuing warps took part in last step's CTA barriers themselves
            } else if constexpr (BULK) {
                if (t > 0) {
                    mbar_wait(&b_full[t & 1], ((t - 1) >> 1) & 1);
                    if (lane == 0 && warp == 0) mbar_expect_tx(&b_full[t & 1], ctas * BLK_STRIDE);
                }
            } else {
                mbar_wait(&b_full[0], t & 1);
            }
            tc_fence_after();
            BTRACE(1);
            const uint32_t a0 = smem_u32(sW), b0 = smem_u32(sB) + (BULK ? (t & 1) * img_bytes : 0);
            const bool leader = elect_one();
            const int kstep = p.mma_split, kfirst = warp;
            const uint32_t dacc = tmem_base + warp * NB;
            constexpr uint32_t B2 = BLK_STRIDE / 16, LO = BLK_BYTES / 16;
#pragma unroll 1
            for (int it = kfirst; it < kblocks; it += kstep) {
                const int kb = KBB ? arrival_kblock(q + 4 * mb, it, kblocks) : it;   // X3: K blocks in their arrival order
                if constexpr (KBB) {
                    if (t > 0) {
                        uint64_t* kf = &b_full[(t & 1) * HB_STRIDE + kb];
                        mbar_wait(kf, ((t - 1) >> 1) & 1);                    // both source blocks of this K block have landed
                        if (lane == 0) mbar_expect_tx(kf, 2 * BLK_STRIDE);    // re-arm for step t + 2 (this warp owns kb)
                    }
                }
                // 64 K elements = two SWIZZLE_64B blocks of the B image, two K=16 slices (32 bytes apart) in each
                const uint64_t bd = umma_desc_sw64(b0 + kb * (2 * BLK_STRIDE));
                const uint32_t ta = tmem_base + 64 + kb * 32;
                if (SPILL && kb >= kb_tmem) {   // this K block of W^T sits in shared memory
                    const uint64_t ad = umma_desc_sw128(a0 + (kb - kb_tmem) * 16384);
                    if (leader) {
                        umma_bf16(dacc, ad, bd, idesc, it != kfirst ? 1u : 0u);
                        umma_bf16(dacc, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(dacc, ad + 4, bd + B2, idesc, 1u);
                        umma_bf16(dacc, ad + 6, bd + B2 + 2, idesc, 1u);
                    }
                } else if (leader) {
                    umma_bf16_ts(dacc, ta, bd, idesc, it != kfirst ? 1u : 0u);
                    umma_bf16_ts(dacc, ta + 8, bd + 2, idesc, 1u);
                    umma_bf16_ts(dacc, ta + 16, bd + B2, idesc, 1u);
                    umma_bf16_ts(dacc, ta + 24, bd + B2 + 2, idesc, 1u);
                }
                if constexpr (X3) {
                    const uint64_t ad = umma_desc_sw128(a0 + kb * 16384);
                    if (leader) {
                        umma_bf16_ts(dacc, ta, bd + LO, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 8, bd + LO + 2, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 16, bd + B2 + LO, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 24, bd + B2 + LO + 2, idesc, 1u);
                        umma_bf16(dacc, ad, bd, idesc, 1u);
                        umma_bf16(dacc, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(dacc, ad + 4, bd + B2, idesc, 1u);
                        umma_bf16(dacc, ad + 6, bd + B2 + 2, idesc, 1u);
                    }
                }
            }
            if (leader) umma_commit(acc_full);
            BTRACE(2);
        }
        __syncwarp();
        // (5) scatter the partial rows to their owner CTA through distributed shared memory
        mbar_wait(acc_full, t & 1);
        tc_fence_after();
        BTRACE(3);
        uint32_t acc[CPT];
        load_partial_sums<CPT>(tmem_base + (static_cast<uint32_t>(lq * 32) << 16) + ch * CPT, NB, p.mma_split, acc);
        tc_fence_before();
        BTRACE(4);
        if constexpr (BULK) {
            // every warp holds the [NB/2][32] sub-block of partial rows that belongs to CTA (lq, mb): stage it, then
            // one bulk copy per warp into that CTA's receive slot for source gate q (complete_tx on its r_full)
            if (warp_leader) bulk_wait_read_all();  // this warp's earlier copies have finished reading shared memory
            __syncthreads();                         // ... for every warp: sP and sOut may be rewritten
            // bf16 mode: partials cross the cluster as fp16 (less DSMEM traffic; the four partials are summed in fp32 on
            // arrival, so the rounding stays far below that of the bf16 operands); X3 mode: fp32 on the wire
            const int pe = (lq * NB + ch * CPT) * 32, re = (q * NB + ch * CPT) * 32;   // element offsets in sP / the peer's sR
            if constexpr (X3) {
#pragma unroll
                for (int c = 0; c < CPT; ++c) sP[pe + c * 32 + lane] = __uint_as_float(acc[c]);
            } else {
                __half* stage = reinterpret_cast<__half*>(sP) + pe + lane;
#pragma unroll
                for (int c = 0; c < CPT; ++c) stage[c * 32] = __float2half_rn(__uint_as_float(acc[c]));
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (warp_leader) {
                const uint32_t peer = rank_of(lq, mb);
                bulk_copy_to_peer(mapa_shared(smem_u32(sR) + re * PART_BYTES, peer), smem_u32(sP) + pe * PART_BYTES,
                                  CPT * 32 * PART_BYTES, mapa_shared(smem_u32(r_full), peer));
                bulk_commit();
            }
            BTRACE(5);
            if constexpr (PRE) {
                // while the partials are in flight: everything of the cell backward that does not depend on the recurrent dh
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    pin_reg(dh_in[e]); pin_reg(bx_in[e]); pin_reg(c_t[e]); pin_reg(c_p[e]);
                    float gi, gf, gg, go;
                    if constexpr (X3) {
                        pin_reg(gts32[e].x); pin_reg(gts32[e].y); pin_reg(gts32[e].z); pin_reg(gts32[e].w);
                        gi = gts32[e].x; gf = gts32[e].y; gg = gts32[e].z; go = gts32[e].w;
                    } else {
                        pin_reg(gts16[e].x); pin_reg(gts16[e].y);
                        const __half2 glo = *reinterpret_cast<const __half2*>(&gts16[e].x), ghi = *reinterpret_cast<const __half2*>(&gts16[e].y);
                        gi = __low2float(glo); gf = __high2float(glo); gg = __low2float(ghi); go = __high2float(ghi);
                    }
                    const float tc = fast_tanh(c_t[e]);
                    pre_dh[e] = bnk.a * dh_in[e] + bnk.b * bx_in[e] + ((p.n0 + grp * NB + warp + 8 * e < N) ? bnk.d : 0.0f);
                    k_o[e] = tc * go * (1.0f - go);
                    k_c[e] = go * (1.0f - tc * tc);
                    k_i[e] = gg * gi * (1.0f - gi);
                    k_f[e] = c_p[e] * gf * (1.0f - gf);
                    k_g[e] = gi * (1.0f - gg * gg);
                    k_carry[e] = gf;
                }
            }
            mbar_wait(r_full, t & 1);
            BTRACE(6);
            if (tid == 0) mbar_expect_tx(r_full, 4 * NB * 32 * PART_BYTES);  // re-arm for the next step
        } else {
#pragma unroll
            for (int c = 0; c < CPT; ++c) st_cluster_f32(remote_base + c * 32 * 4, __uint_as_float(acc[c]));
            cluster_sync_all();
        }
        // (6) finish 32 units: recurrent dh, LSTM cell backward, publish the four gate gradients
        if constexpr (!PRE) {
#pragma unroll
            for (int e = 0; e < EPT; ++e) {   // keep all arithmetic on the values prefetched in (1) below the waits (see pin_reg)
                pin_reg(dh_in[e]); pin_reg(bx_in[e]); pin_reg(c_t[e]); pin_reg(c_p[e]);
                if constexpr (X3) { pin_reg(gts32[e].x); pin_reg(gts32[e].y); pin_reg(gts32[e].z); pin_reg(gts32[e].w); }
                else { pin_reg(gts16[e].x); pin_reg(gts16[e].y); }
            }
        }
        uint2 dgp[EPT], dgl[EPT];
        uint2 dgr[CELL == CELL_GRU ? EPT : 1], dgrl[CELL == CELL_GRU ? EPT : 1];   // GRU: input-side gate gradients (see below)
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int n = warp + 8 * e;
            float dh;
            if constexpr (PRE) dh = pre_dh[e];
            else dh = bnk.a * dh_in[e] + bnk.b * bx_in[e] + ((p.n0 + grp * NB + n < N) ? bnk.d : 0.0f);   // BatchNorm backward on the fly
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                if constexpr (BULK && !X3) dh += __half2float(reinterpret_cast<const __half*>(sR)[(s * NB + n) * 32 + lane]);
                else dh += sR[(s * NB + n) * 32 + lane];
            }
            float gi = 0.0f, gf = 0.0f, gg = 0.0f, go = 0.0f;
            if constexpr (PRE) {
            } else if constexpr (X3) {
                gi = gts32[e].x; gf = gts32[e].y; gg = gts32[e].z; go = gts32[e].w;
            } else {
                const __half2 glo = *reinterpret_cast<const __half2*>(&gts16[e].x), ghi = *reinterpret_cast<const __half2*>(&gts16[e].y);
                gi = __low2float(glo); gf = __high2float(glo); gg = __low2float(ghi); go = __high2float(ghi);
            }
            float d_i, d_f, d_g, d_o;     // the four slots handed to the next BPTT step (what W_hh^T multiplies)
            if constexpr (PRE) {
                d_o = dh * k_o[e];
                const float dc = dc_carry[e] + dh * k_c[e];
                d_i = dc * k_i[e];
                d_f = dc * k_f[e];
                d_g = dc * k_g[e];
                dc_carry[e] = dc * k_carry[e];
            } else if constexpr (CELL == CELL_LSTM) {
                const float tc = fast_tanh(c_t[e]);
                d_o = dh * tc * go * (1.0f - go);
                const float dc = dc_carry[e] + dh * go * (1.0f - tc * tc);
                d_i = dc * gg * gi * (1.0f - gi);
                d_f = dc * c_p[e] * gf * (1.0f - gf);
                d_g = dc * gi * (1.0f - gg * gg);
                dc_carry[e] = dc * gf;
            } else if constexpr (CELL == CELL_GRU) {
                // saved slots (r, z, n, hn = W_hn h_prev); c_p = h_prev. h' = (1 - z) n + z h_prev, n = tanh(gx_n + r hn)
                dh += dc_carry[e];                             // the direct path h' -> h_prev of the step before
                const float dn_pre = dh * (1.0f - gf) * (1.0f - gg * gg);
                d_i = dn_pre * go * gi * (1.0f - gi);          // r gate
                d_f = dh * (c_p[e] - gg) * gf * (1.0f - gf);   // z gate
                d_g = dn_pre * gi;                             // what reaches W_hn: dn_pre * r
                d_o = 0.0f;
                dc_carry[e] = dh * gf;
                // the INPUT weights see dn_pre itself in the n slot: second set of rows for dX / dW_ih
                __nv_bfloat16 ih[4], il[4];
                split_bf16(d_i, ih[0], il[0]);
                split_bf16(d_f, ih[1], il[1]);
                split_bf16(dn_pre, ih[2], il[2]);
                ih[3] = il[3] = __float2bfloat16(0.0f);
                __nv_bfloat162 a01, a23;
                a01.x = ih[0]; a01.y = ih[1]; a23.x = ih[2]; a23.y = ih[3];
                dgr[e] = make_uint2(*reinterpret_cast<uint32_t*>(&a01), *reinterpret_cast<uint32_t*>(&a23));
                if constexpr (X3) {
                    a01.x = il[0]; a01.y = il[1]; a23.x = il[2]; a23.y = il[3];
                    dgrl[e] = make_uint2(*reinterpret_cast<uint32_t*>(&a01), *reinterpret_cast<uint32_t*>(&a23));
                }
            } else {
                // saved slot 0 = h_t; h' = tanh(pre) or relu(pre)
                d_i = p.rnn_relu ? (gi > 0.0f ? dh : 0.0f) : dh * (1.0f - gi * gi);
                d_f = d_g = d_o = 0.0f;
            }
            __nv_bfloat16 hi4[4], lo4[4];
            split_bf16(d_i, hi4[0], lo4[0]);
            split_bf16(d_f, hi4[1], lo4[1]);
            split_bf16(d_g, hi4[2], lo4[2]);
            split_bf16(d_o, hi4[3], lo4[3]);
            if constexpr (BULK) {
                // destination order inside each gate's block; one bf16 store per gate (and part) and lane
                __nv_bfloat16* so = reinterpret_cast<__nv_bfloat16*>(sOut) + n * 32 +
                                    (((lane >> 3) ^ ((n >> 1) & 3)) << 3) + (lane & 7);
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    so[g * PARTS * OUT_CHUNKS * 8] = hi4[g];
                    if constexpr (X3) so[(g * PARTS + 1) * OUT_CHUNKS * 8] = lo4[g];
                }
            } else {
                const int off = image_chunk_offset<NB, PARTS>(unit, n);
                const size_t nxt = static_cast<size_t>((t + 1) & 1) * H * NB * PARTS;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const uint4 ph = pack8_bf16(__bfloat162float(hi4[g]));
                    __nv_bfloat16* dst = imgs + (static_cast<size_t>(g) * 2) * H * NB * PARTS + nxt + off;
                    if ((lane & 7) == 0) *reinterpret_cast<uint4*>(dst) = ph;
                    if constexpr (X3) {
                        const uint4 pl = pack8_bf16(__bfloat162float(lo4[g]));
                        if ((lane & 7) == 0) *reinterpret_cast<uint4*>(dst + NB * 32) = pl;
                    }
                }
            }
            __nv_bfloat162 b01, b23;
            b01.x = hi4[0]; b01.y = hi4[1]; b23.x = hi4[2]; b23.y = hi4[3];
            dgp[e] = make_uint2(*reinterpret_cast<uint32_t*>(&b01), *reinterpret_cast<uint32_t*>(&b23));
            if constexpr (X3) {
                __nv_bfloat162 l01, l23;
                l01.x = lo4[0]; l01.y = lo4[1]; l23.x = lo4[2]; l23.y = lo4[3];
                dgl[e] = make_uint2(*reinterpret_cast<uint32_t*>(&l01), *reinterpret_cast<uint32_t*>(&l23));
            }
        }
        BTRACE(7);
        if constexpr (BULK) {
            fence_proxy_async_smem();
            __syncthreads();
            BTRACE(8);
            if (t + 1 < T) {
                // copy i = (g, mdst): gate g's block [hi | lo] of this CTA's 32 units -> slot (4 mb + q) of CTA (g, mdst)'s
                // buffer; warp w issues copies w and w + 8
                const int me = 4 * mb + q;   // this CTA's slot in every receiver's image (= its cluster rank)
                const uint32_t dst = smem_u32(sB) + ((t + 1) & 1) * img_bytes + me * BLK_STRIDE;
                const uint32_t bar = smem_u32(&b_full[((t + 1) & 1) * HB_STRIDE + (KBB ? (me >> 1) : 0)]);
                {
#pragma unroll
                    for (int i = warp; i < 16; i += 8) {
                        // receiver rank = gate + 4 * unit block; X3: rotated order (exchange_peer)
                        const uint32_t peer = KBB ? exchange_peer(me, i, ctas) : rank_of(i & 3, i >> 2);
                        const int g = peer & 3;
                        if (i < ctas && warp_leader) {
                            bulk_copy_to_peer(mapa_shared(dst, peer), smem_u32(sOut + g * PARTS * OUT_CHUNKS), BLK_STRIDE,
                                              mapa_shared(bar, peer));
                        }
                    }
                }
                if (warp_leader) bulk_commit();
            }
            BTRACE(9);
        } else {
            __threadfence();
            __syncthreads();
            if (tid == 0) red_release_add(flag, 1u);
        }
        // (7) off the critical path: dG rows for the dX / dW GEMMs
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int gn = p.n0 + grp * NB + warp + 8 * e;
            if (gn < N) {
                const size_t go_ = (static_cast<size_t>(tt) * N + gn) * G8 + dg_col;
                if constexpr (CELL == CELL_GRU) {
                    // dg = what the input weights see (dX, dW_ih), dg_rec = what the recurrent weights see (dW_hh)
                    *reinterpret_cast<uint2*>(p.dg + go_) = dgr[e];
                    *reinterpret_cast<uint2*>(p.dg_rec + go_) = dgp[e];
                    if constexpr (X3) {
                        *reinterpret_cast<uint2*>(p.dg_lo + go_) = dgrl[e];
                        *reinterpret_cast<uint2*>(p.dg_rec_lo + go_) = dgl[e];
                    }
                } else {
                    *reinterpret_cast<uint2*>(p.dg + go_) = dgp[e];
                    if constexpr (X3) *reinterpret_cast<uint2*>(p.dg_lo + go_) = dgl[e];
                }
            }
        }
        publish_dg_chunk(p, t, T, next_pub);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA exits while a peer may still address its shared memory
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// ================================================================================================
// Two-tile variants for H > 512 (cfg4: H = 640). H/32 CTAs would not fit one cluster (max 16), so every CTA owns
// 64 hidden units = two 128-row gate tiles: tile 0's weights are resident in TMEM, tile 1's in shared memory
// (TMA-loaded, SWIZZLE_128B); four warps issue the two MMA chains (two per tile, split accumulators). The H/64
// CTAs of a (direction, batch group) form one cluster and exchange h_t with bulk DSMEM copies exactly as above.
// ================================================================================================
template <int NB>
__global__ void __launch_bounds__(LSTM_THREADS, 1)
lstm_fwd2_kernel(const __grid_constant__ CUtensorMap tmW, FwdParams p) {
    constexpr uint32_t BLK_BYTES = NB * 64;
    constexpr int CPT = NB / 2, EPT = NB / 8, S_STRIDE = NB * 4 + 4, OUT_CHUNKS = NB * 4;
    static_assert(4 * NB <= 64, "four split accumulators must fit the 64 accumulator columns");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int H = p.H, T = p.T, N = p.N;
    const int himg_bytes = H * NB * 2;
    uint8_t* sW1 = smem;                                              // tile 1 weights [128 x H] bf16
    uint8_t* sH = sW1 + 128 * H * 2;                                  // two operand buffers
    float* sS = reinterpret_cast<float*>(sH + 2 * himg_bytes);        // [2 tiles][32 units][S_STRIDE]
    uint4* sOut = reinterpret_cast<uint4*>(sS + 2 * 32 * S_STRIDE);   // [2 tiles][OUT_CHUNKS]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + 2 * OUT_CHUNKS);
    uint64_t* w_full = bars;
    uint64_t* h_full = bars + 1;  // [2]
    uint64_t* acc_full = bars + 3;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int j = blockIdx.x, dir = blockIdx.y, grp = blockIdx.z;
    const int ctas = gridDim.x;
    const int kblocks = H / 64;
    announce_resident(p.resident);

    if (tid == 0) {
        tma_prefetch_desc(&tmW);
        mbar_init(w_full, 1);
        mbar_init(&h_full[0], 1);
        mbar_init(&h_full[1], 1);
        mbar_init(acc_full, 4);
        fence_mbar_init();
        mbar_expect_tx(&h_full[0], ctas * 2 * BLK_BYTES);
        mbar_expect_tx(&h_full[1], ctas * 2 * BLK_BYTES);
    }
    uint32_t tmem_cols = 64;
    while (tmem_cols < 64u + H / 2) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    for (int i = tid; i < himg_bytes / 16; i += LSTM_THREADS) reinterpret_cast<uint4*>(sH)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();

    const size_t row0 = static_cast<size_t>(dir) * 4 * H + static_cast<size_t>(2 * j) * 128;  // packed rows of tile 0
    if (warp < 4) load_weights_to_tmem(p.w + row0 * H, H, tmem_base, 64, warp, lane);
    if (tid == 0) {
        mbar_expect_tx(w_full, 128 * H * 2);
        for (int kb = 0; kb < kblocks; ++kb) tma_load_2d(sW1 + kb * 16384, &tmW, w_full, kb * 64, static_cast<int>(row0) + 128);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int lq = warp & 3, ch = warp >> 2;
    const bool warp_leader = elect_one();
    const int row = lq * 32 + lane;
    const int u_loc = row >> 2, q = row & 3;
    const float act_s = (q == 2) ? 2.0f : 1.0f;
    const size_t gx_col = row0 + row;
    const size_t G8 = static_cast<size_t>(8) * H, H2 = static_cast<size_t>(2) * H;
    constexpr uint32_t idesc = umma_idesc_bf16(128, NB);

    float c_state[2][EPT];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < EPT; ++e) c_state[u][e] = 0.0f;

    int gx_gate = p.chunk_T;   // streamed input projection: first scan step of the next chunk
    for (int t = 0; t < T; ++t) {
        const int tt = dir ? (T - 1 - t) : t;
        if (p.gx_ready != nullptr && t == gx_gate) {
            if (lane == 0) wait_gx_chunk(p.gx_ready, p.gx_base + static_cast<unsigned int>(t / p.chunk_T));
            __syncwarp();
            gx_gate += p.chunk_T;
        }
        float gx[2][CPT];
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
            const int gn = p.n0 + grp * NB + ch * CPT + c;
            const float* g = p.gx + (static_cast<size_t>(tt) * N + (gn < N ? gn : 0)) * G8 + gx_col;
            gx[0][c] = (gn < N) ? load_gx(p, g) : 0.0f;
            gx[1][c] = (gn < N) ? load_gx(p, g + 128) : 0.0f;
        }
        if (warp < 4) {
            const int u = warp >> 1, slot = warp & 1;
            if (t == 0 && u == 1) mbar_wait(w_full, 0);
            if (t > 0) {
                mbar_wait(&h_full[t & 1], ((t - 1) >> 1) & 1);
                if (lane == 0 && warp == 0) mbar_expect_tx(&h_full[t & 1], ctas * 2 * BLK_BYTES);
            }
            tc_fence_after();
            const uint32_t a0 = smem_u32(sW1), b0 = smem_u32(sH) + (t & 1) * himg_bytes;
            const uint32_t dacc = tmem_base + warp * NB;
            const bool leader = elect_one();
#pragma unroll 1
            for (int kb = slot; kb < kblocks; kb += 2) {
                const uint64_t bd = umma_desc_sw64(b0 + kb * (NB * 128));
                if (u == 0) {
                    const uint32_t ta = tmem_base + 64 + kb * 32;
                    if (leader) {
                        umma_bf16_ts(dacc, ta, bd, idesc, kb != slot ? 1u : 0u);
                        umma_bf16_ts(dacc, ta + 8, bd + 2, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 16, bd + (NB * 64 / 16), idesc, 1u);
                        umma_bf16_ts(dacc, ta + 24, bd + (NB * 64 / 16) + 2, idesc, 1u);
                    }
                } else {
                    const uint64_t ad = umma_desc_sw128(a0 + kb * 16384);
                    if (leader) {
                        umma_bf16(dacc, ad, bd, idesc, kb != slot ? 1u : 0u);
                        umma_bf16(dacc, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(dacc, ad + 4, bd + (NB * 64 / 16), idesc, 1u);
                        umma_bf16(dacc, ad + 6, bd + (NB * 64 / 16) + 2, idesc, 1u);
                    }
                }
            }
            if (leader) umma_commit(acc_full);
        }
        __syncwarp();
        mbar_wait(acc_full, t & 1);
        tc_fence_after();
        uint32_t acc[2][CPT];
        const uint32_t trow = tmem_base + (static_cast<uint32_t>(lq * 32) << 16) + ch * CPT;
        load_partial_sums<CPT>(trow, NB, 2, acc[0]);
        load_partial_sums<CPT>(trow + 2 * NB, NB, 2, acc[1]);
        tc_fence_before();
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int c = 0; c < CPT; ++c) {
                const float pre = __uint_as_float(acc[u][c]) + gx[u][c];
                sS[(u * 32 + u_loc) * S_STRIDE + (ch * CPT + c) * 4 + q] = act_s * fast_sigmoid(act_s * pre) - (act_s - 1.0f);
            }
        if (warp_leader) bulk_wait_read_all();
        __syncthreads();
        float hv[2][EPT];
        float4 gv[2][EPT];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int n = warp + 8 * e;
                const float4 g4 = *reinterpret_cast<const float4*>(&sS[(u * 32 + lane) * S_STRIDE + n * 4]);
                const float cn = g4.y * c_state[u][e] + g4.x * g4.z;
                c_state[u][e] = cn;
                const float h = g4.w * fast_tanh(cn);
                hv[u][e] = h;
                gv[u][e] = g4;
                reinterpret_cast<__nv_bfloat16*>(sOut)[u * OUT_CHUNKS * 8 + n * 32 + (((lane >> 3) ^ ((n >> 1) & 3)) << 3) +
                                                       (lane & 7)] = __float2bfloat16(h);
            }
        fence_proxy_async_smem();
        __syncthreads();
        if (t + 1 < T) {
            const uint32_t dst = smem_u32(sH) + ((t + 1) & 1) * himg_bytes + (2 * j) * BLK_BYTES;
            const uint32_t bar = smem_u32(&h_full[(t + 1) & 1]);
#pragma unroll
            for (int d = warp; d < 16; d += 8) {
                if (d < ctas && warp_leader)
                    bulk_copy_to_peer(mapa_shared(dst, static_cast<uint32_t>(d)), smem_u32(sOut), 2 * BLK_BYTES,
                                      mapa_shared(bar, static_cast<uint32_t>(d)));
            }
            if (warp_leader) bulk_commit();
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int gn = p.n0 + grp * NB + warp + 8 * e;
                if (gn < N) {
                    const size_t o = (static_cast<size_t>(tt) * N + gn) * H2 + static_cast<size_t>(dir) * H + j * 64 + u * 32 + lane;
                    p.hout[o] = hv[u][e];
                    if (p.c_save) p.c_save[o] = c_state[u][e];
                    if (p.gates_save) {
                        __half2 lo = __floats2half2_rn(gv[u][e].x, gv[u][e].y), hi = __floats2half2_rn(gv[u][e].z, gv[u][e].w);
                        p.gates_save[o] = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
                    }
                }
            }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// BPTT counterpart: CTA (qp, mb) owns the gate pair (2 qp, 2 qp + 1) for the 128 units of block mb and finishes 64 of
// them per step; cluster = (2, H/128). Gate a's transposed slice sits in TMEM, gate b's first 256 K columns too, the
// rest of gate b in shared memory; four warps issue the 2 * H/64 K blocks round-robin into split accumulators.
template <int NB>
__global__ void __launch_bounds__(LSTM_THREADS, 1)
lstm_bwd2_kernel(const __grid_constant__ CUtensorMap tmWT, BwdParams p) {
    constexpr uint32_t BLK_BYTES = NB * 64;
    constexpr int CPT = NB / 2, EPT = NB / 8, OUT_CHUNKS = NB * 4;
    static_assert(4 * NB <= 64, "four split accumulators must fit the 64 accumulator columns");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int H = p.H, T = p.T, N = p.N;
    const int img_bytes = H * NB * 2;
    const int kblocks = H / 64;
    constexpr int KB_TMEM_B = 4;                                      // K blocks of gate b that live in TMEM (256 columns of K)
    uint8_t* sW2 = smem;                                              // gate b, K columns [256, H): [128 x (H-256)] bf16
    uint8_t* sB = sW2 + 128 * (H - 64 * KB_TMEM_B) * 2;               // [2 local gates][2 buffers][H x NB] operand images
    float* sR = reinterpret_cast<float*>(sB + 4 * img_bytes);         // [2 src][2 halves][NB][32] partial dh blocks
    uint4* sOut = reinterpret_cast<uint4*>(sR + 4 * NB * 32);         // [4 gates][2 halves][OUT_CHUNKS]
    float* sP = reinterpret_cast<float*>(sOut + 8 * OUT_CHUNKS);      // [4 lane quarters][NB][32] partial staging
    uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 4 * NB * 32);
    uint64_t* w_full = bars;
    uint64_t* b_full = bars + 1;  // [2]
    uint64_t* acc_full = bars + 3;
    uint64_t* r_full = bars + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    announce_resident(p.resident);
    const int qp = blockIdx.x, mb = blockIdx.y, MB = gridDim.y;
    const int dir = blockIdx.z / p.groups, grp = blockIdx.z % p.groups;
    const int ctas = 2 * MB;
    auto rank_of = [&](int qq, int mm) -> uint32_t { return static_cast<uint32_t>(qq + 2 * mm); };

    if (tid == 0) {
        tma_prefetch_desc(&tmWT);
        mbar_init(w_full, 1);
        mbar_init(&b_full[0], 1);
        mbar_init(&b_full[1], 1);
        mbar_init(acc_full, 4);
        mbar_init(r_full, 1);
        fence_mbar_init();
        mbar_expect_tx(&b_full[0], 2 * img_bytes);
        mbar_expect_tx(&b_full[1], 2 * img_bytes);
        mbar_expect_tx(r_full, 4 * NB * 32 * 4);
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    for (int g = 0; g < 2; ++g)  // buffer 0 of both gate images starts zeroed (dG of "step -1")
        for (int i = tid; i < img_bytes / 16; i += LSTM_THREADS)
            reinterpret_cast<uint4*>(sB + (g * 2) * img_bytes)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();

    // transposed weight rows: (dir, gate, unit); gates 2qp (a) and 2qp+1 (b), units [128 mb, +128)
    const size_t row_a = (static_cast<size_t>(dir * 4 + 2 * qp) * H + mb * 128), row_b = row_a + H;
    const uint32_t col_a = 64, col_b = 64 + H / 2;
    if (warp < 4) {
        load_weights_to_tmem(p.w + row_a * H, H, tmem_base, col_a, warp, lane);
        load_weights_to_tmem(p.w + row_b * H, 64 * KB_TMEM_B, tmem_base, col_b, warp, lane, H);
    }
    if (tid == 0) {
        mbar_expect_tx(w_full, 128 * (H - 64 * KB_TMEM_B) * 2);
        for (int kb = KB_TMEM_B; kb < kblocks; ++kb)
            tma_load_2d(sW2 + (kb - KB_TMEM_B) * 16384, &tmWT, w_full, kb * 64, static_cast<int>(row_b));
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int lq = warp & 3, ch = warp >> 2;
    const bool warp_leader = elect_one();
    const size_t H2 = static_cast<size_t>(2) * H, G8 = static_cast<size_t>(8) * H;
    const int unit0 = mb * 128 + qp * 64 + lane;  // + 32 * half
    const BnCoef bnk2[2] = {load_bn_coef(p, dir * H + unit0), load_bn_coef(p, dir * H + unit0 + 32)};
    constexpr uint32_t idesc = umma_idesc_bf16(128, NB);

    float dc_carry[2][EPT];
#pragma unroll
    for (int hf = 0; hf < 2; ++hf)
#pragma unroll
        for (int e = 0; e < EPT; ++e) dc_carry[hf][e] = 0.0f;

    int next_pub = p.chunk_T;   // streamed gate gradients: scan step count that completes the next chunk
    for (int t = 0; t < T; ++t) {
        const int tt = dir ? t : (T - 1 - t);
        const int tprev = dir ? tt + 1 : tt - 1;
        const bool has_prev = dir ? (tt + 1 < T) : (tt >= 1);
        float dh_in[2][EPT], bx_in[2][EPT], c_t[2][EPT], c_p[2][EPT];
        uint2 gts[2][EPT];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf)
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int gn = p.n0 + grp * NB + warp + 8 * e;
                const bool ok = gn < N;
                const int unit = unit0 + 32 * hf;
                const size_t o = (static_cast<size_t>(tt) * N + (ok ? gn : 0)) * H2 + static_cast<size_t>(dir) * H + unit;
                dh_in[hf][e] = ok ? __ldg(p.dhout + o) : 0.0f;
                bx_in[hf][e] = (p.bn_x != nullptr && ok) ? __ldg(p.bn_x + o) : 0.0f;
                c_t[hf][e] = ok ? __ldg(p.c_save + o) : 0.0f;
                gts[hf][e] = ok ? __ldg(p.gates_save + o) : make_uint2(0u, 0u);
                const size_t op = (static_cast<size_t>(has_prev ? tprev : tt) * N + (ok ? gn : 0)) * H2 +
                                  static_cast<size_t>(dir) * H + unit;
                c_p[hf][e] = (ok && has_prev) ? __ldg(p.c_save + op) : 0.0f;
            }
        // partial dh[128 units, NB] = W_a^T dG_a + W_b^T dG_b, 2 * kblocks K blocks round-robin over four issuing warps
        if (warp < 4) {
            if (t == 0) mbar_wait(w_full, 0);
            if (t > 0) {
                mbar_wait(&b_full[t & 1], ((t - 1) >> 1) & 1);
                if (lane == 0 && warp == 0) mbar_expect_tx(&b_full[t & 1], 2 * img_bytes);
            }
            tc_fence_after();
            const uint32_t a0 = smem_u32(sW2);
            const uint32_t dacc = tmem_base + warp * NB;
            const bool leader = elect_one();
#pragma unroll 1
            for (int it = warp; it < 2 * kblocks; it += 4) {
                const int g = it >= kblocks ? 1 : 0, kb = it - g * kblocks;
                const uint64_t bd = umma_desc_sw64(smem_u32(sB) + (g * 2 + (t & 1)) * img_bytes + kb * (NB * 128));
                const uint32_t first = it == warp ? 0u : 1u;
                if (g == 0 || kb < KB_TMEM_B) {
                    const uint32_t ta = tmem_base + (g == 0 ? col_a : col_b) + kb * 32;
                    if (leader) {
                        umma_bf16_ts(dacc, ta, bd, idesc, first);
                        umma_bf16_ts(dacc, ta + 8, bd + 2, idesc, 1u);
                        umma_bf16_ts(dacc, ta + 16, bd + (NB * 64 / 16), idesc, 1u);
                        umma_bf16_ts(dacc, ta + 24, bd + (NB * 64 / 16) + 2, idesc, 1u);
                    }
                } else {
                    const uint64_t ad = umma_desc_sw128(a0 + (kb - KB_TMEM_B) * 16384);
                    if (leader) {
                        umma_bf16(dacc, ad, bd, idesc, first);
                        umma_bf16(dacc, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(dacc, ad + 4, bd + (NB * 64 / 16), idesc, 1u);
                        umma_bf16(dacc, ad + 6, bd + (NB * 64 / 16) + 2, idesc, 1u);
                    }
                }
            }
            if (leader) umma_commit(acc_full);
        }
        __syncwarp();
        mbar_wait(acc_full, t & 1);
        tc_fence_after();
        uint32_t acc[CPT];
        load_partial_sums<CPT>(tmem_base + (static_cast<uint32_t>(lq * 32) << 16) + ch * CPT, NB, 4, acc);
        tc_fence_before();
        // rows 32 lq.. of the unit block belong to CTA (lq >> 1, mb), half lq & 1: one bulk copy per warp
        if (warp_leader) bulk_wait_read_all();
        __syncthreads();
        {
            float* stage = sP + (lq * NB + ch * CPT) * 32 + lane;
#pragma unroll
            for (int c = 0; c < CPT; ++c) stage[c * 32] = __uint_as_float(acc[c]);
            fence_proxy_async_smem();
            __syncwarp();
            if (warp_leader) {
                const uint32_t peer = rank_of(lq >> 1, mb);
                bulk_copy_to_peer(mapa_shared(smem_u32(sR + ((qp * 2 + (lq & 1)) * NB + ch * CPT) * 32), peer),
                                  smem_u32(sP + (lq * NB + ch * CPT) * 32), CPT * 32 * 4, mapa_shared(smem_u32(r_full), peer));
                bulk_commit();
            }
            mbar_wait(r_full, t & 1);
            if (tid == 0) mbar_expect_tx(r_full, 4 * NB * 32 * 4);
        }
        uint2 dgp[2][EPT];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf)   // keep all arithmetic on the prefetched values below the waits (see pin_reg)
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                pin_reg(dh_in[hf][e]); pin_reg(bx_in[hf][e]); pin_reg(c_t[hf][e]); pin_reg(c_p[hf][e]);
                pin_reg(gts[hf][e].x); pin_reg(gts[hf][e].y);
            }
#pragma unroll
        for (int hf = 0; hf < 2; ++hf)
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int n = warp + 8 * e;
                float dh = bnk2[hf].a * dh_in[hf][e] + bnk2[hf].b * bx_in[hf][e] + ((p.n0 + grp * NB + n < N) ? bnk2[hf].d : 0.0f) +
                           sR[((0 * 2 + hf) * NB + n) * 32 + lane] + sR[((1 * 2 + hf) * NB + n) * 32 + lane];
                const __half2 lo = *reinterpret_cast<const __half2*>(&gts[hf][e].x);
                const __half2 hi = *reinterpret_cast<const __half2*>(&gts[hf][e].y);
                const float gi = __low2float(lo), gf = __high2float(lo), gg = __low2float(hi), go = __high2float(hi);
                const float tc = fast_tanh(c_t[hf][e]);
                const float d_o = dh * tc * go * (1.0f - go);
                const float dc = dc_carry[hf][e] + dh * go * (1.0f - tc * tc);
                const float d_i = dc * gg * gi * (1.0f - gi);
                const float d_f = dc * c_p[hf][e] * gf * (1.0f - gf);
                const float d_g = dc * gi * (1.0f - gg * gg);
                dc_carry[hf][e] = dc * gf;
                __nv_bfloat16* so = reinterpret_cast<__nv_bfloat16*>(sOut) + hf * OUT_CHUNKS * 8 + n * 32 +
                                    (((lane >> 3) ^ ((n >> 1) & 3)) << 3) + (lane & 7);
                so[0 * 2 * OUT_CHUNKS * 8] = __float2bfloat16(d_i);
                so[1 * 2 * OUT_CHUNKS * 8] = __float2bfloat16(d_f);
                so[2 * 2 * OUT_CHUNKS * 8] = __float2bfloat16(d_g);
                so[3 * 2 * OUT_CHUNKS * 8] = __float2bfloat16(d_o);
                __nv_bfloat162 b01 = __floats2bfloat162_rn(d_i, d_f), b23 = __floats2bfloat162_rn(d_g, d_o);
                dgp[hf][e] = make_uint2(*reinterpret_cast<uint32_t*>(&b01), *reinterpret_cast<uint32_t*>(&b23));
            }
        fence_proxy_async_smem();
        __syncthreads();
        if (t + 1 < T) {
            // gate g's two adjacent 32-unit blocks -> K blocks (4 mb + 2 qp, +1) of local gate (g & 1) in CTA (g >> 1, mb')
            const uint32_t koff = (4 * mb + 2 * qp) * BLK_BYTES;
            for (int i = warp; i < 4 * MB; i += 8) {
                const int g = i / MB, mdst = i - g * MB;
                const uint32_t peer = rank_of(g >> 1, mdst);
                const uint32_t dst = smem_u32(sB) + ((g & 1) * 2 + ((t + 1) & 1)) * img_bytes + koff;
                if (warp_leader)
                    bulk_copy_to_peer(mapa_shared(dst, peer), smem_u32(sOut + g * 2 * OUT_CHUNKS), 2 * BLK_BYTES,
                                      mapa_shared(smem_u32(&b_full[(t + 1) & 1]), peer));
            }
            if (warp_leader) bulk_commit();
        }
#pragma unroll
        for (int hf = 0; hf < 2; ++hf)
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int gn = p.n0 + grp * NB + warp + 8 * e;
                const int unit = unit0 + 32 * hf;
                if (gn < N)
                    *reinterpret_cast<uint2*>(p.dg + (static_cast<size_t>(tt) * N + gn) * G8 + static_cast<size_t>(dir) * 4 * H +
                                              static_cast<size_t>(unit >> 5) * 128 + (unit & 31) * 4) = dgp[hf][e];
            }
        publish_dg_chunk(p, t, T, next_pub);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// H in (512, 640]: the two-tile cluster kernels (64 units per CTA); CTCB200_LSTM_EXCHANGE=global keeps the global-exchange path
bool two_tile_path(int H) {
    const char* e = getenv("CTCB200_LSTM_EXCHANGE");
    if (e && e[0] == 'g') return false;
    return H > 512 && H <= 640 && H % 128 == 0;
}

// CTCB200_LSTM_PIPE=0 selects the un-pipelined forward kernel (one element phase per step over all 16 columns)
bool pipelined_fwd() {
    const char* e = getenv("CTCB200_LSTM_PIPE");
    return e == nullptr || e[0] != '0';
}

// warps that issue slices of the per-step MMA chain (each into its own TMEM accumulator, 64 columns in total)
int mma_issuers(int NB, int H) {
    int n = 64 / NB;  // accumulators that fit in front of the weight columns
    const char* e = getenv("CTCB200_LSTM_MMA_ISSUERS");
    if (e) n = atoi(e);
    if (n > 4) n = 4;
    while (n > 1 && (n > H / 64 || n * NB > 64)) n >>= 1;
    return n < 1 ? 1 : n;
}

// A recurrent CTA owns its SM: it holds (nearly) all 512 TMEM columns for the whole launch, so a tensor-core CTA of ANOTHER kernel
// (the GEMMs the host runs beside the recurrence on the idle SMs: weight gradients under BPTT, later chunks of a streamed
// input projection under the forward pass) must never become co-resident with it — its tcgen05.alloc would block until the
// recurrent kernel ends, and a forward kernel that is itself waiting for that GEMM's output would never end (observed: the
// bf16 kernels keep their weights in TMEM and need only ~50 KB of shared memory, which leaves room for a second CTA). Asking
// for at least 200 KB of dynamic shared memory makes the SM exclusive for every kernel that uses more than 27 KB.
constexpr size_t EXCLUSIVE_SMEM = 200 * 1024;
size_t exclusive_smem(size_t b) { return b < EXCLUSIVE_SMEM ? EXCLUSIVE_SMEM : b; }

size_t lstm_smem_bytes(int NB, int H, bool bwd, int ex, bool x3) {
    const bool bulk = ex == 3;
    const size_t parts = x3 ? 2 : 1;
    size_t b = (x3 ? static_cast<size_t>(128) * H * 2 : 0) + static_cast<size_t>(bulk ? 2 : 1) * H * NB * 2 * parts;
    if (!x3 && ex == 0 && H > TMEM_K_MAX) b += static_cast<size_t>(128) * (H - TMEM_K_MAX) * 2;   // W K blocks past TMEM
    if (bwd) b += static_cast<size_t>(4) * NB * 32 * 4 + (bulk ? static_cast<size_t>(4) * parts * NB * 4 * 16 + static_cast<size_t>(4) * NB * 32 * 4 : 0);
    else b += static_cast<size_t>(32) * (NB * 4 + 4) * 4 + (bulk ? parts * NB * 4 * 16 : 0);
    return exclusive_smem(b + 256 + 1024);
}

// How the CTAs of one (direction, batch group) hand h_t / dG_t to each other every step:
//   3 (default for H <= 512)  one cluster; one bulk (TMA-engine) DSMEM copy per peer, complete_tx on the peer's mbarrier
//   0 (H > 512, or no cluster of the needed size can be scheduled)  global image + global release/acquire counter,
//                             cooperative launch
// CTCB200_LSTM_EXCHANGE=global forces 0 (A/B measurements). Measured on B200 (cfg2, NB=16, cycles/step): bulk 3.2k
// (2.5k pipelined), global 9.3k; the DSMEM-store and L2+mbarrier variants of round 1 (6.6k / 6.8k) were removed.
int exchange_mode(int H) {
    const char* e = getenv("CTCB200_LSTM_EXCHANGE");
    if (e && e[0] == 'g') return 0;
    return H <= 512 ? 3 : 0;  // H/32 CTAs (forward) and 4*H/128 CTAs (backward) fit one cluster of <= 16
}

int pick_nb(int N, int H, int force_nb, bool bwd, bool cl) {
    if (force_nb == 16 || force_nb == 32) return force_nb;
    if (cl) return N <= 16 ? 16 : (((N + 15) / 16) * (bwd ? 4 * (H / 128) : H / 32) * 2 <= 128 ? 16 : 32);
    const int sms = device_sm_count();
    const int per_group = bwd ? 2 * 4 * (H / 128) : 2 * (H / 32);
    // prefer the narrow batch tile (shorter per-step chain) when every group fits at once
    const int g16 = (N + 15) / 16;
    const int budget = bwd ? (sms / 4) * 4 - 16 : sms;  // clusters of 4 cannot use every SM
    if (g16 * per_group <= budget) return 16;
    return 32;
}

// Can at least one cluster of this shape be resident? (fails on parts / partitions whose GPCs are too small)
template <typename Kern>
int cluster_probe(Kern kern, dim3 grid, dim3 cluster, size_t smem, int threads) {   // co-resident clusters (0: none)
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    if (cluster.x * cluster.y * cluster.z > 8 &&
        cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = cluster.x; attr.val.clusterDim.y = cluster.y; attr.val.clusterDim.z = cluster.z;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

template <typename Kern>
int cluster_capacity(Kern kern, dim3 grid, dim3 cluster, size_t smem, int threads = LSTM_THREADS) {
    // the answer depends only on (device, kernel, cluster shape, shared memory): remember the last few probes
    struct Entry { int dev; const void* k; unsigned cx, cy; size_t smem; int n; };
    static Entry cache[32];
    static int n_cache = 0;
    const int dev = current_device();
    for (int i = 0; i < n_cache; ++i)
        if (cache[i].dev == dev && cache[i].k == reinterpret_cast<const void*>(kern) && cache[i].cx == cluster.x &&
            cache[i].cy == cluster.y && cache[i].smem == smem)
            return cache[i].n;
    const int n = cluster_probe(kern, grid, cluster, smem, threads);
    if (n_cache < 32) cache[n_cache++] = Entry{dev, reinterpret_cast<const void*>(kern), cluster.x, cluster.y, smem, n};
    return n;
}
template <typename Kern>
bool cluster_ok(Kern kern, dim3 grid, dim3 cluster, size_t smem, int threads = LSTM_THREADS) {
    return cluster_capacity(kern, grid, cluster, smem, threads) >= 1;
}

using FwdKern = void (*)(CUtensorMap, FwdParams);
using BwdKern = void (*)(CUtensorMap, BwdParams);
FwdKern fwd_kernel(int NB, int ex, bool x3, int cell = CELL_LSTM) {
    if (cell == CELL_GRU) {
        if (x3) return ex == 3 ? lstm_fwd_kernel<16, 3, true, CELL_GRU> : lstm_fwd_kernel<16, 0, true, CELL_GRU>;
        return ex == 3 ? lstm_fwd_kernel<16, 3, false, CELL_GRU> : lstm_fwd_kernel<16, 0, false, CELL_GRU>;
    }
    if (cell == CELL_RNN) {
        if (x3) return ex == 3 ? lstm_fwd_kernel<16, 3, true, CELL_RNN> : lstm_fwd_kernel<16, 0, true, CELL_RNN>;
        return ex == 3 ? lstm_fwd_kernel<16, 3, false, CELL_RNN> : lstm_fwd_kernel<16, 0, false, CELL_RNN>;
    }
    if (x3) return ex == 3 ? lstm_fwd_kernel<16, 3, true> : lstm_fwd_kernel<16, 0, true>;
    if (NB == 16) return ex == 3 ? lstm_fwd_kernel<16, 3, false> : lstm_fwd_kernel<16, 0, false>;
    return ex == 3 ? lstm_fwd_kernel<32, 3, false> : lstm_fwd_kernel<32, 0, false>;
}
BwdKern bwd_kernel(int NB, int ex, bool x3, int cell = CELL_LSTM) {
    if (cell == CELL_GRU) {
        if (x3) return ex == 3 ? lstm_bwd_kernel<16, 3, true, CELL_GRU> : lstm_bwd_kernel<16, 0, true, CELL_GRU>;
        return ex == 3 ? lstm_bwd_kernel<16, 3, false, CELL_GRU> : lstm_bwd_kernel<16, 0, false, CELL_GRU>;
    }
    if (cell == CELL_RNN) {
        if (x3) return ex == 3 ? lstm_bwd_kernel<16, 3, true, CELL_RNN> : lstm_bwd_kernel<16, 0, true, CELL_RNN>;
        return ex == 3 ? lstm_bwd_kernel<16, 3, false, CELL_RNN> : lstm_bwd_kernel<16, 0, false, CELL_RNN>;
    }
    if (x3) return ex == 3 ? lstm_bwd_kernel<16, 3, true> : lstm_bwd_kernel<16, 0, true>;
    if (NB == 16) return ex == 3 ? lstm_bwd_kernel<16, 3, false> : lstm_bwd_kernel<16, 0, false>;
    return ex == 3 ? lstm_bwd_kernel<32, 3, false> : lstm_bwd_kernel<32, 0, false>;
}

template <typename Kern, typename Params>
int launch_clustered(Kern kern, dim3 grid, dim3 cluster, size_t smem, bool cooperative, const CUtensorMap& tm,
                     const Params& p, cudaStream_t stream, int threads = LSTM_THREADS, cudaEvent_t start_event = nullptr) {
    CTCB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    if (cluster.x * cluster.y * cluster.z > 8)
        CTCB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attrs[3];
    int n_attrs = 0;
    if (cluster.x * cluster.y * cluster.z > 1) {
        attrs[n_attrs].id = cudaLaunchAttributeClusterDimension;
        attrs[n_attrs].val.clusterDim.x = cluster.x; attrs[n_attrs].val.clusterDim.y = cluster.y; attrs[n_attrs].val.clusterDim.z = cluster.z;
        ++n_attrs;
    }
    if (start_event != nullptr) {
        // programmatic event: fires once every block of this grid has started, i.e. the grid is resident — other streams can
        // cudaStreamWaitEvent on it to hand the remaining SMs to independent work (a dependency the CUDA scheduler sees)
        attrs[n_attrs].id = cudaLaunchAttributeProgrammaticEvent;
        attrs[n_attrs].val.programmaticEvent.event = start_event;
        attrs[n_attrs].val.programmaticEvent.flags = 0;
        attrs[n_attrs].val.programmaticEvent.triggerAtBlockStart = 1;
        ++n_attrs;
    }
    if (cooperative) {
        attrs[n_attrs].id = cudaLaunchAttributeCooperative;
        attrs[n_attrs].val.cooperative = 1;
        ++n_attrs;
    }
    cfg.attrs = attrs;
    cfg.numAttrs = n_attrs;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tm, p);
    if (e != cudaSuccess && cooperative) {
        // some driver / tool combinations refuse cooperative + cluster together; co-residency is then guaranteed
        // by the caller's CTA budget (one CTA per SM, grid <= schedulable clusters) on an otherwise idle device
        (void)cudaGetLastError();
        cfg.numAttrs = n_attrs - 1;
        e = cudaLaunchKernelEx(&cfg, kern, tm, p);
    }
    CTCB_CUDA(e);
    return OK;
}

// CTCB200_LSTM_TRACE=1 asks for the per-phase cycle breakdown. In the pipelined forward kernel the clock stamps cost ~14 % of its
// run time even when switched off at run time (every warp role tests the pointer at several points of every half-step:
// 1.16 -> 1.00 ms per cfg2 layer without them, tools/rec_ab_head.py), so that kernel carries them only with -DCTCB200_TRACE
// (python -m ctc_pytorch_b200._build --trace). The BPTT kernel keeps its run-time switch: compiled without the stamps it came
// out 3 % SLOWER (1.494 -> 1.535 ms; the stamps happen to keep ptxas from a worse schedule), measured in the same run.
static bool trace_requested() { return getenv("CTCB200_LSTM_TRACE") != nullptr; }
static void pipe_trace_needs_build(FwdParams& p) {
#ifndef CTCB200_TRACE
    if (p.trace) {
        static bool told = false;
        if (!told) fprintf(stderr, "ctcb200: tracing the pipelined forward kernel needs the trace build: python -m ctc_pytorch_b200._build --trace\n");
        told = true;
        p.trace = nullptr;
    }
#else
    (void)p;
#endif
}

// development aid (CTCB200_LSTM_TRACE=1): per-phase cycle breakdown of the forward recurrence on stderr
struct FwdTraceDump {
    const FwdParams& p; cudaStream_t s; bool pipe;
    ~FwdTraceDump() {
        if (!p.trace) return;
        cudaStreamSynchronize(s);
        const int T = p.T;
        long long* h = static_cast<long long*>(malloc(sizeof(long long) * 16 * T));
        cudaMemcpy(h, p.trace, sizeof(long long) * 16 * T, cudaMemcpyDeviceToHost);
        if (pipe) {
            // stamps relative to the start of half A's element phase: A0..A5 = start, acc ready, loaded, gates regrouped,
            // h staged + arrive, stores issued; B0..B4 likewise; [11] = copy warp issued half A; M: hA landed, A issued,
            // hB landed, B issued
            double rel[16] = {0}, tot = 0;
            int cnt = 0;
            for (int t = 8; t + 1 < T; ++t, ++cnt) {
                for (int k = 0; k < 16; ++k) rel[k] += double(h[t * 16 + k] - h[t * 16]);
                tot += double(h[(t + 1) * 16] - h[t * 16]);
            }
            fprintf(stderr, "lstm_fwd_pipe trace (cycles, avg over %d steps): step %.0f | A:", cnt, tot / cnt);
            for (int k = 0; k < 6; ++k) fprintf(stderr, " %.0f", rel[k] / cnt);
            fprintf(stderr, " | B:");
            for (int k = 6; k < 12; ++k) fprintf(stderr, " %.0f", rel[k] / cnt);
            fprintf(stderr, " | M(hA landed, A issued, hB landed, B issued):");
            for (int k = 12; k < 16; ++k) fprintf(stderr, " %.0f", rel[k] / cnt);
            fprintf(stderr, "\n");
            free(h);
            return;
        }
        double acc[16] = {0};
        int cnt = 0;
        for (int t = 8; t + 1 < T; ++t, ++cnt) {
            for (int k = 1; k < 8; ++k) acc[k] += double(h[t * 16 + k] - h[t * 16 + k - 1]);
            acc[0] += double(h[(t + 1) * 16] - h[t * 16]);
            for (int k = 9; k < 14; ++k) acc[k] += double(h[t * 16 + k] - h[t * 16 + k - 1]);
        }
        fprintf(stderr, "lstm_fwd trace (cycles/step avg over %d steps): total %.0f | t0: start->hfull %.0f, mma issue %.0f, "
                "commit->acc %.0f, tmem ld %.0f, act+sync %.0f, cell+sync %.0f, push+sync+arrive %.0f | t255: ld %.0f act %.0f "
                "sync %.0f cell %.0f push %.0f\n", cnt, acc[0] / cnt, acc[1] / cnt, acc[2] / cnt, acc[3] / cnt, acc[4] / cnt,
                acc[5] / cnt, acc[6] / cnt, acc[7] / cnt, acc[9] / cnt, acc[10] / cnt, acc[11] / cnt, acc[12] / cnt, acc[13] / cnt);
        free(h);
    }
};

struct BwdTraceDump {
    const BwdParams& p; cudaStream_t s;
    ~BwdTraceDump() {
        if (!p.trace) return;
        cudaStreamSynchronize(s);
        const int T = p.T;
        long long* h = static_cast<long long*>(malloc(sizeof(long long) * 16 * T));
        cudaMemcpy(h, p.trace, sizeof(long long) * 16 * T, cudaMemcpyDeviceToHost);
        double rel[10] = {0}, tot = 0;
        int cnt = 0;
        for (int t = 8; t + 1 < T; ++t, ++cnt) {
            for (int k = 0; k < 10; ++k) rel[k] += double(h[t * 16 + k] - h[t * 16]);
            tot += double(h[(t + 1) * 16] - h[t * 16]);
        }
        fprintf(stderr, "lstm_bwd trace (CTA 0 thread 0, cycles after the step start, avg over %d steps): step %.0f | first K block landed "
                "%.0f, MMAs issued %.0f, acc ready %.0f, tcgen05.ld done %.0f, partials staged + reduce-scatter issued %.0f, partials "
                "landed %.0f, element phase done %.0f, CTA barrier %.0f, all-gather issued %.0f\n", cnt, tot / cnt, rel[1] / cnt,
                rel[2] / cnt, rel[3] / cnt, rel[4] / cnt, rel[5] / cnt, rel[6] / cnt, rel[7] / cnt, rel[8] / cnt, rel[9] / cnt);
        free(h);
    }
};

}  // namespace
}  // namespace ctcb200

using namespace ctcb200;

extern "C" CTCB200_API int64_t ctcb200_lstm_scratch_bytes(int N, int H) {
    // two directions x groups(16-wide worst case) x (4 gates x 2 parities) images (32-wide, or 16-wide hi+lo) + flags
    const int64_t groups = (N + 15) / 16;
    return 2 * groups * 8 * static_cast<int64_t>(H) * 32 * 2 + 2 * groups * 32 * 4 + 1024;
}

extern "C" CTCB200_API int ctcb200_lstm_bwd_ctas(int N, int H, int batch_tile) {
    // SMs the (first) BPTT launch occupies: one CTA per SM, 4 gates x H/128 unit blocks x 2 directions x batch groups
    if (H % 128 != 0 || H < 128 || H > MAX_HIDDEN || N <= 0) return 0;
    const int nb = two_tile_path(H) ? 16 : pick_nb(N, H, batch_tile, true, exchange_mode(H) != 0);
    const int groups = (N + nb - 1) / nb;
    const int per_group = two_tile_path(H) ? 2 * 2 * (H / 128) : 2 * 4 * (H / 128);
    const int sms = device_sm_count();
    const int total = per_group * groups;
    return total < sms ? total : sms;
}

namespace ctcb200 {
namespace {
// One body for ctcb200_lstm_fwd / ctcb200_lstm_fwd_streamed / ctcb200_lstm_fwd_ctas. plan_only: nothing is launched; *plan_ctas
// receives the number of CTAs (= SMs) the launch would occupy when it is ONE clustered launch (the only form a streamed input
// projection can run under: every batch group resident at once, nothing cooperative), else 0.
int lstm_fwd_impl(const float* gx, const void* whh_packed, const void* whh_lo_packed, float* hout, float* c_save,
                  void* gates_save, void* scratch, int T, int N, int H, int batch_tile, int cell, void* resident_counter,
                  const void* gx_ready, uint32_t gx_base, int chunk_T, bool x3_plan, bool plan_only, int* plan_ctas,
                  ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const bool x3 = plan_only ? x3_plan : whh_lo_packed != nullptr;
    if (plan_ctas) *plan_ctas = 0;
    CTCB_REQUIRE(cell >= 0 && cell <= 3, "lstm_fwd: cell %d not in {0 LSTM, 1 GRU, 2 RNN tanh, 3 RNN relu}", cell);
    const int cell_k = cell == 0 ? CELL_LSTM : (cell == 1 ? CELL_GRU : CELL_RNN);
    const bool plain = cell_k == CELL_LSTM;   // the pipelined / two-tile fast paths exist for the LSTM cell only
    CTCB_REQUIRE(T > 0 && N > 0, "lstm_fwd: empty T=%d N=%d", T, N);
    CTCB_REQUIRE(H % 128 == 0 && H >= 128 && H <= (x3 ? MAX_HIDDEN_X3 : MAX_HIDDEN),
                 "lstm_fwd: hidden size %d must be a multiple of 128 in [128,%d]", H, x3 ? MAX_HIDDEN_X3 : MAX_HIDDEN);
    FwdParams p;
    p.gx = gx; p.hout = hout; p.c_save = c_save;
    p.gates_save = x3 ? nullptr : static_cast<uint2*>(gates_save);
    p.gates_save32 = x3 ? static_cast<float4*>(gates_save) : nullptr;
    p.himg = nullptr; p.flags = nullptr; p.trace = nullptr; p.act_approx = 0; p.rnn_relu = cell == 3 ? 1 : 0;
    p.w = static_cast<const __nv_bfloat16*>(whh_packed);
    p.T = T; p.N = N; p.H = H; p.n0 = 0;
    CTCB_REQUIRE((reinterpret_cast<uintptr_t>(resident_counter) & 3) == 0 && (reinterpret_cast<uintptr_t>(gx_ready) & 3) == 0,
                 "lstm_fwd: resident_counter / gx_ready must be 4-byte aligned");
    CTCB_REQUIRE(gx_ready == nullptr || chunk_T >= 2, "lstm_fwd: a streamed input projection needs chunk_T >= 2 (got %d)", chunk_T);
    p.resident = static_cast<unsigned int*>(resident_counter);
    p.gx_ready = static_cast<const unsigned int*>(gx_ready);
    p.gx_base = gx_base;
    p.chunk_T = (gx_ready != nullptr) ? chunk_T : 0x3fffffff;
    if (!x3 && plain && two_tile_path(H)) {
        // H > 512: 64 units per CTA (tile 0 in TMEM, tile 1 in shared memory), H/64 CTAs per cluster, NB = 16
        constexpr int NB2 = 16;
        const int groups2 = (N + NB2 - 1) / NB2;
        CUtensorMap tmW2;
        int rc2 = plan_only ? OK : make_tmap_bf16_2d(&tmW2, whh_packed, static_cast<uint64_t>(8) * H, H, H, 128, 64);
        if (rc2 != OK) return rc2;
        const size_t smem2 = exclusive_smem(static_cast<size_t>(128) * H * 2 + static_cast<size_t>(2) * H * NB2 * 2 +
                                            static_cast<size_t>(2) * 32 * (NB2 * 4 + 4) * 4 + static_cast<size_t>(2) * NB2 * 4 * 16 + 64 + 1024);
        CTCB_REQUIRE(smem2 <= 227 * 1024, "lstm_fwd: shared memory %zu exceeds 227 KB (H=%d)", smem2, H);
        p.mma_split = 4; p.groups = groups2;
        if (cluster_ok(lstm_fwd2_kernel<NB2>, dim3(H / 64, 2, groups2), dim3(H / 64, 1, 1), smem2)) {
            if (plan_only) {   // streaming needs every cluster of the launch resident at once
                if (2 * groups2 <= cluster_capacity(lstm_fwd2_kernel<NB2>, dim3(H / 64, 2, groups2), dim3(H / 64, 1, 1), smem2))
                    *plan_ctas = (H / 64) * 2 * groups2;
                return OK;
            }
            return launch_clustered(lstm_fwd2_kernel<NB2>, dim3(H / 64, 2, groups2), dim3(H / 64, 1, 1), smem2, false, tmW2, p,
                                    stream);
        }
    }
    int ex = exchange_mode(H);
    {   // fall back to the global-memory exchange when a cluster of this size cannot be scheduled on this device
        const int nb_try = (x3 || !plain) ? 16 : pick_nb(N, H, batch_tile, false, ex != 0);
        if (ex != 0 && !cluster_ok(fwd_kernel(nb_try, ex, x3, cell_k), dim3(H / 32, 2, (N + nb_try - 1) / nb_try), dim3(H / 32, 1, 1),
                                   lstm_smem_bytes(nb_try, H, false, ex, x3)))
            ex = 0;
    }
    const bool cl = ex != 0;
    const int NB = (x3 || !plain) ? 16 : pick_nb(N, H, batch_tile, false, cl);
    const int groups_total = (N + NB - 1) / NB;
    CUtensorMap tmW;   // only read by the split-operand kernels (W_lo slice -> shared memory)
    int rc = plan_only ? OK : make_tmap_bf16_2d(&tmW, x3 ? whh_lo_packed : whh_packed, static_cast<uint64_t>(8) * H, H, H, 128, 64);
    if (rc != OK) return rc;
    const size_t smem = lstm_smem_bytes(NB, H, false, ex, x3);
    CTCB_REQUIRE(smem <= 227 * 1024, "lstm_fwd: shared memory %zu exceeds 227 KB (H=%d)", smem, H);
    {
        const char* act = getenv("CTCB200_LSTM_ACT");
        p.act_approx = (!x3 && plain && act != nullptr && act[0] == 'a') ? 1 : 0;
    }
    p.mma_split = mma_issuers(NB, H);
    p.groups = groups_total;
    if (!plan_only && trace_requested()) {
        static long long* dbuf = nullptr;
        if (!dbuf) CTCB_CUDA(cudaMalloc(&dbuf, sizeof(long long) * 16 * 4096));
        if (T <= 4096) {
            CTCB_CUDA(cudaMemsetAsync(dbuf, 0, sizeof(long long) * 16 * T, stream));
            p.trace = dbuf;
        }
    }
    FwdTraceDump trace_dump{p, stream, false};
    if (cl && !x3 && plain && NB == 16 && pipelined_fwd()) {
        pipe_trace_needs_build(p);
        trace_dump.pipe = true;
        // software-pipelined kernel: two 8-column halves per group, dedicated tensor-core warps
        dim3 grid(H / 32, 2, groups_total), cluster(H / 32, 1, 1);
        const size_t smem_p = exclusive_smem(static_cast<size_t>(2) * H * 16 * 2 + 4 * 512 + 4 * 8 * 128 * 4 + 128 + 1024);
        CUtensorMap tmGx;   // gate pre-activations as a 2-D f32 tensor [T*N rows, 8H columns], boxes of 8 rows x 128 columns
        rc = plan_only ? OK : make_tmap_f32_2d(&tmGx, gx, static_cast<uint64_t>(T) * N, static_cast<uint64_t>(8) * H, static_cast<uint64_t>(8) * H, 8, 128);
        if (rc == OK && cluster_ok(lstm_fwd_pipe_kernel, grid, cluster, smem_p, PIPE_THREADS)) {
            if (plan_only) {
                if (2 * groups_total <= cluster_capacity(lstm_fwd_pipe_kernel, grid, cluster, smem_p, PIPE_THREADS))
                    *plan_ctas = (H / 32) * 2 * groups_total;
                return OK;
            }
            return launch_clustered(lstm_fwd_pipe_kernel, grid, cluster, smem_p, false, tmGx, p, stream, PIPE_THREADS);
        }
    }
    if (cl) {
        // independent clusters: no co-residency requirement between them, one launch covers every batch group
        dim3 grid(H / 32, 2, groups_total), cluster(H / 32, 1, 1);
        if (plan_only) {
            if (2 * groups_total <= cluster_capacity(fwd_kernel(NB, ex, x3, cell_k), grid, cluster, smem))
                *plan_ctas = (H / 32) * 2 * groups_total;
            return OK;
        }
        return launch_clustered(fwd_kernel(NB, ex, x3, cell_k), grid, cluster, smem, false, tmW, p, stream);
    }
    if (plan_only) return OK;   // global-memory exchange: several cooperative launches, no streaming
    CTCB_REQUIRE(gx_ready == nullptr && resident_counter == nullptr,
                 "lstm_fwd: a streamed input projection needs the clustered kernels (ask ctcb200_lstm_fwd_ctas first)");
    const int per_group = 2 * (H / 32);
    const int sms = device_sm_count();
    CTCB_REQUIRE(per_group <= sms, "lstm_fwd: one batch group needs %d CTAs but the device has %d SMs", per_group, sms);
    const int groups_per_launch = sms / per_group;
    const size_t parts = x3 ? 2 : 1;
    uint8_t* scr = static_cast<uint8_t*>(scratch);
    for (int g0 = 0; g0 < groups_total; g0 += groups_per_launch) {
        const int groups = (groups_total - g0 < groups_per_launch) ? groups_total - g0 : groups_per_launch;
        const size_t img_bytes = static_cast<size_t>(2) * groups * 2 * H * NB * 2 * parts;
        const size_t flag_bytes = static_cast<size_t>(2) * groups * 32 * 4;
        CTCB_CUDA(cudaMemsetAsync(scr, 0, img_bytes + flag_bytes, stream));
        p.himg = reinterpret_cast<__nv_bfloat16*>(scr);
        p.flags = reinterpret_cast<unsigned int*>(scr + img_bytes);
        p.groups = groups; p.n0 = g0 * NB;
        rc = launch_clustered(fwd_kernel(NB, 0, x3, cell_k), dim3(H / 32, 2, groups), dim3(1, 1, 1), smem, true, tmW, p, stream);
        if (rc != OK) return rc;
    }
    return OK;
}
}  // namespace
}  // namespace ctcb200

extern "C" CTCB200_API int ctcb200_lstm_fwd(const float* gx, const void* whh_packed, const void* whh_lo_packed, float* hout,
                                            float* c_save, void* gates_save, void* scratch, int T, int N, int H,
                                            int batch_tile, int cell, ctcb200_stream_t stream) {
    return lstm_fwd_impl(gx, whh_packed, whh_lo_packed, hout, c_save, gates_save, scratch, T, N, H, batch_tile, cell, nullptr,
                         nullptr, 0u, 0, false, false, nullptr, stream);
}

extern "C" CTCB200_API int ctcb200_lstm_fwd_streamed(const float* gx, const void* whh_packed, const void* whh_lo_packed,
                                                     float* hout, float* c_save, void* gates_save, void* scratch, int T, int N,
                                                     int H, int batch_tile, int cell, void* resident_counter,
                                                     const void* gx_ready, uint32_t gx_base, int chunk_T,
                                                     ctcb200_stream_t stream) {
    // the kernel launched here waits for GEMM chunks: none of them may be a kernel's first (lazily loading) launch
    if (gx_ready != nullptr) {
        const int rc = gemm_preload();
        if (rc != OK) return rc;
    }
    return lstm_fwd_impl(gx, whh_packed, whh_lo_packed, hout, c_save, gates_save, scratch, T, N, H, batch_tile, cell,
                         resident_counter, gx_ready, gx_base, chunk_T, false, false, nullptr, stream);
}

extern "C" CTCB200_API int ctcb200_lstm_fwd_ctas(int N, int H, int batch_tile, int x3, int cell) {
    int ctas = 0;
    if (lstm_fwd_impl(nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 1, N, H, batch_tile, cell, nullptr, nullptr,
                      0u, 0, x3 != 0, true, &ctas, nullptr) != OK)
        return 0;
    return ctas;
}

namespace ctcb200 {
namespace {
// One body for ctcb200_lstm_bwd / ctcb200_lstm_bwd_streamed / ctcb200_lstm_bwd_plan (plan_only: nothing is launched, *plan_ctas
// = CTAs of the launch when it is ONE clustered launch — the form whose per-chunk progress counts are simply CTAs x chunks —
// else 0).
int lstm_bwd_impl(const float* dhout, const void* whhT_packed, const void* whhT_lo_packed, const float* c_save,
                  const void* gates_save, void* dg, void* dg_lo, void* dg_rec, void* dg_rec_lo, void* scratch, int T, int N, int H,
                  int batch_tile, int cell, const float* bn_x, const float* bn_coef, void* resident_counter, void* resident_event,
                  void* progress_counter, int chunk_T, bool x3_plan, bool plan_only, int* plan_ctas, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaEvent_t start_ev = static_cast<cudaEvent_t>(resident_event);
    const bool x3 = plan_only ? x3_plan : whhT_lo_packed != nullptr;
    if (plan_ctas) *plan_ctas = 0;
    CTCB_REQUIRE(cell >= 0 && cell <= 3, "lstm_bwd: cell %d not in {0 LSTM, 1 GRU, 2 RNN tanh, 3 RNN relu}", cell);
    const int cell_k = cell == 0 ? CELL_LSTM : (cell == 1 ? CELL_GRU : CELL_RNN);
    const bool plain = cell_k == CELL_LSTM;
    CTCB_REQUIRE(plan_only || cell_k != CELL_GRU || (dg_rec != nullptr && (!x3 || dg_rec_lo != nullptr)),
                 "lstm_bwd: the GRU cell needs dg_rec (and dg_rec_lo in the split-operand mode)");
    CTCB_REQUIRE(T > 0 && N > 0, "lstm_bwd: empty T=%d N=%d", T, N);
    CTCB_REQUIRE((reinterpret_cast<uintptr_t>(resident_counter) & 3) == 0, "lstm_bwd: resident_counter must be 4-byte aligned");
    CTCB_REQUIRE((bn_x == nullptr) == (bn_coef == nullptr), "lstm_bwd: bn_x and bn_coef must be given together");
    CTCB_REQUIRE(H % 128 == 0 && H >= 128 && H <= (x3 ? MAX_HIDDEN_X3 : MAX_HIDDEN),
                 "lstm_bwd: hidden size %d must be a multiple of 128 in [128,%d]", H, x3 ? MAX_HIDDEN_X3 : MAX_HIDDEN);
    CTCB_REQUIRE(plan_only || !x3 || dg_lo != nullptr, "lstm_bwd: the split-operand mode needs dg_lo");
    CTCB_REQUIRE((reinterpret_cast<uintptr_t>(progress_counter) & 3) == 0, "lstm_bwd: progress_counter must be 4-byte aligned");
    CTCB_REQUIRE(progress_counter == nullptr || chunk_T >= 1, "lstm_bwd: streamed gate gradients need chunk_T >= 1 (got %d)", chunk_T);
    BwdParams p;
    p.dhout = dhout; p.c_save = c_save;
    p.gates_save = x3 ? nullptr : static_cast<const uint2*>(gates_save);
    p.gates_save32 = x3 ? static_cast<const float4*>(gates_save) : nullptr;
    p.dg = static_cast<__nv_bfloat16*>(dg); p.dg_lo = static_cast<__nv_bfloat16*>(dg_lo);
    p.dg_rec = static_cast<__nv_bfloat16*>(dg_rec); p.dg_rec_lo = static_cast<__nv_bfloat16*>(dg_rec_lo);
    p.rnn_relu = cell == 3 ? 1 : 0;
    p.dgimg = nullptr; p.flags = nullptr; p.trace = nullptr;
    p.resident = static_cast<unsigned int*>(resident_counter);
    p.bn_x = bn_x; p.bn_coef = bn_coef;
    p.progress = static_cast<unsigned int*>(progress_counter);
    p.chunk_T = progress_counter != nullptr ? chunk_T : 0x3fffffff;
    p.w = static_cast<const __nv_bfloat16*>(whhT_packed);
    p.T = T; p.N = N; p.H = H; p.n0 = 0;
    if (!x3 && plain && two_tile_path(H)) {
        constexpr int NB2 = 16;
        const int groups2 = (N + NB2 - 1) / NB2;
        CUtensorMap tmWT2;
        int rc2 = plan_only ? OK : make_tmap_bf16_2d(&tmWT2, whhT_packed, static_cast<uint64_t>(8) * H, H, H, 128, 64);
        if (rc2 != OK) return rc2;
        const size_t smem2 = exclusive_smem(static_cast<size_t>(128) * (H - 256) * 2 + static_cast<size_t>(4) * H * NB2 * 2 +
                                            static_cast<size_t>(4) * NB2 * 32 * 4 * 2 + static_cast<size_t>(8) * NB2 * 4 * 16 + 64 + 1024);
        CTCB_REQUIRE(smem2 <= 227 * 1024, "lstm_bwd: shared memory %zu exceeds 227 KB (H=%d)", smem2, H);
        p.mma_split = 4; p.groups = groups2;
        if (cluster_ok(lstm_bwd2_kernel<NB2>, dim3(2, H / 128, 2 * groups2), dim3(2, H / 128, 1), smem2)) {
            if (plan_only) { *plan_ctas = 2 * (H / 128) * 2 * groups2; return OK; }
            return launch_clustered(lstm_bwd2_kernel<NB2>, dim3(2, H / 128, 2 * groups2), dim3(2, H / 128, 1), smem2, false,
                                    tmWT2, p, stream, LSTM_THREADS, start_ev);
        }
    }
    int ex = exchange_mode(H);
    {
        const int nb_try = (x3 || !plain) ? 16 : pick_nb(N, H, batch_tile, true, ex != 0);
        if (ex != 0 && !cluster_ok(bwd_kernel(nb_try, ex, x3, cell_k), dim3(4, H / 128, 2 * ((N + nb_try - 1) / nb_try)),
                                   dim3(4, H / 128, 1), lstm_smem_bytes(nb_try, H, true, ex, x3)))
            ex = 0;
    }
    const bool cl = ex != 0;
    const int NB = (x3 || !plain) ? 16 : pick_nb(N, H, batch_tile, true, cl);
    const int groups_total = (N + NB - 1) / NB;
    const int MB = H / 128;
    CUtensorMap tmWT;   // only read by the split-operand kernels (W^T_lo slice -> shared memory)
    int rc = plan_only ? OK : make_tmap_bf16_2d(&tmWT, x3 ? whhT_lo_packed : whhT_packed, static_cast<uint64_t>(8) * H, H, H, 128, 64);
    if (rc != OK) return rc;
    const size_t smem = lstm_smem_bytes(NB, H, true, ex, x3);
    CTCB_REQUIRE(smem <= 227 * 1024, "lstm_bwd: shared memory %zu exceeds 227 KB (H=%d)", smem, H);
    p.mma_split = mma_issuers(NB, H);
    p.groups = groups_total;
    if (!plan_only && trace_requested()) {
        static long long* dbuf = nullptr;
        if (!dbuf) CTCB_CUDA(cudaMalloc(&dbuf, sizeof(long long) * 16 * 4096));
        if (T <= 4096) {
            CTCB_CUDA(cudaMemsetAsync(dbuf, 0, sizeof(long long) * 16 * T, stream));
            p.trace = dbuf;
        }
    }
    BwdTraceDump trace_dump{p, stream};
    if (plan_only) {
        if (cl) *plan_ctas = 4 * MB * 2 * groups_total;
        return OK;
    }
    CTCB_REQUIRE(cl || progress_counter == nullptr,
                 "lstm_bwd: streamed gate gradients need the clustered kernels (ask ctcb200_lstm_bwd_plan first)");
    if (cl) {
        dim3 grid(4, MB, 2 * groups_total), cluster(4, MB, 1);
        return launch_clustered(bwd_kernel(NB, ex, x3, cell_k), grid, cluster, smem, false, tmWT, p, stream, LSTM_THREADS, start_ev);
    }
    const int per_group = 2 * 4 * MB;
    const int sms = device_sm_count();
    const int budget = (sms / 4) * 4 - 16;  // clusters of 4 strand a few SMs
    CTCB_REQUIRE(per_group <= budget, "lstm_bwd: one batch group needs %d CTAs; device budget %d", per_group, budget);
    const int groups_per_launch = budget / per_group;
    const size_t parts = x3 ? 2 : 1;
    uint8_t* scr = static_cast<uint8_t*>(scratch);
    for (int g0 = 0; g0 < groups_total; g0 += groups_per_launch) {
        const int groups = (groups_total - g0 < groups_per_launch) ? groups_total - g0 : groups_per_launch;
        const size_t img_bytes = static_cast<size_t>(2) * groups * 4 * 2 * H * NB * 2 * parts;
        const size_t flag_bytes = static_cast<size_t>(2) * groups * 32 * 4;
        CTCB_CUDA(cudaMemsetAsync(scr, 0, img_bytes + flag_bytes, stream));
        p.dgimg = reinterpret_cast<__nv_bfloat16*>(scr);
        p.flags = reinterpret_cast<unsigned int*>(scr + img_bytes);
        p.groups = groups; p.n0 = g0 * NB;
        if (g0 > 0) p.resident = nullptr;
        dim3 grid(4, MB, 2 * groups), cluster(4, 1, 1);
        const bool coop = getenv("CTCB200_BWD_NO_COOP") == nullptr;  // profilers may reject cooperative + cluster
        rc = launch_clustered(bwd_kernel(NB, 0, x3, cell_k), grid, cluster, smem, coop, tmWT, p, stream, LSTM_THREADS, g0 == 0 ? start_ev : nullptr);
        if (rc != OK) return rc;
    }
    return OK;
}
}  // namespace
}  // namespace ctcb200

extern "C" CTCB200_API int ctcb200_lstm_bwd(const float* dhout, const void* whhT_packed, const void* whhT_lo_packed,
                                            const float* c_save, const void* gates_save, void* dg, void* dg_lo, void* dg_rec,
                                            void* dg_rec_lo, void* scratch, int T, int N, int H, int batch_tile, int cell,
                                            const float* bn_x, const float* bn_coef, void* resident_counter,
                                            void* resident_event, ctcb200_stream_t stream) {
    return lstm_bwd_impl(dhout, whhT_packed, whhT_lo_packed, c_save, gates_save, dg, dg_lo, dg_rec, dg_rec_lo, scratch, T, N, H,
                         batch_tile, cell, bn_x, bn_coef, resident_counter, resident_event, nullptr, 0, false, false, nullptr,
                         stream);
}

extern "C" CTCB200_API int ctcb200_lstm_bwd_streamed(const float* dhout, const void* whhT_packed, const void* whhT_lo_packed,
                                                     const float* c_save, const void* gates_save, void* dg, void* dg_lo,
                                                     void* dg_rec, void* dg_rec_lo, void* scratch, int T, int N, int H,
                                                     int batch_tile, int cell, const float* bn_x, const float* bn_coef,
                                                     void* resident_counter, void* progress_counter, int chunk_T,
                                                     ctcb200_stream_t stream) {
    return lstm_bwd_impl(dhout, whhT_packed, whhT_lo_packed, c_save, gates_save, dg, dg_lo, dg_rec, dg_rec_lo, scratch, T, N, H,
                         batch_tile, cell, bn_x, bn_coef, resident_counter, nullptr, progress_counter, chunk_T, false, false,
                         nullptr, stream);
}

extern "C" CTCB200_API int ctcb200_lstm_bwd_plan(int N, int H, int batch_tile, int x3, int cell) {
    int ctas = 0;
    if (lstm_bwd_impl(nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 1, N, H, batch_tile,
                      cell, nullptr, nullptr, nullptr, nullptr, nullptr, 0, x3 != 0, true, &ctas, nullptr) != OK)
        return 0;
    return ctas;
}
