// fm_kernel.cuh -- the fused persistent MoE-forward kernel for sm_100a.
//
// One launch = one MoE layer forward on this rank (reference: flashmoe::moe::forward, csrc/include/flashmoe/moe/moe.cuh:77-144):
//
//   prologue  mbarriers + TMEM allocation for the later phases (off the critical path)
//   phase G   router    x.Wg^T -> online softmax -> top-k -> capacity slots         (reference moe/gate.cuh:473-720)
//             grid barrier (the only one, like the reference's gate.cuh:761)
//   phase D   dispatch  token rows -> owner rank's receive buffer over NVLink (TMA bulk copies) + one flag per expert
//                                                                                    (reference os/packet.cuh:21-286)
//   phase F   expert FFN  persistent tcgen05 tile loop over CTA pairs: GEMM0(+bias+act) -> h, GEMM1(+bias) -> for k <= 2
//             scaled and ADDED straight into the token's output row on the source rank (REDG.BF16x8 over peer memory),
//             otherwise stored to the source rank's return buffer + per-row-block flag
//                                                                                    (reference os/processor/processor.cuh:340-468,
//                                                                                    685-750; the OS CTA of os/os.cuh, scheduler.cuh,
//                                                                                    subscriber.cuh is replaced by an atomic tile
//                                                                                    claim + flag waits in one warp per CTA pair)
//   phase C   completion: wait for the experts' done flags (fused path) or gather-combine the k returned rows per token
//                                                                                    (reference processor.cuh:27-205)
//
// CTA = 384 threads, one CTA per SM, all co-resident (74 clusters of 2; cooperative launch, and co-residency is checked on
// the host with cudaOccupancyMaxActiveClusters).  After the grid barrier the warps specialise: warp 0 = TMA producer,
// warp 1 = tcgen05.mma issuer (leader CTA of the pair), warp 3 = tile scheduler (leader CTA), warps 2 and 4-11 = dispatch,
// then warps 4-11 = epilogue (TMEM -> registers -> bias/activation/combine scaling -> bf16 -> swizzled smem transpose ->
// 16-byte global / peer stores or adds; two warps per TMEM lane quarter, each draining half of the tile's columns) and
// warp 2 = publisher (the release fence + counter / flag traffic of every finished tile, off the epilogue warps' critical
// path); warp 2 also owns the TMEM allocation.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/flashmoe_b200.h"
#include "fm_ptx.cuh"

namespace fm {

constexpr int BLOCK_M = 128;   // token rows per tile (= reference BLOCK_M)
constexpr int BLOCK_N = 256;   // output columns per tile (one tcgen05.mma N)
constexpr int BLOCK_K = 64;    // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int NSCHED = 4;
// the scheduler claims the next tile when this many k-blocks of the current one remain (config B on one B200:
// 8 -> 144.5 us per forward, 12 -> 142.3, 14 -> 140.6; 16 and larger alike)
constexpr int CLAIM_AHEAD_KB = 16;
constexpr int NUM_THREADS = 384;
constexpr int NUM_WARPS = NUM_THREADS / 32;
constexpr int EPI_WARP0 = 4;   // warps 4..11: warp % 4 selects the TMEM lane quarter, (warp - 4) / 4 the column half
constexpr int NUM_EPI_WARPS = 8;
constexpr int TMEM_COLS = 512; // two 128x256 fp32 accumulators per CTA (double-buffered against the epilogue)
constexpr int TRACE_SLOTS = 128; // per CTA: [0..6] phase stamps, [8..14] sub-phase stamps (13 = first tile of a remote packet
                                 // ready, 14 = all done flags seen); per tile i < 16 of this CTA (pair):
                                 // [16+i] dependencies resolved (scheduler), [32+i] first k-block landed, [48+i] last MMA
                                 // issued (MMA thread), [64+i] accumulator complete (epilogue sees tmem_full), [80+i]
                                 // epilogue stores issued, [96+i] published, [112+i] claimed (scheduler)

constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;                  // 16 KiB
constexpr int PIPE_BYTES = 196608;                                    // 4 x 48 KiB (solo) = 6 x 32 KiB (CTA pair)
constexpr int MAX_STAGES = 6;
constexpr int EPI_ROW_BYTES = 128;                                    // 64 bf16; 16-byte pieces XOR-swizzled by (row & 7)
constexpr int EPI_WARP_BYTES = 32 * EPI_ROW_BYTES;                    // 4 KiB per epilogue warp
constexpr int OFF_EPI = PIPE_BYTES;                                   // 196608
constexpr int OFF_BARS = OFF_EPI + NUM_EPI_WARPS * EPI_WARP_BYTES;    // 229376
// barriers: full[6] empty[6] tmem_full[2] tmem_empty[2] sched_full[4] sched_empty[4] prod_take[4] xrows disp_done
//           pub_full[2] pub_empty[2]
constexpr int BAR_FULL = 0, BAR_EMPTY = MAX_STAGES, BAR_TMEM_FULL = 2 * MAX_STAGES, BAR_TMEM_EMPTY = BAR_TMEM_FULL + 2;
constexpr int BAR_SCHED_FULL = BAR_TMEM_EMPTY + 2, BAR_SCHED_EMPTY = BAR_SCHED_FULL + NSCHED;
constexpr int BAR_PROD_TAKE = BAR_SCHED_EMPTY + NSCHED;
constexpr int BAR_XROWS = BAR_PROD_TAKE + NSCHED;                     // dispatch phase: bulk row load
constexpr int BAR_DISP_DONE = BAR_XROWS + 1;                          // this CTA's dispatch no longer uses the stage area
constexpr int BAR_PUB_FULL = BAR_DISP_DONE + 1;                       // epilogue warps -> publisher: tile's stores issued
constexpr int BAR_PUB_EMPTY = BAR_PUB_FULL + 2;                       // publisher -> epilogue warps: slot consumed
constexpr int BAR_WG = BAR_PUB_EMPTY + 2;                             // router: bulk-staged gate weights
constexpr int BAR_REMOTE = BAR_WG + 1;                                // dispatch, warp 2: staged rows for other ranks
constexpr int GATE_STAGES = 8;                                        // router GEMM on tensor cores: up to 8 smem stages
constexpr int BAR_GFULL = BAR_REMOTE + 1;                             // full / empty per stage, accumulator complete
constexpr int BAR_GEMPTY = BAR_GFULL + GATE_STAGES;
constexpr int BAR_GACC = BAR_GEMPTY + GATE_STAGES;
constexpr int NUM_BARS = BAR_GACC + 2;                                // 54 (one spare keeps the ring 16-byte aligned)
constexpr int OFF_RING = OFF_BARS + NUM_BARS * 8;                     // 16-byte aligned
constexpr int OFF_TMEM_PTR = OFF_RING + NSCHED * 64;
constexpr int OFF_MISC = OFF_TMEM_PTR + 16;
constexpr int SMEM_USED = OFF_MISC + 64;
constexpr int SMEM_BYTES = SMEM_USED + 1024;                          // + slack for manual 1 KiB alignment
static_assert(OFF_RING % 16 == 0, "ring entries are copied with 16-byte accesses");
static_assert(SMEM_BYTES <= 232448, "227 KiB of dynamic shared memory per CTA");

template <bool PAIR>
struct PipeCfg {   // solo: one CTA per 128x256 tile; pair: two CTAs share one 256x256 tile (cta_group::2)
    static constexpr int STAGES = PAIR ? 6 : 4;
    static constexpr int B_ROWS_DIV = PAIR ? 2 : 1;                   // each CTA of a pair stages half of the B rows
    static constexpr int STAGE_BYTES = PIPE_BYTES / STAGES;           // 32 KiB / 48 KiB
};

// gate-phase aliases of the (not yet used) pipeline stage area
constexpr int G_OFF_WG = 0;              // bf16 [EG][Hc]           <= 64 KiB
constexpr int G_WG_BYTES = 65536;
constexpr int G_OFF_LOGIT = 65536;       // f32  [TS][E+1]          <= 64 KiB
constexpr int G_LOGIT_BYTES = 65536;
constexpr int G_OFF_SEL = 131072;        // int16 sel_e[tpc*k] then int32 rank[tpc*k]   <= 48 KiB
constexpr int G_SEL_MAX = 8192;          // max tpc*k
constexpr int G_OFF_BASE = 131072 + 49152;  // int32 base[E] + total[E] + own[E]   <= 12 KiB (E <= 1024)
constexpr int G_XROWS_BYTES = 131072;       // dispatch: staged token rows (reuses the Wg / logits scratch)
static_assert(G_OFF_BASE + 12288 <= OFF_EPI, "gate scratch must fit in the stage area");

struct TileBlock {  // one contiguous run of work items: all tiles of one GEMM of one packet (or of a packet pair)
    int kind;       // 0 = GEMM0 (x.W_up^T), 1 = GEMM1 (h.W_down^T)
    int pkt;        // local packet index = src * nLx + le
    int start;      // first global item id of this block
    int pkt2;       // CTA pairs: -1 = the pair's second 128-row half is the NEXT row block of `pkt`; >= 0 = it is the SAME
                    // row block of packet pkt2 (same local expert, another source rank) -- see the host's work list
};

struct FmParams {
    CUtensorMap tm_a0;  // recv_x  as [W*nLx*pEC, H]  box {64, 128}
    CUtensorMap tm_b0;  // expert_weights as [nLx*2*P, H]  box {64, 256}  (W_up rows)
    CUtensorMap tm_a1;  // hidden  as [W*nLx*pEC, P]  box {64, 128}
    CUtensorMap tm_b1;  // expert_weights as [nLx*2*H, P]  box {64, 256}  (W_down rows)
    CUtensorMap tm_gx;  // router on tensor cores: x as [S, H], box {64, 32}
    CUtensorMap tm_gw;  // router on tensor cores: Wg_eff [E, H], box {64, E_pad} (CTA pair: {64, E_pad / 2})
    int tc_gate;        // 1 = logits by tcgen05.mma (E <= 256); 0 = register-blocked CUDA-core GEMV
    int S, H, P, E, k, W, rank, nLx, EC, pEC, TCM, act;
    int TN0, TN1, tpc, num_pkts, num_blocks, total_items;
    unsigned int epoch, phase_mask;
    unsigned long long bar_target, timeout_ns;
    const __nv_bfloat16 *x, *wg, *b_up, *b_down;
    __nv_bfloat16* out;
    int* topk_idx;             // [S,k]
    __nv_bfloat16* topk_w;     // [S,k]
    float* mcw;                // [S]
    int* slot;                 // [S,k]
    int* counts;               // [E]
    __nv_bfloat16* gate_out;   // [S,E]
    int* chunk_counts;         // [grid, E]
    unsigned int* claim;       // [1]
    unsigned int* g0_done;     // [num_pkts, TCM]
    unsigned int* g1_done;     // [num_pkts, TCM]
    unsigned long long* grid_bar;
    int* recv_cnt;             // [num_pkts]
    const TileBlock* blocks;   // [num_blocks + 1] (sentinel start = total_items)
    __nv_bfloat16* hidden;     // [W*nLx*pEC, P]
    __nv_bfloat16* recv_x;     // local symmetric: [W, nLx, pEC, H]
    unsigned long long* recv_flag;  // [W, nLx]  {epoch, rows}: published as soon as the source rank knows the count
    unsigned int* recv_rows;   // local symmetric [2, W*nLx, TCM]: rows of row block b of packet (src, le) that have landed,
                               // indexed by epoch parity (the other parity is zeroed by CTA 0 during this launch)
    __nv_bfloat16* ret_y;      // [E, pEC, H]
    unsigned long long* ret_flag;   // [E, TCM]
    __nv_bfloat16* peer_recv_x[FM_MAX_WORLD];
    unsigned long long* peer_recv_flag[FM_MAX_WORLD];
    unsigned int* peer_recv_rows[FM_MAX_WORLD];
    __nv_bfloat16* peer_ret_y[FM_MAX_WORLD];
    unsigned long long* peer_ret_flag[FM_MAX_WORLD];
    // fused GEMM1 -> combine path (fused != 0): the GEMM1 epilogue scales each row and adds it straight into the
    // source rank's output rows (peer REDG over NVLink); no return buffer, no per-row-block flags, no gather pass
    int fused;
    unsigned int* pkt_done;            // [num_pkts] GEMM1 tiles finished per packet
    uint4* recv_meta;                  // local symmetric [W*nLx*pEC] {token, p~ (f32 bits), mCw (f32 bits), 0}
    unsigned long long* done_flag;     // local symmetric [E] {epoch, 0}: expert e's contributions to my tokens are all in
    __nv_bfloat16* out_acc;            // my accumulation target: caller's out (W == 1) or the symmetric out buffer
    uint4* peer_recv_meta[FM_MAX_WORLD];
    unsigned long long* peer_done_flag[FM_MAX_WORLD];
    __nv_bfloat16* peer_out_acc[FM_MAX_WORLD];
    // training mode (is_training = 1): [2][2E+1] f32 by epoch parity = {gML[E] mean gate probability per expert,
    // gMeC[E] mean routed fraction per expert, loss} (reference moe/gate.cuh:608-635,698-706,763-773); nullptr otherwise
    float* aux;
    int dense;          // E == 1: no router GEMV, no dispatch copy; GEMM0 reads x in place (reference moe/fffn.cuh:31-167)
    DebugRecord* dbg;
    unsigned long long* trace;  // optional [grid][TRACE_SLOTS] %globaltimer stamps (nullptr = off)
};

// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void trace_stamp(const FmParams& p, int slot) {
    if (p.trace != nullptr && slot < TRACE_SLOTS)
        p.trace[(size_t)blockIdx.x * TRACE_SLOTS + slot] = globaltimer_ns();
}

__device__ __forceinline__ void grid_barrier(const FmParams& p) {
    __syncthreads();
    if (threadIdx.x == 0) {
        atom_acq_rel_gpu_add_u64(p.grid_bar, 1ull);
        SpinGuard g;
        while (ld_acquire_gpu_u64(p.grid_bar) < p.bar_target)
            g.tick(p.dbg, p.timeout_ns, FM_TRAP_GRID_BARRIER, 0, 0, 0);
    }
    __syncthreads();
}

// sum over lanes of acc[i] ends up in lane i (31 shuffles instead of 160)
__device__ __forceinline__ float warp_transpose_reduce(float (&acc)[32], int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int j = 0; j < off; ++j) {
            const float send = upper ? acc[j] : acc[j + off];
            const float keep = upper ? acc[j + off] : acc[j];
            acc[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return acc[0];
}

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
}

// ============================================================================================================
// Phase G: router.  CTA b owns tokens [b*tpc, min(S, (b+1)*tpc)).
//   logits[t,e] = sum_h x[t,h] * Wg_eff[e,h]       Wg_eff = gate_weights viewed flat as [E,H]  (moe.cuh:107-109)
//   softmax with the reference's online recurrence and fast intrinsics (gate.cuh:575-584), top-k by k rounds of
//   strict-'>' scans in ascending expert order on fp32 p (gate.cuh:654-670), mCw = sum of the picked p.
//   Slots: ascending-token order within the CTA's chunk here; chunk bases after the grid barrier (a legal
//   interleaving of the reference's BlockScan + atomicAdd(eC) order, gate.cuh:678-718).
// ============================================================================================================
// Router logits on the tensor cores (E <= 256): logits[t, e] = sum_h x[t,h] * Wg_eff[e,h] for one sub-chunk of <= 128 tokens
// of this CTA as ONE tcgen05.mma accumulator: A = the tokens' x rows (TMA, 32-row boxes straight from x), B = Wg_eff padded
// to a multiple of 16 experts (TMA; rows past E read as zero), D = [128 tokens x E_pad] fp32 in TMEM columns [0, E_pad).
// A CTA pair runs it as cta_group::2 (M = 256: each CTA's own tokens; each CTA stages half of the Wg rows), because all
// tcgen05 instructions of a kernel must use one cta_group; the two CTAs therefore walk the sub-chunks in lock-step.
// Two smem stages in the router's weight scratch (one when E_pad > 128).  Afterwards warps 0-3 copy the accumulator to
// the logits scratch (thread = token row), where the softmax / top-k code finds it exactly like after the GEMV.
// The reference computes the same product with mma.sync tiles padded to 64 experts (gate.cuh:526-535); fp32 accumulation
// order differs between the two (and from the oracle's), which is what the oracle's ambiguity flags are for.
struct GateTcState { int gkb; uint32_t accphase; };
template <bool PAIR>
__device__ __forceinline__ void gate_logits_tc(const FmParams& p, uint8_t* smem, int t0, int s0, int n_sub, int rows_span,
                                               int rows_cap, uint32_t crank, uint32_t tmem_base, float* logit_s, int ldl,
                                               GateTcState& st) {
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BARS);
    uint64_t* gfull = bars + BAR_GFULL;
    uint64_t* gempty = bars + BAR_GEMPTY;
    uint64_t* gacc = bars + BAR_GACC;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int E = p.E, E_pad = (E + 15) & ~15;
    const int b_rows = PAIR ? E_pad / 2 : E_pad;                 // Wg_eff rows this CTA stages
    const int b_bytes = b_rows * BLOCK_K * 2;
    const int nk = p.H / BLOCK_K;
    const int nb32 = (rows_span + 31) / 32;                      // 32-row boxes of x per k-block (same in both CTAs of a pair)
    const int a_bytes = nb32 * 32 * BLOCK_K * 2;                 // x rows actually staged; the MMA reads 128 rows from the stage
                                                                 // base -- rows beyond a_bytes are whatever follows (their
                                                                 // accumulator rows are never read)
    const uint32_t tx_cta = (uint32_t)(a_bytes + b_bytes);
    // stages live in the router's weight + logits scratch (the logits are written only after the last MMA of the
    // sub-chunk has completed); compact stride = what a FULL sub-chunk stages, so a 28-token chunk with 8 experts gets 8
    // stages of 5 KB.  The layout (stride, stage count, offset of the Wg rows) is the same for every sub-chunk of the
    // launch -- the stage / phase arithmetic runs across sub-chunks -- only the number of x boxes loaded follows rows_span
    // (the last sub-chunk of a CTA is usually shorter).
    const int a_cap = ((rows_cap + 31) / 32) * 32 * BLOCK_K * 2;
    const int stage_bytes = (a_cap + b_bytes + 1023) & ~1023;
    const int NS = max(1, min(GATE_STAGES, (G_WG_BYTES + G_LOGIT_BYTES - (A_STAGE_BYTES - a_cap)) / stage_bytes));
    if (warp == 0 && lane == 0) {          // TMA issuer of this CTA
        for (int kb = 0; kb < nk; ++kb) {
            const int g = st.gkb + kb, s = g % NS;
            const uint32_t ph = (uint32_t)(g / NS) & 1u;
            mbar_wait(&gempty[s], ph ^ 1u, p.dbg, p.timeout_ns, FM_TRAP_MBAR_EMPTY, 910 + s);
            uint8_t* sa = smem + G_OFF_WG + s * stage_bytes;
            if (PAIR) {
                if (crank == 0) mbar_arrive_expect_tx(&gfull[s], 2u * tx_cta);
                const uint32_t leader_full = mapa_shared(smem_u32(&gfull[s]), 0);
                for (int j = 0; j < nb32; ++j)
                    tma_load_2d_pair(sa + j * 4096, &p.tm_gx, kb * BLOCK_K, t0 + s0 + j * 32, leader_full);
                tma_load_2d_pair(sa + a_cap, &p.tm_gw, kb * BLOCK_K, (int)crank * b_rows, leader_full);
            } else {
                mbar_arrive_expect_tx(&gfull[s], tx_cta);
                for (int j = 0; j < nb32; ++j) tma_load_2d(sa + j * 4096, &p.tm_gx, kb * BLOCK_K, t0 + s0 + j * 32, &gfull[s]);
                tma_load_2d(sa + a_cap, &p.tm_gw, kb * BLOCK_K, 0, &gfull[s]);
            }
        }
    } else if (warp == 1 && lane == 0 && crank == 0) {   // MMA issuer (leader CTA)
        const uint32_t idesc = umma_idesc_bf16_f32(PAIR ? 2 * BLOCK_M : BLOCK_M, (uint32_t)E_pad);
        for (int kb = 0; kb < nk; ++kb) {
            const int g = st.gkb + kb, s = g % NS;
            const uint32_t ph = (uint32_t)(g / NS) & 1u;
            mbar_wait(&gfull[s], ph, p.dbg, p.timeout_ns, FM_TRAP_MBAR_FULL, 910 + s);
            tcgen05_fence_after();
            const uint32_t sa = smem_u32(smem + G_OFF_WG + s * stage_bytes);
            const uint64_t da = umma_smem_desc_sw128(sa);
            const uint64_t db = umma_smem_desc_sw128(sa + a_cap);
#pragma unroll
            for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
                if (PAIR) umma_bf16_ss_pair(tmem_base, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc, (kb | kk) != 0 ? 1u : 0u);
                else umma_bf16_ss(tmem_base, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc, (kb | kk) != 0 ? 1u : 0u);
            }
            if (PAIR) umma_commit_pair(&gempty[s]); else umma_commit(&gempty[s]);
        }
        if (PAIR) umma_commit_pair(gacc); else umma_commit(gacc);
    }
    st.gkb += nk;
    // accumulator complete (in a pair the commit is multicast to both CTAs' barriers)
    mbar_wait(gacc, st.accphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_TMEM_FULL, 911);
    st.accphase ^= 1u;
    tcgen05_fence_after();
    if (warp < 4) {   // TMEM lanes [32w, 32w+32) = token rows; 16 columns (experts) per load
        const int row = warp * 32 + lane;
        for (int c0 = 0; c0 < E_pad; c0 += 16) {
            uint32_t v[16];
            tmem_ld_32x32b_x16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
            tmem_ld_wait();
            if (row < n_sub) {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (c0 + i < E) logit_s[row * ldl + c0 + i] = __uint_as_float(v[i]);
            }
        }
    }
    tcgen05_fence_before();
}

// E == 1 (reference: the dense fffn kernel is selected instead of the MoE kernel, moe.cuh:174-177): every token goes to
// expert 0 with probability 1, slot = token index, nothing is dropped (EC >= S).  No GEMV, no softmax.
__device__ __forceinline__ void gate_phase_dense(const FmParams& p, int t0, int n_tok) {
    const int tid = threadIdx.x;
    for (int i = tid; i < n_tok; i += NUM_THREADS) {
        const int t = t0 + i;
        p.topk_idx[t] = 0;
        p.topk_w[t] = __float2bfloat16_rn(1.0f);
        p.mcw[t] = 1.0f;
        p.gate_out[t] = __float2bfloat16_rn(1.0f);
        p.slot[t] = t;
    }
    if (blockIdx.x == 0 && tid == 0) {
        p.counts[0] = p.S;
        p.recv_cnt[0] = p.S;
        if (p.aux != nullptr) {   // mean probability 1, routed fraction 1, loss 1 * 1 / 1
            float* a = p.aux + (size_t)(p.epoch & 1u) * 3;
            a[0] = 1.0f; a[1] = 1.0f; a[2] = 1.0f;
        }
    }
}

template <bool PAIR>
__device__ __forceinline__ void gate_phase(const FmParams& p, uint8_t* smem, int t0, int n_tok, uint32_t crank) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int E = p.E, H = p.H, k = p.k;
    __nv_bfloat16* wg_s = reinterpret_cast<__nv_bfloat16*>(smem + G_OFF_WG);
    float* logit_s = reinterpret_cast<float*>(smem + G_OFF_LOGIT);
    int16_t* sel_e = reinterpret_cast<int16_t*>(smem + G_OFF_SEL);
    int* rank_s = reinterpret_cast<int*>(smem + G_OFF_SEL + G_SEL_MAX * 2);

    float* aux_s = reinterpret_cast<float*>(smem + G_OFF_BASE + 8192);   // training: this chunk's sum_t p[t,e]
    if (p.aux != nullptr)
        for (int e = tid; e < E; e += NUM_THREADS) aux_s[e] = 0.0f;   // ordered by the block syncs of the first stage below

    uint64_t* wgbar = reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_WG;   // initialised in the kernel prologue
    uint32_t wgphase = 0;
    const int EG = E < 128 ? E : 128;                      // experts staged per group
    int Hc = (G_WG_BYTES / (EG * 2)) & ~255;               // H columns staged per chunk (multiple of 256)
    if (Hc > H) Hc = H;
    const int ldl = E + 1;                                  // padded logits row (bank spread for thread-per-row)
    int TS = G_LOGIT_BYTES / (ldl * 4);                     // tokens per sub-chunk
    const bool tc = p.tc_gate != 0;
    if (tc) TS = min(TS, BLOCK_M);                          // one tcgen05 accumulator = 128 token rows
    else if (TS > n_tok) TS = n_tok;
    // tensor-core logits: the two CTAs of a pair issue one cta_group::2 MMA per sub-chunk together, so both walk the same
    // number of sub-chunks (tpc tokens) even if this CTA owns fewer tokens
    const int span = tc ? p.tpc : n_tok;
    GateTcState tcs;
    tcs.gkb = 0; tcs.accphase = 0u;
    uint32_t tmem_base = 0;
    if (tc) {
        // TMEM was allocated in the prologue by warp 2; in a pair the partner's barriers and TMEM must exist before the
        // first remote completion / multicast commit (the grid barrier, which used to order that, comes later)
        tcgen05_fence_before();
        if (PAIR) cluster_sync_all(); else __syncthreads();
        tcgen05_fence_after();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM_PTR);
    }

    for (int s0 = 0; s0 < span; s0 += TS) {
        const int n_sub = max(0, min(TS, n_tok - s0));
        if (tc) {
            if (s0 > 0) {   // the accumulator columns and the logits scratch are reused: everybody is done with the previous ones
                tcgen05_fence_before();
                if (PAIR) cluster_sync_all(); else __syncthreads();
                tcgen05_fence_after();
            }
            gate_logits_tc<PAIR>(p, smem, t0, s0, n_sub, min(TS, p.tpc - s0), min(TS, p.tpc), crank, tmem_base, logit_s, ldl, tcs);
        } else {
        for (int i = tid; i < n_sub * ldl; i += NUM_THREADS) logit_s[i] = 0.0f;
        for (int eg0 = 0; eg0 < E; eg0 += EG) {
            const int eg_len = min(EG, E - eg0);
            for (int hc0 = 0; hc0 < H; hc0 += Hc) {
                const int hc_len = min(Hc, H - hc0);
                __syncthreads();  // previous users of wg_s are done (also orders the logit_s zero fill)
                // stage Wg_eff[eg0 .. eg0+eg_len, hc0 .. hc0+hc_len) -> wg_s[e][Hc] through the TMA engine (1-D bulk copies,
                // one per expert row, or a single one when the rows are contiguous on both sides): no register round trip,
                // and the copy runs under the x loads issued below
                if (warp == 0) {
                    if (lane == 0) {
                        fence_proxy_async_smem();   // earlier generic accesses to this scratch -> async-proxy writes
                        mbar_arrive_expect_tx(wgbar, (uint32_t)(eg_len * hc_len * 2));
                    }
                    __syncwarp();
                    if (hc_len == H && Hc == H) {
                        if (lane == 0) bulk_load_1d(wg_s, p.wg + (size_t)eg0 * H, (uint32_t)(eg_len * H * 2), wgbar);
                    } else {
                        for (int e = lane; e < eg_len; e += 32)
                            bulk_load_1d(wg_s + (size_t)e * Hc, p.wg + (size_t)(eg0 + e) * H + hc0, (uint32_t)(hc_len * 2), wgbar);
                    }
                }
                const bool single = hc_len <= 1024;
                uint4 xv[4][4];
                // the first token block's x rows (HBM) are requested while Wg is in flight, so both latencies overlap
                if (single && warp * 4 < n_sub) {
                    const int ntk0 = min(4, n_sub - warp * 4);
                    const __nv_bfloat16* xr0 = p.x + (size_t)(t0 + s0 + warp * 4) * H + hc0;
#pragma unroll
                    for (int tk = 0; tk < 4; ++tk)
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int h = i * 256 + lane * 8;
                            xv[tk][i] = (tk < ntk0 && h < hc_len) ? ld_global_nc_v4(xr0 + (size_t)tk * H + h)
                                                                  : make_uint4(0u, 0u, 0u, 0u);
                        }
                }
                mbar_wait(wgbar, wgphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_FULL, 902);
                wgphase ^= 1;
                // register-blocked GEMV: a warp takes 4 tokens x 8 experts at a time (32 accumulators per lane, one per
                // (token, expert) pair), lanes split the H columns in 16-byte pieces; all of a step's global loads are
                // issued before the first FMA, and each staged Wg piece is reused by the 4 tokens.
                for (int tb = warp * 4; tb < n_sub; tb += NUM_WARPS * 4) {
                    const int ntk = min(4, n_sub - tb);
                    const __nv_bfloat16* xr = p.x + (size_t)(t0 + s0 + tb) * H + hc0;
                    if (single && tb != warp * 4) {
#pragma unroll
                        for (int tk = 0; tk < 4; ++tk)
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int h = i * 256 + lane * 8;
                                xv[tk][i] = (tk < ntk && h < hc_len) ? ld_global_nc_v4(xr + (size_t)tk * H + h)
                                                                     : make_uint4(0u, 0u, 0u, 0u);
                            }
                    }
                    for (int g8 = 0; g8 * 8 < eg_len; ++g8) {
                        const int ne = min(8, eg_len - g8 * 8);
                        float acc[32];
#pragma unroll
                        for (int e = 0; e < 32; ++e) acc[e] = 0.0f;
                        for (int pg = 0; pg < hc_len; pg += 1024) {
                            if (!single) {
#pragma unroll
                                for (int tk = 0; tk < 4; ++tk)
#pragma unroll
                                    for (int i = 0; i < 4; ++i) {
                                        const int h = pg + i * 256 + lane * 8;
                                        xv[tk][i] = (tk < ntk && h < hc_len) ? ld_global_nc_v4(xr + (size_t)tk * H + h)
                                                                             : make_uint4(0u, 0u, 0u, 0u);
                                    }
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int h = pg + i * 256 + lane * 8;
                                if (h < hc_len) {
                                    const __nv_bfloat16* wrow = wg_s + (size_t)(g8 * 8) * Hc + h;
                                    float xf[4][8];   // the 4 tokens' 8 columns, unpacked once per piece
#pragma unroll
                                    for (int tk = 0; tk < 4; ++tk) unpack8(xv[tk][i], xf[tk]);
#pragma unroll
                                    for (int e = 0; e < 8; ++e) {
                                        if (e < ne) {
                                            float wf[8];
                                            unpack8(*reinterpret_cast<const uint4*>(wrow + (size_t)e * Hc), wf);
#pragma unroll
                                            for (int tk = 0; tk < 4; ++tk)
#pragma unroll
                                                for (int q = 0; q < 8; ++q)
                                                    acc[tk * 8 + e] = fmaf(xf[tk][q], wf[q], acc[tk * 8 + e]);
                                        }
                                    }
                                }
                            }
                        }
                        const float tot = warp_transpose_reduce(acc, lane);   // lane -> (token lane/8, expert lane%8)
                        const int tk = lane >> 3, e = lane & 7;
                        if (tk < ntk && e < ne) logit_s[(tb + tk) * ldl + eg0 + g8 * 8 + e] += tot;
                    }
                }
            }
        }
        }   // GEMV path
        __syncthreads();
        if (tid == 0) trace_stamp(p, 11);
        if (p.fused && s0 == 0 && warp == NUM_WARPS - 1) {
        // The accumulation rows of this chunk's tokens start at zero (reference clearState zeroes the output,
        // moe.cuh:43-48).  Done by the TMA engine from a zeroed piece of the (still unused) epilogue staging area, so no
        // thread stalls on a store queue (as plain stores this cost 1.5-3 us on the router's critical path wherever it was
        // placed), and issued only now, after the GEMV: the engine works in order, and at the start of the kernel these
        // stores sat in front of the gate-weight load (+5 us).  The LAST warp issues them (the softmax / top-k rounds below
        // fill the warps from 0 upwards: with config B's 28 tokens per CTA warps 7-11 have none, and as warp 4's job
        // the 3 us of this block were on the router's critical path) and waits for them in dispatch_phase before the
        // local rows are acknowledged -- an expert only adds into a token's row after an acknowledgement of this CTA.
        uint8_t* zbuf = smem + OFF_EPI;
        const int row_bytes = H * 2, zbytes = min(row_bytes, 8192);
        for (int i = lane * 16; i < zbytes; i += 512) *reinterpret_cast<uint4*>(zbuf + i) = make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async_smem();
        __syncwarp();
        const int pieces = row_bytes / zbytes;   // H is a multiple of 64, rows above 8 KiB are multiples of 8 KiB or handled below
        for (int i = lane; i < n_tok * pieces; i += 32)
            bulk_store_1d(reinterpret_cast<uint8_t*>(p.out_acc + (size_t)(t0 + i / pieces) * H) + (size_t)(i % pieces) * zbytes, zbuf,
                          (uint32_t)zbytes);
        const int rem = row_bytes - pieces * zbytes;   // (row_bytes not a multiple of 8 KiB: the tail of every row)
        if (rem > 0)
            for (int i = lane; i < n_tok; i += 32)
                bulk_store_1d(reinterpret_cast<uint8_t*>(p.out_acc + (size_t)(t0 + i) * H) + (size_t)pieces * zbytes, zbuf, (uint32_t)rem);
        bulk_commit_group();
        if (lane == 0) trace_stamp(p, 10);
    }
        if (E <= 8) {
            // E <= 8: a group of LPT = pow2ceil(E) lanes per token.  Every lane of the group runs the reference's
            // sequential online-softmax recurrence itself (gate.cuh:575-584; E <= 32 steps on broadcast smem reads, so the
            // result is bit-identical to the thread-per-row form), then lane `sub` owns expert `sub`: its probability,
            // the coalesced gateOut store, and its candidate in the k rounds of argmax -- a shuffle reduction that
            // keeps the larger value and, on equal values, the lower index = the strict-'>' ascending scan of
            // gate.cuh:654-670.
            int LPT = 1;
            while (LPT < E) LPT <<= 1;
            const int TPW = 32 / LPT, sub = lane & (LPT - 1);
            for (int tb = warp * TPW; tb < n_sub; tb += NUM_WARPS * TPW) {
                const int ti_raw = tb + lane / LPT;
                const bool valid = ti_raw < n_sub;
                const int ti = valid ? ti_raw : n_sub - 1;
                const float* l = logit_s + ti * ldl;
                const int t = t0 + s0 + ti;
                float dI = 0.0f, mI = -INFINITY;
#pragma unroll 8
                for (int e = 0; e < E; ++e) {
                    const float pM = mI;
                    mI = fmaxf(mI, l[e]);
                    dI = fmaf(dI, fast_expf(pM - mI), fast_expf(l[e] - mI));
                }
                const bool own = sub < E;
                const float pe = own ? __fdividef(fast_expf(l[sub] - mI), dI) : -INFINITY;
                if (own && valid) p.gate_out[(size_t)t * E + sub] = __float2bfloat16_rn(pe);
                bool taken = !own;
                float sum = 0.0f;
                for (int i = 0; i < k; ++i) {
                    float bv = taken ? -INFINITY : pe;
                    int bi = taken ? 0x7fffffff : sub;
                    for (int off = LPT >> 1; off >= 1; off >>= 1) {
                        const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
                        const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
                    }
                    if (bi == sub) taken = true;
                    sum += bv;
                    if (sub == 0 && valid) {
                        p.topk_idx[(size_t)t * k + i] = bi;
                        p.topk_w[(size_t)t * k + i] = __float2bfloat16_rn(bv);
                        sel_e[(s0 + ti) * k + i] = (int16_t)bi;
                    }
                }
                if (sub == 0 && valid) p.mcw[t] = sum;
                __syncwarp();
                if (own && valid) logit_s[ti * ldl + sub] = pe;   // probabilities (training-mode column sums read them)
            }
        } else if (E <= 1024) {
            // 8 < E <= 1024: the same scheme with C = ceil(E / LPT) <= 32 experts per lane (lane `sub` owns experts sub,
            // sub + LPT, ...): 8 / 4 / 2 / 1 tokens per warp, so that a sub-chunk of up to 96 tokens is one round of the CTA's
            // 12 warps (the recurrence is a dependent chain of E steps per token whatever the lane count; one lane per
            // expert would serialise 111 tokens of the 16k-token sweep point into 10 rounds, a thread per token leaves one
            // or two warps doing ~5 E dependent steps each: 17 us at E = 128 with 56 tokens).  Every lane of a group runs the sequential
            // recurrence itself; a lane scans its own experts in ascending order with a strict '>', the group reduction
            // prefers the larger value and, on equal values, the lower index -- together the reference's ascending scan.
            const int LPT = E <= 128 ? 4 : E <= 256 ? 8 : E <= 512 ? 16 : 32;
            const int TPW = 32 / LPT, sub = lane & (LPT - 1);
            for (int tb = warp * TPW; tb < n_sub; tb += NUM_WARPS * TPW) {
                const int ti_raw = tb + lane / LPT;
                const bool valid = ti_raw < n_sub;
                const int ti = valid ? ti_raw : n_sub - 1;   // (idle groups compute on a copy of the last row, write nothing)
                float* l = logit_s + ti * ldl;
                const int t = t0 + s0 + ti;
                float dI = 0.0f, mI = -INFINITY;
                // (unrolled so that the loads, the running maxima and the exponentials of 8 steps are in flight together;
                // the dependent chain is then one max and one fma per step -- same operations in the same order)
#pragma unroll 8
                for (int e = 0; e < E; ++e) {
                    const float pM = mI;
                    mI = fmaxf(mI, l[e]);
                    dI = fmaf(dI, fast_expf(pM - mI), fast_expf(l[e] - mI));
                }
                __syncwarp();   // every lane of the group has read the logits before they are replaced by probabilities
                if (valid)
#pragma unroll 4
                    for (int e = sub; e < E; e += LPT) {
                        const float pe = __fdividef(fast_expf(l[e] - mI), dI);
                        l[e] = pe;
                        p.gate_out[(size_t)t * E + e] = __float2bfloat16_rn(pe);
                    }
                unsigned int taken = 0u;
                float sum = 0.0f;
                for (int i = 0; i < k; ++i) {
                    float bv = -INFINITY;
                    int bi = 0x7fffffff;
                    if (valid) {
                        int c = 0;
#pragma unroll 4
                        for (int e = sub; e < E; e += LPT, ++c) {
                            const float v = l[e];
                            if (v > bv && !((taken >> c) & 1u)) { bv = v; bi = e; }
                        }
                    }
                    for (int off = LPT >> 1; off >= 1; off >>= 1) {
                        const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
                        const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
                    }
                    if (bi == 0x7fffffff) { bi = 0; }   // nothing comparable left (NaN logits): the thread-per-token form's default
                    if ((bi & (LPT - 1)) == sub) taken |= 1u << (bi / LPT);
                    sum += bv;
                    if (sub == 0 && valid) {
                        p.topk_idx[(size_t)t * k + i] = bi;
                        p.topk_w[(size_t)t * k + i] = __float2bfloat16_rn(bv);
                        sel_e[(s0 + ti) * k + i] = (int16_t)bi;
                    }
                }
                if (sub == 0 && valid) p.mcw[t] = sum;
                __syncwarp();
            }
        } else
        // thread-per-token softmax + top-k, the same per-thread recurrence the reference runs after its transpose
        for (int ti = tid; ti < n_sub; ti += NUM_THREADS) {
            float* l = logit_s + ti * ldl;
            const int t = t0 + s0 + ti;
            float dI = 0.0f, mI = -INFINITY;
            for (int e = 0; e < E; ++e) {
                const float pM = mI;
                mI = fmaxf(mI, l[e]);
                dI = fmaf(dI, fast_expf(pM - mI), fast_expf(l[e] - mI));
            }
            for (int e = 0; e < E; ++e) {
                const float pe = __fdividef(fast_expf(l[e] - mI), dI);
                l[e] = pe;
                p.gate_out[(size_t)t * E + e] = __float2bfloat16_rn(pe);
            }
            int picked[8];
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                picked[i] = -1;
                if (i < k) {
                    float sV = -INFINITY;
                    int sIdx = 0;
                    for (int j = 0; j < E; ++j) {
                        bool taken = false;
#pragma unroll
                        for (int q = 0; q < 8; ++q) taken |= (q < i) && (picked[q] == j);
                        if (l[j] > sV && !taken) {
                            sIdx = j;
                            sV = l[j];
                        }
                    }
                    picked[i] = sIdx;
                    sum += sV;
                    p.topk_idx[(size_t)t * k + i] = sIdx;
                    p.topk_w[(size_t)t * k + i] = __float2bfloat16_rn(sV);
                    sel_e[(s0 + ti) * k + i] = (int16_t)sIdx;
                }
            }
            p.mcw[t] = sum;
        }
        if (tid == 0) trace_stamp(p, 15);
        __syncthreads();
        if (p.aux != nullptr) {
            // column sums of the fp32 probabilities of this sub-chunk (the reference block-reduces each gate tile's
            // columns, gate.cuh:611-627): warp w owns experts w, w + NUM_WARPS, ...; lanes stride over the tokens
            for (int e = warp; e < E; e += NUM_WARPS) {
                float acc = 0.0f;
                for (int ti = lane; ti < n_sub; ti += 32) acc += logit_s[ti * ldl + e];
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
                if (lane == 0) aux_s[e] += acc;
            }
            __syncthreads();
        }
    }
    if (tid == 0) trace_stamp(p, 12);
    // The Wg / logits scratch is free from here on: start staging this chunk's token rows for the dispatch phase now
    // (one bulk load, same barrier and layout dispatch_phase expects for its first group), so the load runs under the
    // slot ranks, the grid barrier and the prefix pass instead of after them.
    if (tid == 32 && n_tok > 0) {   // (warp 1: warp 0 is about to compute the slot ranks)
        const int row_bytes = H * 2;
        const int rows0 = max(1, min(n_tok, G_XROWS_BYTES / row_bytes));
        uint64_t* xbar = reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_XROWS;
        fence_proxy_async_smem();
        mbar_arrive_expect_tx(xbar, (uint32_t)(rows0 * row_bytes));
        bulk_load_1d(smem, p.x + (size_t)t0 * H, (uint32_t)(rows0 * row_bytes), xbar);
    }
    if (p.aux != nullptr) {   // gML[e] += (sum over this chunk) / S   (gate.cuh:628-634: atomicAdd(gML + e, colAgg / S))
        float* gml = p.aux + (size_t)(p.epoch & 1u) * (2 * E + 1);
        for (int e = tid; e < E; e += NUM_THREADS) atomicAdd(gml + e, __fdividef(aux_s[e], (float)p.S));
    }
    // position of every (token, pick) among this chunk's selections of the same expert, ascending (token, pick) order.
    // One warp walks the entries 32 at a time: lanes holding the same expert find each other with match.any, the rank
    // inside the group is a popcount, the running per-expert count lives in shared memory (O(n) instead of O(n^2);
    // the 64k-token sweep point has 886 entries per CTA).
    int* cnt_s = reinterpret_cast<int*>(smem + G_OFF_BASE);
    for (int e = tid; e < E; e += NUM_THREADS) cnt_s[e] = 0;
    __syncthreads();
    const int n_ent = n_tok * k;
    if (warp == 0) {
        for (int i0 = 0; i0 < n_ent; i0 += 32) {
            const int i = i0 + lane;
            const bool valid = i < n_ent;
            const int e = valid ? (int)sel_e[i] : (E + lane);        // invalid lanes get unique keys
            const unsigned int same = __match_any_sync(0xffffffffu, e);
            const unsigned int before = same & ((1u << lane) - 1u);
            if (valid) rank_s[i] = cnt_s[e] + __popc(before);
            __syncwarp();
            if (valid && before == 0u) cnt_s[e] += __popc(same);    // one lane per distinct expert of the group
            __syncwarp();
        }
    }
    __syncthreads();
    for (int e = tid; e < E; e += NUM_THREADS) p.chunk_counts[(size_t)blockIdx.x * E + e] = cnt_s[e];
}

// ============================================================================================================
// Phase D: dispatch (after the grid barrier).  slot = (selections of e by lower chunks) + rank in chunk; kept iff
// slot < EC (gate.cuh:713-717).  Whole token rows go straight into the owner rank's receive buffer (peer-mapped, NVLink)
// -- the reference's P2P branch (os/packet.cuh:114-116,151-166) -- as TMA bulk copies staged through shared memory.
// Signalling (os/packet.cuh:214-237 sends one {rows, tiles, seq} word per (source, expert) once the LAST of its dispatch
// CTAs is done): here the 8-byte {epoch, rows} flag is published as soon as the count is known -- right after the
// prefix pass, before any row moves (also for 0 rows, like the reference's "noop" signal) -- and the data itself is
// acknowledged per 128-row block: every CTA adds the number of rows it has landed in block b of packet (me, e) to the
// owner's arrival counter recv_rows[epoch parity][pkt][b] with a release at system scope.  A GEMM0 tile starts when ITS
// row blocks are complete, not when the slowest CTA of the source rank has finished.
// Runs on warps 2, 4-11 only (see the kernel body).
// ============================================================================================================
constexpr int DISP_THREADS = 288;   // warps 2, 4..11; warps 0, 1, 3 are already in their FFN roles (producer / MMA / scheduler)
__device__ __forceinline__ void disp_sync() { asm volatile("bar.sync 2, 288;" ::: "memory"); }

__device__ __forceinline__ void dispatch_phase(const FmParams& p, uint8_t* smem, int t0, int n_tok) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tid = (warp == 2 ? 0 : (warp - 3) * 32) + lane;   // 0..287 within the dispatch subset
    const int E = p.E, H = p.H, k = p.k, G = gridDim.x;
    const int16_t* sel_e = reinterpret_cast<const int16_t*>(smem + G_OFF_SEL);
    const int* rank_s = reinterpret_cast<const int*>(smem + G_OFF_SEL + G_SEL_MAX * 2);
    int* base_s = reinterpret_cast<int*>(smem + G_OFF_BASE);        // selections of e by lower chunks
    int* total_s = base_s + 1024;                                    // selections of e by all chunks
    int* own_s = base_s + 2048;                                      // selections of e by this chunk

    // one pass over chunk_counts [G, E] gives the prefix (lower chunks), this chunk's own counts and the totals
    for (int e = tid; e < E; e += DISP_THREADS) { base_s[e] = 0; total_s[e] = 0; }
    disp_sync();
    const int E4 = E >> 2;
    if ((E & 3) == 0 && E4 <= DISP_THREADS && (DISP_THREADS % E4) == 0) {
        // 16-byte loads, four experts at a time; a thread always meets the same four (DISP_THREADS is a multiple of E / 4),
        // so it sums in registers and touches shared memory once.  (E = 128: 2 batches of loads instead of 9.)
        const int nb4 = (int)blockIdx.x * E4, n4 = G * E4;
        int pt[4] = {0, 0, 0, 0}, pb[4] = {0, 0, 0, 0};
        for (int i0 = tid; i0 < n4; i0 += 8 * DISP_THREADS) {
            int4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * DISP_THREADS;
                v[u] = i < n4 ? ld_global_cg_i4(reinterpret_cast<const int4*>(p.chunk_counts) + i) : make_int4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * DISP_THREADS;
                if (i >= n4) break;
                if (i >= nb4 && i < nb4 + E4) *reinterpret_cast<int4*>(own_s + 4 * (i - nb4)) = v[u];
                pt[0] += v[u].x; pt[1] += v[u].y; pt[2] += v[u].z; pt[3] += v[u].w;
                if (i < nb4) { pb[0] += v[u].x; pb[1] += v[u].y; pb[2] += v[u].z; pb[3] += v[u].w; }
            }
        }
        if (tid < n4) {
            const int e0 = 4 * (tid % E4);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (pt[q] != 0) atomicAdd(&total_s[e0 + q], pt[q]);
                if (pb[q] != 0) atomicAdd(&base_s[e0 + q], pb[q]);
            }
        }
    } else {
        const int nb = (int)blockIdx.x * E, n = G * E;
        const bool fixed_e = (E <= DISP_THREADS) && (DISP_THREADS % E) == 0;   // then a thread always meets one e
        int part_b = 0, part_t = 0, cur_e = -1;
        for (int i0 = tid; i0 < n; i0 += 8 * DISP_THREADS) {
            int v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {   // all loads of the batch are in flight before the first use
                const int i = i0 + u * DISP_THREADS;
                v[u] = i < n ? p.chunk_counts[i] : 0;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * DISP_THREADS;
                if (i >= n) break;
                const int e = i % E;
                if (i >= nb && i < nb + E) own_s[e] = v[u];
                if (fixed_e) { part_t += v[u]; if (i < nb) part_b += v[u]; cur_e = e; }
                else if (v[u] != 0) { atomicAdd(&total_s[e], v[u]); if (i < nb) atomicAdd(&base_s[e], v[u]); }
            }
        }
        if (cur_e >= 0) {
            if (part_t != 0) atomicAdd(&total_s[cur_e], part_t);
            if (part_b != 0) atomicAdd(&base_s[cur_e], part_b);
        }
    }
    disp_sync();
    if (tid == 0) trace_stamp(p, 8);
    // the count of packet (me, e) is known: CTA (e mod G) tells the owner now.  Nothing precedes this word that the
    // reader depends on (the rows are acknowledged through recv_rows), so a relaxed system-scope store is enough.
    for (int e = (int)blockIdx.x + tid * G; e < E; e += DISP_THREADS * G) {
        const int tot = total_s[e];
        p.counts[e] = tot;
        const int rows = tot < p.EC ? tot : p.EC;
        const int owner = e / p.nLx, le = e - owner * p.nLx;
        st_relaxed_sys_u64(p.peer_recv_flag[owner] + (size_t)p.rank * p.nLx + le,
                           ((unsigned long long)p.epoch << 32) | (unsigned int)rows);
        if (p.aux != nullptr) {
            // gMeC[e] = selections of e / S (gate.cuh:698-706 adds each tile's count / S; the chunk totals are summed
            // first here), loss += gML[e] * gMeC[e] / E (gate.cuh:763-773).  Every CTA's gML atomics precede its arrival
            // at the grid barrier, so gML is complete here.
            float* a = p.aux + (size_t)(p.epoch & 1u) * (2 * E + 1);
            const float ce = __fdividef((float)tot, (float)p.S);
            a[E + e] = ce;
            const float me = *reinterpret_cast<volatile float*>(a + e);
            atomicAdd(a + 2 * E, __fdividef(me * ce, (float)E));
        }
    }
    const unsigned int par = p.epoch & 1u;
    // Row copies.
    //   * Rows for experts on THIS rank (warps 4-11): the chunk's token rows are contiguous in x, so one bulk load stages up
    //     to 128 KiB of them in shared memory (the first group was requested at the end of the router) and every kept
    //     (token, pick) pair is one cp.async.bulk store of a whole row through the TMA engine (no per-lane chains).  They
    //     land in ~4 us and are acknowledged at once (gpu-scope release); the stage area is handed to the TMA producer, the
    //     warps become epilogue warps, and the expert FFN starts on the local packets while
    //   * rows for experts on OTHER ranks (warp 2, from the moment the slots are known) cross NVLink as 16-byte peer stores
    //     read straight from x (L2 hits), sixteen pieces per lane in flight.  The link bounds them (S*k*(1-1/W)*H*2 bytes
    //     at ~770 GB/s) and back-pressures the issuing warp -- which has no other duty until the first tile needs
    //     publishing; it then waits for the stores with a system-scope release and acknowledges them.
    uint64_t* xbar = reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_XROWS;   // initialised in the kernel prologue
    uint8_t* x_s = smem;   // the router's Wg / logits scratch is free now
    const int row_bytes = H * 2;
    const int rows_per_group = max(1, min(n_tok, G_XROWS_BYTES / row_bytes));
    const bool any_remote = p.W > 1;
    const int first_local = p.rank * p.nLx;
    auto ack = [&](int e, int lo, int hi, bool local) {
        // this chunk's rows of expert e occupy slots [lo, hi) of packet (me, e): add the rows landed per 128-row block.
        // The release covers every store of the threads that met at the preceding barrier.
        if (hi <= lo) return;
        const int owner = e / p.nLx, le = e - owner * p.nLx;
        unsigned int* ctr = p.peer_recv_rows[owner] + ((size_t)par * p.num_pkts + (size_t)(p.rank * p.nLx + le)) * p.TCM;
        for (int b = lo / BLOCK_M; b <= (hi - 1) / BLOCK_M; ++b) {
            const int n = min(hi, (b + 1) * BLOCK_M) - max(lo, b * BLOCK_M);
            if (local) red_release_gpu_add_u32(ctr + b, (unsigned int)n);
            else red_release_sys_add_u32(ctr + b, (unsigned int)n);
        }
    };
    constexpr int LOCAL_THREADS = DISP_THREADS - 32;   // warps 4..11
    if (warp != 2) {
        // ---------------------------------------------------------------- warps 4-11: slots, routing records, local rows
        const int ltid = tid - 32;
        uint32_t xphase = 0;
        for (int g0 = 0; g0 < n_tok; g0 += rows_per_group) {
            const int rows = min(rows_per_group, n_tok - g0);
            if (ltid == 0 && g0 > 0) {   // group 0 was requested at the end of the router (gate_phase)
                mbar_arrive_expect_tx(xbar, (uint32_t)(rows * row_bytes));
                bulk_load_1d(x_s, p.x + (size_t)(t0 + g0) * H, (uint32_t)(rows * row_bytes), xbar);
            }
            mbar_wait(xbar, xphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_FULL, 900);
            xphase ^= 1;
            for (int i = ltid; i < rows * k; i += LOCAL_THREADS) {   // one thread per (token, pick)
                const int tl = i / k, j = i - tl * k;
                const int ti = g0 + tl, t = t0 + ti;
                const int e = sel_e[ti * k + j];
                const int s = base_s[e] + rank_s[ti * k + j];
                p.slot[(size_t)t * k + j] = s;
                if (s < p.EC) {
                    const int owner = e / p.nLx, le = e - owner * p.nLx;
                    const size_t row = (size_t)(p.rank * p.nLx + le) * p.pEC + s;
                    if (p.fused) {   // what the expert's GEMM1 epilogue needs to combine this row
                        uint4 m;
                        m.x = (unsigned int)t;
                        m.y = __float_as_uint(__bfloat162float(p.topk_w[(size_t)t * k + j]));
                        m.z = __float_as_uint(p.mcw[t]);
                        m.w = 0u;
                        st_global_v4(p.peer_recv_meta[owner] + row, m);
                    }
                    if (owner == p.rank)
                        bulk_store_1d(p.recv_x + row * H, x_s + (size_t)tl * row_bytes, (uint32_t)row_bytes);
                }
            }
            bulk_commit_group();
            if (g0 + rows_per_group < n_tok) {   // the staging buffer is reused: wait until the bulk stores have read it
                bulk_wait_group_read0();
                asm volatile("bar.sync 4, 256;" ::: "memory");
            }
        }
        // (the zero-fill stores, an older bulk group of warp 11, read the first 8 KiB of the epilogue staging area, which
        // is warp 2's window: they must have been read before warp 2 starts -- all but the newest group, the row stores)
        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        if (any_remote) asm volatile("bar.arrive 3, 288;" ::: "memory");   // every slot (p.slot) is written: warp 2 may start
        bulk_wait_group0();        // this thread's local row stores (and warp 11's zero-fill stores) are complete ...
        fence_proxy_async_all();   // ... and ordered (async proxy) before the generic-proxy counter traffic below
        asm volatile("bar.sync 4, 256;" ::: "memory");
        if (any_remote) asm volatile("bar.arrive 6, 288;" ::: "memory");   // local rows + zero-fill complete (warp 2's acks wait for this)
        if (ltid == 0) trace_stamp(p, 9);
        if (any_remote) asm volatile("bar.sync 5, 288;" ::: "memory");   // warp 2 has taken what it needs from the stage area
        if (ltid < 32) {   // warp 4: acknowledge the local experts, then hand the stage area to the TMA producer
            for (int e = first_local + ltid; e < first_local + p.nLx; e += 32) ack(e, base_s[e], min(base_s[e] + own_s[e], p.EC), true);
            __syncwarp();
            // (more than 256 experts on several ranks: warp 2 still needs base / own for its acknowledgements and releases)
            if (ltid == 0 && (!any_remote || E <= 256)) mbar_arrive(reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_DISP_DONE);
        }
        return;
    }
    // -------------------------------------------------------------------- warp 2
    if (!any_remote) return;
    // the slot ranges of the remote experts go into registers (E <= 256) before the stage area -- where base / own live --
    // is released by warp 4; beyond that the release waits for this warp
    constexpr int RMAX = 8;
    int rlo[RMAX], rhi[RMAX];
    const bool in_regs = E <= 32 * RMAX;
#pragma unroll
    for (int i = 0; i < RMAX; ++i) {
        const int e = lane + 32 * i;
        const bool remote = in_regs && e < E && (e < first_local || e >= first_local + p.nLx);
        rlo[i] = remote ? base_s[e] : 0;
        rhi[i] = remote ? min(base_s[e] + own_s[e], p.EC) : 0;
    }
    __syncwarp();
    if (in_regs) asm volatile("bar.arrive 5, 288;" ::: "memory");   // done with the stage area
    asm volatile("bar.sync 3, 288;" ::: "memory");                  // every slot of this chunk (p.slot) is written
    {
        // Remote rows through the TMA engine (SM-issued peer stores reached only ~400 GB/s over NVLink, bulk stores ~600):
        // a window of the epilogue staging area -- unused until this CTA's first tile is complete; its first 8 KiB hold the
        // zero source of the output zero-fill -- is filled with a run of consecutive token rows of x (one bulk load), every
        // kept (token, pick) pair of those tokens that belongs to another rank is one bulk store of a whole row to that
        // rank's receive buffer, and when the engine has read the window the next run follows.  The link paces the stores.
        uint8_t* win = smem + OFF_EPI + 8192;
        const int win_bytes = NUM_EPI_WARPS * EPI_WARP_BYTES - 8192;
        const int rows_win = max(1, win_bytes / row_bytes);
        uint64_t* rbar = reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_REMOTE;
        uint32_t rphase = 0;
        const bool fits = row_bytes <= win_bytes;   // (d_model > 12288: rows go piecewise, below)
        for (int tw = 0; tw < n_tok; tw += rows_win) {
            const int rows = min(rows_win, n_tok - tw);
            // does any pair of these tokens go to another rank?  (expert and slot from the routing tables in global memory)
            bool mine = false;
            for (int i = lane; i < rows * k; i += 32) {
                const size_t gi = (size_t)(t0 + tw) * k + i;
                const int owner = p.topk_idx[gi] / p.nLx;
                mine |= owner != p.rank && p.slot[gi] < p.EC;
            }
            const unsigned int anyone = __ballot_sync(0xffffffffu, mine);
            if (anyone == 0u) continue;
            if (fits) {
                if (lane == 0) {
                    fence_proxy_async_smem();
                    mbar_arrive_expect_tx(rbar, (uint32_t)(rows * row_bytes));
                    bulk_load_1d(win, p.x + (size_t)(t0 + tw) * H, (uint32_t)(rows * row_bytes), rbar);
                }
                mbar_wait(rbar, rphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_FULL, 903);
                rphase ^= 1;
                for (int i = lane; i < rows * k; i += 32) {
                    const size_t gi = (size_t)(t0 + tw) * k + i;
                    const int e = p.topk_idx[gi];
                    const int owner = e / p.nLx;
                    const int sl = p.slot[gi];
                    if (owner != p.rank && sl < p.EC)
                        bulk_store_1d(p.peer_recv_x[owner] + ((size_t)(p.rank * p.nLx + (e - owner * p.nLx)) * p.pEC + sl) * H,
                                      win + (size_t)(i / k) * row_bytes, (uint32_t)row_bytes);
                }
                bulk_commit_group();
                bulk_wait_group_read0();   // the engine has read the window
                __syncwarp();
            } else {
                // very wide rows: one token at a time, in window-sized pieces
                for (int off = 0; off < row_bytes; off += win_bytes) {
                    const int nb = min(win_bytes, row_bytes - off);
                    if (lane == 0) {
                        fence_proxy_async_smem();
                        mbar_arrive_expect_tx(rbar, (uint32_t)nb);
                        bulk_load_1d(win, reinterpret_cast<const uint8_t*>(p.x + (size_t)(t0 + tw) * H) + off, (uint32_t)nb, rbar);
                    }
                    mbar_wait(rbar, rphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_FULL, 904);
                    rphase ^= 1;
                    for (int i = lane; i < k; i += 32) {
                        const size_t gi = (size_t)(t0 + tw) * k + i;
                        const int e = p.topk_idx[gi];
                        const int owner = e / p.nLx;
                        const int sl = p.slot[gi];
                        if (owner != p.rank && sl < p.EC)
                            bulk_store_1d(reinterpret_cast<uint8_t*>(p.peer_recv_x[owner] +
                                              ((size_t)(p.rank * p.nLx + (e - owner * p.nLx)) * p.pEC + sl) * H) + off,
                                          win, (uint32_t)nb);
                    }
                    bulk_commit_group();
                    bulk_wait_group_read0();
                    __syncwarp();
                }
            }
        }
        asm volatile("bar.arrive 7, 288;" ::: "memory");   // the staging area belongs to the epilogue warps from here
        bulk_wait_group0();        // the rows have arrived on the other ranks ...
        fence_proxy_async_all();   // ... and are ordered before the generic-proxy acknowledgements
    }
    __syncwarp();
    // the remote acknowledgements also tell the peers that this chunk's output rows are zeroed (TMA stores issued by warp 11
    // in the router, completed before it arrives here) and that the routing records are written
    asm volatile("bar.sync 6, 288;" ::: "memory");
    if (in_regs) {
#pragma unroll
        for (int i = 0; i < RMAX; ++i) ack(lane + 32 * i, rlo[i], rhi[i], false);
    } else {
        for (int e = lane; e < E; e += 32)
            if (e < first_local || e >= first_local + p.nLx) ack(e, base_s[e], min(base_s[e] + own_s[e], p.EC), false);
        __syncwarp();
        asm volatile("bar.arrive 5, 288;" ::: "memory");
        if (lane == 0) mbar_arrive(reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_DISP_DONE);
    }
}

// ============================================================================================================
// Phase F: expert FFN.  Work items (global order, claimed with one atomic counter by the pair's scheduler warp):
//   runs of all tiles of one GEMM of one packet, in the order of the host's build_work_list (own rank's packets first,
//   then rank+1, ...).  item -> (row-block pair m fastest, column tile n).  The item list is a static superset: row
//   blocks beyond the packet's row count are skipped once the packet flag is known.  A GEMM1 tile waits for
//   g0_done[pkt][m] == TN0 (both row blocks of the pair).
// ============================================================================================================
struct TileInfo {     // 64 bytes, written by the (leader's) scheduler warp, read by producer / MMA / epilogue / publisher warps.
                      // Per-half fields are indexed by the CTA's rank in the pair (solo CTAs use index 0).
    int kind;         // 0 GEMM0, 1 GEMM1, -1 stop
    int ntile;
    int le;           // local expert (both halves share it: same B operand)
    int b_row;        // TMA row coordinate of the B tile (rank 1 of a pair: + BLOCK_N/2)
    int pad[2];       // keeps the struct at 4 x 16 bytes (ring slot size, DSMEM mirror)
    int pkt[2];       // local packet index src * nLx + le of each half
    int mblk[2];      // 128-row block of that packet
    int rows[2];      // valid rows of that block (0 = this half is idle)
    int src[2];       // source rank of the packet
    int cnt[2];       // rows of the whole packet
};
static_assert(sizeof(TileInfo) == 64, "TileInfo must be 4 x 16 bytes");

template <bool PAIR>
__device__ __forceinline__ void wait_sched_full(const FmParams& p, uint64_t* bar, uint32_t parity, unsigned int info) {
    if (PAIR) mbar_wait_cluster(bar, parity, p.dbg, p.timeout_ns, FM_TRAP_MBAR_SCHED_FULL, info);  // data came over DSMEM
    else mbar_wait(bar, parity, p.dbg, p.timeout_ns, FM_TRAP_MBAR_SCHED_FULL, info);
}
// consumers of a ring slot release it on the LEADER's barrier (the scheduler lives there)
template <bool PAIR>
__device__ __forceinline__ void release_to_leader(uint64_t* bar, uint32_t crank) {
    if (PAIR && crank != 0) mbar_arrive_cluster_plain(bar, 0);
    else mbar_arrive(bar);
}

// warp 3 (leader CTA in pair mode): claims work items and resolves their dependencies AHEAD of the TMA producer, so the
// atomic, the packet-flag and the h-row-block-counter round trips overlap the previous tile's loads (the job of the
// reference's OS CTA: subscriber decode + scheduler doorbells, os/subscriber.cuh, os/scheduler.cuh -- here one warp, no queues).
template <bool PAIR>
__device__ __forceinline__ void ffn_scheduler(const FmParams& p, uint8_t* smem, uint64_t* bars) {
    uint64_t* sched_full = bars + BAR_SCHED_FULL;
    uint64_t* sched_empty = bars + BAR_SCHED_EMPTY;
    uint64_t* prod_take = bars + BAR_PROD_TAKE;
    TileInfo* ring = reinterpret_cast<TileInfo*>(smem + OFF_RING);
    const int lane = threadIdx.x & 31;
    const int nh = PAIR ? 2 : 1;                            // 128-row halves per work item
    int q = 0, qphase = 0, cursor = 0, n = 0;
    bool seen_remote = false;   // trace only: first tile of a packet from another rank
    for (;;) {
        if (lane == 0 && n >= 1) {  // bounded look-ahead: wait until the producer is close to finishing tile n-1
            const int pq = (q + NSCHED - 1) % NSCHED;
            mbar_wait(&prod_take[pq], ((n - 1) / NSCHED) & 1, p.dbg, p.timeout_ns, FM_TRAP_MBAR_SCHED_EMPTY, 200 + pq);
        }
        __syncwarp();
        // The whole warp walks the claim loop in lock-step; lane h resolves the dependencies of half h of the item (the
        // two halves' flag / counter round trips overlap), lane 0 assembles and publishes the descriptor.
        int kind = -1, nt = 0, le = 0;
        int h_pkt = 0, h_mb = 0, h_src = 0, h_rows = 0, h_cnt = 0;
        for (;;) {
            int id = 0;
            if (lane == 0) id = (int)atomicAdd(p.claim, 1u);
            id = __shfl_sync(0xffffffffu, id, 0);
            if (id >= p.total_items) break;
            if (lane == 0 && n < 16) trace_stamp(p, 112 + n);   // claim time of tile n (ready time is slot 16+n)
            while (id >= p.blocks[cursor + 1].start) ++cursor;
            const TileBlock blk = p.blocks[cursor];
            const int local = id - blk.start;
            // item -> (row block(s), column tile); row blocks fastest.  Within-packet pairing: halves = row blocks
            // 2m, 2m+1 of one packet.  Cross-source pairing (pkt2 >= 0): halves = row block m of two packets.
            const bool cross = PAIR && blk.pkt2 >= 0;
            const int m_items = (PAIR && !cross) ? (p.TCM + 1) / 2 : p.TCM;
            const int m = local % m_items;
            nt = local / m_items;
            le = blk.pkt % p.nLx;
            const int h = lane;
            h_pkt = (h == 1 && cross) ? blk.pkt2 : blk.pkt;
            h_mb = cross ? m : (PAIR ? 2 * m + (h & 1) : m);
            h_src = h_pkt / p.nLx;
            h_rows = 0; h_cnt = 0;
            if (h < nh && h_mb < p.TCM) {
                const bool same_gpu = h_src == p.rank;   // flag and counters written from this GPU: gpu scope suffices
                // wait for the packet (src, le): flag = {epoch, rows}  (reference subscriber.cuh:52-185)
                unsigned long long f = ((unsigned long long)p.epoch << 32) | (unsigned int)p.S;   // dense: all S rows, in x
                bool stale = false;
                if (!p.dense) {
                    SpinGuard g;
                    for (;;) {
                        f = same_gpu ? ld_acquire_gpu_u64(p.recv_flag + h_pkt) : ld_acquire_sys_u64(p.recv_flag + h_pkt);
                        const int ahead = (int)((unsigned int)(f >> 32) - p.epoch);
                        if (ahead == 0) break;
                        // The source rank is already in a LATER forward: it only gets there after every real tile of
                        // this packet has been returned to it, so whatever item of the static superset is left here
                        // is an empty row block.
                        if (ahead > 0) { stale = true; break; }
                        g.tick(p.dbg, p.timeout_ns, FM_TRAP_RECV_FLAG, h_pkt, (unsigned int)(f >> 32), p.epoch);
                    }
                }
                if (!stale) {
                    h_cnt = (int)(f & 0xffffffffull);
                    if (h == 0 || cross) {   // once per packet and GEMM (its first item): bookkeeping that needs the count
                        if (local == 0 && blk.kind == 0 && !p.dense) p.recv_cnt[h_pkt] = h_cnt;
                        if (p.fused && local == 0 && blk.kind == 1 && h_cnt == 0)   // nothing to contribute: tell the source now
                            st_release_sys_u64(p.peer_done_flag[h_src] + (size_t)(p.rank * p.nLx + le),
                                               (unsigned long long)p.epoch << 32);
                    }
                    h_rows = max(0, min(BLOCK_M, h_cnt - h_mb * BLOCK_M));
                }
                if (h_rows > 0) {
                    SpinGuard g;
                    const unsigned int* rctr = p.recv_rows + ((size_t)(p.epoch & 1u) * p.num_pkts + h_pkt) * p.TCM + h_mb;
                    if (blk.kind == 1) {  // GEMM1 needs the whole h row block (reference notifyNext, processor.cuh:490-615)
                        const unsigned int* ctr = p.g0_done + (size_t)h_pkt * p.TCM + h_mb;
                        while (ld_acquire_gpu_u32(ctr) < (unsigned int)p.TN0)
                            g.tick(p.dbg, p.timeout_ns, FM_TRAP_G0_DONE, h_pkt, h_mb, 0);
                    } else if ((p.phase_mask & 1u) && !p.dense) {  // GEMM0 needs the rows of this block to have landed (dispatch acks)
                        for (;;) {
                            const unsigned int got = same_gpu ? ld_acquire_gpu_u32(rctr) : ld_acquire_sys_u32(rctr);
                            if (got >= (unsigned int)h_rows) break;
                            g.tick(p.dbg, p.timeout_ns, FM_TRAP_RECV_ROWS, h_pkt, h_mb, h_rows);
                        }
                    }
                }
            }
            __syncwarp();
            const bool any = __any_sync(0xffffffffu, h_rows > 0 && lane < nh);
            if (!any) continue;   // every half is an empty row block of the static superset
            kind = blk.kind;
            break;
        }
        // lane 0 collects both halves
        TileInfo ti;
        ti.kind = kind; ti.ntile = nt; ti.le = le;
        // expert_weights [nLx,2,P,H]: W_up(le) starts at row le*2*P of the [.,H] view; W_down(le) (the [P,H]
        // block flat-viewed as [H,P]) starts at row (le*2+1)*H of the [.,P] view.
        ti.b_row = kind < 0 ? 0 : (kind == 0 ? le * 2 * p.P : (le * 2 + 1) * p.H) + nt * BLOCK_N;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            ti.pkt[h] = __shfl_sync(0xffffffffu, h_pkt, h);
            ti.mblk[h] = __shfl_sync(0xffffffffu, h_mb, h);
            ti.src[h] = __shfl_sync(0xffffffffu, h_src, h);
            ti.rows[h] = (kind >= 0 && h < nh) ? __shfl_sync(0xffffffffu, h_rows, h) : 0;
            ti.cnt[h] = __shfl_sync(0xffffffffu, h_cnt, h);
        }
        if (lane == 0) {
            if (ti.kind >= 0 && n < 16) trace_stamp(p, 16 + n);
            if (ti.kind >= 0 && (ti.src[0] != p.rank || (PAIR && ti.rows[1] > 0 && ti.src[1] != p.rank)) && !seen_remote) {
                seen_remote = true;
                trace_stamp(p, 13);
            }
            mbar_wait(&sched_empty[q], qphase ^ 1, p.dbg, p.timeout_ns, FM_TRAP_MBAR_SCHED_EMPTY, q);
            ring[q] = ti;
            if (PAIR) {  // mirror the descriptor into the peer CTA's ring over DSMEM, then signal both rings
                const uint4* src4 = reinterpret_cast<const uint4*>(&ti);
                const uint32_t remote = mapa_shared(smem_u32(&ring[q]), 1);
#pragma unroll
                for (int i = 0; i < 4; ++i) st_shared_cluster_v4(remote + 16 * i, src4[i]);
                mbar_arrive_cluster(&sched_full[q], 1);
            }
            mbar_arrive(&sched_full[q]);
        }
        if (++q == NSCHED) { q = 0; qphase ^= 1; }
        ++n;
        if (kind < 0) break;
        __syncwarp();
    }
}

// warp 0 of every CTA: TMA producer.  In pair mode each CTA loads its own A row block and its half of the B rows; all
// completion bytes are credited to the leader's `full` barrier (the only one the MMA issuer waits on).
template <bool PAIR>
__device__ __forceinline__ void ffn_producer(const FmParams& p, uint8_t* smem, uint64_t* bars, uint32_t crank) {
    using PC = PipeCfg<PAIR>;
    uint64_t* full = bars + BAR_FULL;
    uint64_t* empty = bars + BAR_EMPTY;
    uint64_t* sched_full = bars + BAR_SCHED_FULL;
    uint64_t* sched_empty = bars + BAR_SCHED_EMPTY;
    uint64_t* prod_take = bars + BAR_PROD_TAKE;
    const TileInfo* ring = reinterpret_cast<const TileInfo*>(smem + OFF_RING);
    const int lane = threadIdx.x & 31;
    int stage = 0, phase = 0, q = 0, qphase = 0;
    bool first = true, stamped = false;
    for (;;) {
        int kind = -1;
        TileInfo ti;
        if (lane == 0) {
            wait_sched_full<PAIR>(p, &sched_full[q], qphase, 300 + q);
            ti = ring[q];
            release_to_leader<PAIR>(&sched_empty[q], crank);
            kind = ti.kind;
        }
        kind = __shfl_sync(0xffffffffu, kind, 0);
        if (kind < 0) break;
        int nk = 0;
        if (lane == 0) {
            if (first && (p.phase_mask & 1u))   // the stage area doubles as the dispatch staging buffer
                mbar_wait(&bars[BAR_DISP_DONE], 0, p.dbg, p.timeout_ns, FM_TRAP_MBAR_EMPTY, 901);
            first = false;
            fence_proxy_async_global();  // rows written by generic-proxy stores (peers / other SMs) -> TMA reads
            nk = (kind == 0 ? p.H : p.P) / BLOCK_K;
        }
        nk = __shfl_sync(0xffffffffu, nk, 0);
        const CUtensorMap* ta = kind == 0 ? &p.tm_a0 : &p.tm_a1;
        const CUtensorMap* tb = kind == 0 ? &p.tm_b0 : &p.tm_b1;
        constexpr int b_rows = BLOCK_N / PC::B_ROWS_DIV;
        constexpr uint32_t tx = (uint32_t)A_STAGE_BYTES + (uint32_t)(b_rows * BLOCK_K * 2);
        const int take_at = min(nk - 1, max(0, nk - CLAIM_AHEAD_KB));
        int a_row = 0, b_row = 0;
        if (lane == 0) {
            const int hh = PAIR ? (int)crank : 0;
            a_row = ti.pkt[hh] * p.pEC + ti.mblk[hh] * BLOCK_M;
            b_row = ti.b_row + (PAIR ? (int)crank * b_rows : 0);
        }
        for (int kb = 0; kb < nk; ++kb) {
            uint8_t* sa = smem + stage * PC::STAGE_BYTES;
            if (lane == 0) {
                if (kb == take_at && crank == 0) mbar_arrive(&prod_take[q]);  // lets the scheduler claim the next tile
                mbar_wait(&empty[stage], phase ^ 1, p.dbg, p.timeout_ns, FM_TRAP_MBAR_EMPTY, stage);
                if (PAIR) {
                    // the leader's expect_tx covers both CTAs' bytes (every completion is credited to ITS barrier), so
                    // the partner's producer needs no arrival of its own: it only has to wait for its `empty` slot
                    if (crank == 0) mbar_arrive_expect_tx(&full[stage], 2u * tx);
                    const uint32_t leader_full = mapa_shared(smem_u32(&full[stage]), 0);
                    tma_load_2d_pair(sa, ta, kb * BLOCK_K, a_row, leader_full);
                    tma_load_2d_pair(sa + A_STAGE_BYTES, tb, kb * BLOCK_K, b_row, leader_full);
                } else {
                    mbar_arrive_expect_tx(&full[stage], tx);
                    tma_load_2d(sa, ta, kb * BLOCK_K, a_row, &full[stage]);
                    tma_load_2d(sa + A_STAGE_BYTES, tb, kb * BLOCK_K, b_row, &full[stage]);
                }
                if (!stamped) { trace_stamp(p, 7); stamped = true; }   // first loads of the first tile issued
            }
            if (++stage == PC::STAGES) { stage = 0; phase ^= 1; }
        }
        if (++q == NSCHED) { q = 0; qphase ^= 1; }
        __syncwarp();
    }
}

// warp 1 (leader CTA only in pair mode): the single thread that issues tcgen05.mma
template <bool PAIR>
__device__ __forceinline__ void ffn_mma(const FmParams& p, uint8_t* smem, uint64_t* bars, uint32_t tmem_base) {
    using PC = PipeCfg<PAIR>;
    uint64_t* full = bars + BAR_FULL;
    uint64_t* empty = bars + BAR_EMPTY;
    uint64_t* tmem_full = bars + BAR_TMEM_FULL;
    uint64_t* tmem_empty = bars + BAR_TMEM_EMPTY;
    uint64_t* sched_full = bars + BAR_SCHED_FULL;
    uint64_t* sched_empty = bars + BAR_SCHED_EMPTY;
    const TileInfo* ring = reinterpret_cast<const TileInfo*>(smem + OFF_RING);
    const int lane = threadIdx.x & 31;
    int stage = 0, phase = 0, q = 0, qphase = 0, as = 0, aphase = 0, nt = 0;
    for (;;) {
        int kind = -1, nk = 0;
        if (lane == 0) {
            mbar_wait(&sched_full[q], qphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_SCHED_FULL, q);
            kind = ring[q].kind;
            nk = kind < 0 ? 0 : (kind == 0 ? p.H : p.P) / BLOCK_K;
            mbar_arrive(&sched_empty[q]);
        }
        kind = __shfl_sync(0xffffffffu, kind, 0);
        if (++q == NSCHED) { q = 0; qphase ^= 1; }
        if (kind < 0) break;
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_bf16_f32(PAIR ? 2 * BLOCK_M : BLOCK_M, (uint32_t)BLOCK_N);
            mbar_wait(&tmem_empty[as], aphase ^ 1, p.dbg, p.timeout_ns, FM_TRAP_MBAR_TMEM_EMPTY, as);
            tcgen05_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)as * BLOCK_N;
            for (int kb = 0; kb < nk; ++kb) {
                mbar_wait(&full[stage], phase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_FULL, stage);
                if (kb == 0 && nt < 16) trace_stamp(p, 32 + nt);
                tcgen05_fence_after();
                const uint32_t sa = smem_u32(smem + stage * PC::STAGE_BYTES);
                const uint64_t da = umma_smem_desc_sw128(sa);
                const uint64_t db = umma_smem_desc_sw128(sa + A_STAGE_BYTES);
#pragma unroll
                for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
                    // +32 bytes per UMMA_K step inside the 128-byte swizzle row (address field is in 16-byte units)
                    if (PAIR) umma_bf16_ss_pair(d_tmem, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                                                (kb | kk) != 0 ? 1u : 0u);
                    else umma_bf16_ss(d_tmem, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                                      (kb | kk) != 0 ? 1u : 0u);
                }
                // smem slot reusable once these MMAs have read it (pair: signalled to both CTAs' producers)
                if (PAIR) umma_commit_pair(&empty[stage]); else umma_commit(&empty[stage]);
                if (++stage == PC::STAGES) { stage = 0; phase ^= 1; }
            }
            // accumulator complete -> epilogue warps (of both CTAs in pair mode)
            if (PAIR) umma_commit_pair(&tmem_full[as]); else umma_commit(&tmem_full[as]);
            if (nt < 16) trace_stamp(p, 48 + nt);
        }
        if (++as == 2) { as = 0; aphase ^= 1; }
        ++nt;
        __syncwarp();
    }
}

__device__ __noinline__ float gelu_erf(float v) {   // GELU, erf form (cutlass::epilogue::thread::GELU); out of line on purpose
    return 0.5f * v * (1.0f + erff(v * 0.70710678118654752f));
}

enum : int { EPI_G0_RELU = 0, EPI_G0_GELU = 1, EPI_G1_STORE = 2, EPI_G1_FUSED_ADD = 3, EPI_G1_FUSED_COPY = 4 };

struct DrainArgs {
    uint8_t* stg;                  // this warp's 32 x 128 B transpose tile (16-byte pieces XOR-swizzled by row & 7)
    uint32_t t_row;                // TMEM address of this warp's lane quarter, accumulator column 0
    int c0, c1;                    // this warp's 64-column chunks [c0, c1) of the tile
    int lane, quarter, my_rows, N, n0;
    const __nv_bfloat16* bias;     // [N] or nullptr
    __nv_bfloat16* out_rows;       // row 0 of the destination row block (h staging or return buffer)
    __nv_bfloat16* acc_base;       // fused GEMM1: the source rank's output accumulator
    int my_tok;                    // fused GEMM1: token of accumulator row (quarter*32 + lane)
    float my_pw, my_mcw;
    uint64_t* release_bar;         // tmem_empty barrier of this accumulator
    uint32_t crank;
    bool stamp;
};

// TMEM -> registers (thread = accumulator row) -> bias / activation / combine scaling in fp32 -> bf16 (RNE) -> smem
// transpose -> full-line 16-byte global stores (or REDG adds).  64 accumulator columns per step.
template <int MODE, bool HAS_BIAS, bool PAIR>
__device__ __forceinline__ void drain_accumulator(const FmParams& p, const DrainArgs& a) {
    uint8_t* my_row = a.stg + a.lane * EPI_ROW_BYTES;
    const int sw = a.lane & 7;
    for (int c = a.c0; c < a.c1; ++c) {
        uint32_t v[2][32];
        tmem_ld_32x32b_x32(a.t_row + c * 64, v[0]);
        tmem_ld_32x32b_x32(a.t_row + c * 64 + 32, v[1]);
        tmem_ld_wait();
        if (c == a.c1 - 1) {  // last TMEM read of this warp: hand its share of the accumulator back to the MMA issuer
            tcgen05_fence_before();
            __syncwarp();
            if (a.lane == 0) release_to_leader<PAIR>(a.release_bar, a.crank);
        }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {   // 8 columns -> one 16-byte smem store
                float f[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[half][g * 8 + i]);
                if (HAS_BIAS) {
                    float bv[8];
                    unpack8(ld_global_nc_v4(a.bias + a.n0 + c * 64 + half * 32 + g * 8), bv);
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[i] += bv[i];
                }
                if (MODE == EPI_G0_RELU) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[i] = fmaxf(f[i], 0.0f);                 // ReLU (types.cuh:151-159)
                } else if (MODE == EPI_G0_GELU) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[i] = gelu_erf(f[i]);
                } else if (MODE == EPI_G1_FUSED_ADD) {
                    // the reference's combine arithmetic on the bf16-rounded y (processor.cuh:110-169):
                    // term = rne( p~ (x) rne( y / mCw ) ); the bf16 accumulation itself is the REDG below
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[i] = a.my_pw * rne_bf16(__fdividef(rne_bf16(f[i]), a.my_mcw));
                }
                uint4 o;
                o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
                o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
                *reinterpret_cast<uint4*>(my_row + (((half * 4 + g) ^ sw) << 4)) = o;
            }
        }
        __syncwarp();
        // transposed read-back: 8 lanes cover one row's 128 bytes, 4 rows per instruction, full-line stores
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int r = it * 4 + (a.lane >> 3), seg = a.lane & 7;
            const uint4 o = *reinterpret_cast<const uint4*>(a.stg + r * EPI_ROW_BYTES + ((seg ^ (r & 7)) << 4));
            const int row_in_tile = a.quarter * 32 + r;
            if (MODE == EPI_G1_FUSED_ADD || MODE == EPI_G1_FUSED_COPY) {
                // row -> its token's output row on the source rank (k == 1: plain copy, reference processor.cuh:170-203)
                const int tok = __shfl_sync(0xffffffffu, a.my_tok, r);
                if (row_in_tile < a.my_rows) {
                    __nv_bfloat16* dst = a.acc_base + (size_t)tok * a.N + a.n0 + c * 64 + seg * 8;
                    if (MODE == EPI_G1_FUSED_ADD) red_add_bf16x8(dst, o); else st_global_v4(dst, o);
                }
            } else if (row_in_tile < a.my_rows) {
                st_global_v4(a.out_rows + (size_t)row_in_tile * a.N + a.n0 + c * 64 + seg * 8, o);
            }
        }
        __syncwarp();
    }
}

// warps 4-11 of every CTA: TMEM -> registers -> bias/activation -> bf16 -> smem transpose -> coalesced global / peer stores.
// Warp w reads TMEM lanes [32*(w%4), +32) (a hardware restriction) and the column half (w-4)/4 of the tile.  The
// release fence and the counter / flag traffic that make a finished tile visible to its consumers are NOT done here:
// lane 0 of every epilogue warp arrives on pub_full[] and the publisher warp takes over (ffn_publisher).
template <bool PAIR>
__device__ __forceinline__ void ffn_epilogue(const FmParams& p, uint8_t* smem, uint64_t* bars, uint32_t tmem_base,
                                             uint32_t crank) {
    uint64_t* tmem_full = bars + BAR_TMEM_FULL;
    uint64_t* tmem_empty = bars + BAR_TMEM_EMPTY;
    uint64_t* sched_full = bars + BAR_SCHED_FULL;
    uint64_t* sched_empty = bars + BAR_SCHED_EMPTY;
    uint64_t* pub_full = bars + BAR_PUB_FULL;
    uint64_t* pub_empty = bars + BAR_PUB_EMPTY;
    const TileInfo* ring = reinterpret_cast<const TileInfo*>(smem + OFF_RING);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int quarter = warp & 3;  // TMEM lanes [32*quarter, 32*quarter+32) are the only ones this warp may read
    const int chalf = (warp - EPI_WARP0) >> 2;
    uint8_t* stg = smem + OFF_EPI + (warp - EPI_WARP0) * EPI_WARP_BYTES;
    int q = 0, qphase = 0, as = 0, aphase = 0, ps = 0, pphase = 0, ntiles = 0;
    for (;;) {
        wait_sched_full<PAIR>(p, &sched_full[q], qphase, 100 + q);
        const TileInfo ti = ring[q];
        __syncwarp();
        if (lane == 0) release_to_leader<PAIR>(&sched_empty[q], crank);
        if (++q == NSCHED) { q = 0; qphase ^= 1; }
        if (ti.kind < 0) break;
        const int N = ti.kind == 0 ? p.P : p.H;
        const int n0 = ti.ntile * BLOCK_N;
        const int hh = PAIR ? (int)crank : 0;
        const int my_rows = ti.rows[hh], my_mblk = ti.mblk[hh], my_pkt = ti.pkt[hh], my_src = ti.src[hh];
        const __nv_bfloat16* bias = ti.kind == 0 ? (p.b_up ? p.b_up + (size_t)ti.le * p.P : nullptr)
                                                 : (p.b_down ? p.b_down + (size_t)ti.le * p.H : nullptr);
        // destination rows: GEMM0 -> local h staging; GEMM1 -> the SOURCE rank's return buffer (peer store),
        // like the reference's GEMM1 epilogue writing into the peer heap (packet.cuh:338-340, processor.cuh:713-720)
        __nv_bfloat16* out_rows;
        if (ti.kind == 0) {
            out_rows = p.hidden + ((size_t)my_pkt * p.pEC + (size_t)my_mblk * BLOCK_M) * p.P;
        } else {
            const int e_global = p.rank * p.nLx + ti.le;
            out_rows = p.peer_ret_y[my_src] + ((size_t)e_global * p.pEC + (size_t)my_mblk * BLOCK_M) * p.H;
        }
        // 64-column chunks of the tile that exist (N is a multiple of 64, not necessarily of the tile width), split
        // between the two warps of this lane quarter
        constexpr int per_half = BLOCK_N / 128;
        const int nvalid = my_rows > 0 ? min(BLOCK_N / 64, (N - n0) / 64) : 0;
        const int c0 = min(chalf * per_half, nvalid), c1 = min(c0 + per_half, nvalid);
        // fused GEMM1 -> combine: this thread owns accumulator row (quarter*32 + lane); fetch that row's routing record
        const bool fuse = p.fused != 0 && ti.kind == 1;
        int my_tok = 0;
        float my_pw = 0.0f, my_mcw = 1.0f;
        if (fuse && p.dense) {
            my_tok = my_mblk * BLOCK_M + quarter * 32 + lane;   // row i of the only packet IS token i
        } else if (fuse && quarter * 32 + lane < my_rows) {
            const uint4 m = ld_global_v4(p.recv_meta + (size_t)my_pkt * p.pEC + (size_t)my_mblk * BLOCK_M + quarter * 32 + lane);
            my_tok = (int)m.x;
            my_pw = __uint_as_float(m.y);
            my_mcw = __uint_as_float(m.z);
        }
        __nv_bfloat16* acc_base = fuse ? p.peer_out_acc[my_src] : nullptr;

        mbar_wait(&tmem_full[as], aphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_TMEM_FULL, as);
        tcgen05_fence_after();
        if (ntiles == 0 && p.W > 1 && (p.phase_mask & 1u))   // the staging area served as warp 2's window for the remote rows
            asm volatile("bar.sync 7, 288;" ::: "memory");
        const bool stamp_tile = ntiles < 16 && tid == EPI_WARP0 * 32;
        if (stamp_tile) trace_stamp(p, 64 + ntiles);
        const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)as * BLOCK_N;
        if (c1 > c0) {
            DrainArgs da;
            da.stg = stg; da.t_row = t_row; da.c0 = c0; da.c1 = c1; da.lane = lane; da.quarter = quarter;
            da.my_rows = my_rows; da.N = N; da.n0 = n0; da.bias = bias; da.out_rows = out_rows; da.acc_base = acc_base;
            da.my_tok = my_tok; da.my_pw = my_pw; da.my_mcw = my_mcw; da.release_bar = &tmem_empty[as]; da.crank = crank;
            da.stamp = false;
            // one specialised instantiation per (epilogue kind, bias) pair: no per-element or per-group branching
            const int mode = ti.kind == 0 ? (p.act == 0 ? EPI_G0_RELU : EPI_G0_GELU)
                                          : (!fuse ? EPI_G1_STORE : (p.k > 1 ? EPI_G1_FUSED_ADD : EPI_G1_FUSED_COPY));
            if (bias == nullptr) {
                switch (mode) {
                    case EPI_G0_RELU: drain_accumulator<EPI_G0_RELU, false, PAIR>(p, da); break;
                    case EPI_G0_GELU: drain_accumulator<EPI_G0_GELU, false, PAIR>(p, da); break;
                    case EPI_G1_STORE: drain_accumulator<EPI_G1_STORE, false, PAIR>(p, da); break;
                    case EPI_G1_FUSED_ADD: drain_accumulator<EPI_G1_FUSED_ADD, false, PAIR>(p, da); break;
                    default: drain_accumulator<EPI_G1_FUSED_COPY, false, PAIR>(p, da); break;
                }
            } else {
                switch (mode) {
                    case EPI_G0_RELU: drain_accumulator<EPI_G0_RELU, true, PAIR>(p, da); break;
                    case EPI_G0_GELU: drain_accumulator<EPI_G0_GELU, true, PAIR>(p, da); break;
                    case EPI_G1_STORE: drain_accumulator<EPI_G1_STORE, true, PAIR>(p, da); break;
                    case EPI_G1_FUSED_ADD: drain_accumulator<EPI_G1_FUSED_ADD, true, PAIR>(p, da); break;
                    default: drain_accumulator<EPI_G1_FUSED_COPY, true, PAIR>(p, da); break;
                }
            }
        } else {  // nothing to drain for this warp (row block or columns past the end): still release the accumulator
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) release_to_leader<PAIR>(&tmem_empty[as], crank);
        }
        if (stamp_tile) trace_stamp(p, 80 + ntiles);
        if (++as == 2) { as = 0; aphase ^= 1; }

        // hand the tile to the publisher: this warp's stores are issued (h will be read through the async proxy)
        if (ti.kind == 0) fence_proxy_async_global();
        __syncwarp();
        if (lane == 0) {
            mbar_wait(&pub_empty[ps], pphase ^ 1, p.dbg, p.timeout_ns, FM_TRAP_MBAR_PUB, ps);
            mbar_arrive(&pub_full[ps]);
        }
        if (++ps == 2) { ps = 0; pphase ^= 1; }
        ++ntiles;
    }
}

// warp 2 of every CTA: makes finished tiles visible.  For every tile of the ring, once all epilogue warps of this CTA
// have issued their stores: GEMM0 -> release-add on the row block's h counter (reference notifyNext's tSA counter,
// processor.cuh:490-615); GEMM1 -> system-scope fence, then the packet / row-block counter and, from the last tile, the
// flag on the source rank (reference processor.cuh:722-750).  The fences wait for the stores / REDs to drain (1-2 us,
// more over NVLink); here they overlap the next tile's epilogue instead of delaying it.
template <bool PAIR>
__device__ __forceinline__ void ffn_publisher(const FmParams& p, uint8_t* smem, uint64_t* bars, uint32_t crank) {
    uint64_t* sched_full = bars + BAR_SCHED_FULL;
    uint64_t* sched_empty = bars + BAR_SCHED_EMPTY;
    uint64_t* pub_full = bars + BAR_PUB_FULL;
    uint64_t* pub_empty = bars + BAR_PUB_EMPTY;
    const TileInfo* ring = reinterpret_cast<const TileInfo*>(smem + OFF_RING);
    const int lane = threadIdx.x & 31;
    int q = 0, qphase = 0, ps = 0, pphase = 0, ntiles = 0;
    for (;;) {
        int kind = -1;
        if (lane == 0) {
            wait_sched_full<PAIR>(p, &sched_full[q], qphase, 400 + q);
            const TileInfo ti = ring[q];
            release_to_leader<PAIR>(&sched_empty[q], crank);
            kind = ti.kind;
            if (kind >= 0) {
                const int hh = PAIR ? (int)crank : 0;
                const int my_rows = ti.rows[hh], my_mblk = ti.mblk[hh], my_pkt = ti.pkt[hh], my_src = ti.src[hh];
                mbar_wait(&pub_full[ps], pphase, p.dbg, p.timeout_ns, FM_TRAP_MBAR_PUB, 10 + ps);
                mbar_arrive(&pub_empty[ps]);
                if (my_rows > 0) {
                    if (kind == 0) {
                        fence_proxy_async_global();
                        red_release_gpu_add_u32(p.g0_done + (size_t)my_pkt * p.TCM + my_mblk, 1u);
                    } else if (p.fused) {
                        if (my_src == p.rank && p.out_acc == p.out) {
                            // local packet, output left in place: nobody waits for a flag (see finish_fused) -- no fence,
                            // no counter, no flag; kernel completion covers these adds
                        } else {
                        fence_acq_rel_sys();   // this tile's adds are performed before the packet counter moves
                        const unsigned int old = atom_acq_rel_gpu_add_u32(p.pkt_done + my_pkt, 1u);
                        const unsigned int want = (unsigned int)(((ti.cnt[hh] + BLOCK_M - 1) / BLOCK_M) * p.TN1);
                        if (old + 1u == want) {   // every GEMM1 tile of packet (src, le) has been added into src's output
                            st_release_sys_u64(p.peer_done_flag[my_src] + (size_t)(p.rank * p.nLx + ti.le),
                                               (unsigned long long)p.epoch << 32);
                        }
                        }
                    } else {
                        fence_acq_rel_sys();
                        const unsigned int old = atom_acq_rel_gpu_add_u32(p.g1_done + (size_t)my_pkt * p.TCM + my_mblk, 1u);
                        if (old == (unsigned int)p.TN1 - 1u) {  // whole rows of this block are on the source rank
                            fence_acq_rel_sys();
                            const int e_global = p.rank * p.nLx + ti.le;
                            st_release_sys_u64(p.peer_ret_flag[my_src] + (size_t)e_global * p.TCM + my_mblk,
                                               ((unsigned long long)p.epoch << 32) | (unsigned int)my_rows);
                        }
                    }
                }
                if (ntiles < 16) trace_stamp(p, 96 + ntiles);
            }
        }
        kind = __shfl_sync(0xffffffffu, kind, 0);
        if (++q == NSCHED) { q = 0; qphase ^= 1; }
        if (++ps == 2) { ps = 0; pphase ^= 1; }
        ++ntiles;
        if (kind < 0) break;
        __syncwarp();
    }
}

// kernel prologue: barriers of every later phase + TMEM; runs before the router so it costs nothing on the critical path
template <bool PAIR>
__device__ __forceinline__ void ffn_setup(const FmParams& p, uint8_t* smem) {
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BARS);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + OFF_TMEM_PTR);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 1 && (tid & 31) == 0) {
        // arrival counts: full = leader's expect_tx; empty / tmem_full = one tcgen05.commit; tmem_empty = one lane per
        // epilogue warp (of both CTAs); pub_full = one lane per epilogue warp of this CTA; sched_empty = every ring reader
        const int nc = PAIR ? 2 : 1;
        for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&bars[BAR_FULL + i], 1); mbar_init(&bars[BAR_EMPTY + i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars[BAR_TMEM_FULL + i], 1);
            mbar_init(&bars[BAR_TMEM_EMPTY + i], NUM_EPI_WARPS * nc);
            mbar_init(&bars[BAR_PUB_FULL + i], NUM_EPI_WARPS);
            mbar_init(&bars[BAR_PUB_EMPTY + i], 1);
        }
        for (int i = 0; i < NSCHED; ++i) {
            mbar_init(&bars[BAR_SCHED_FULL + i], 1);
            mbar_init(&bars[BAR_SCHED_EMPTY + i], 1 + (2 + NUM_EPI_WARPS) * nc);   // MMA lane + per CTA: producer, publisher, epilogue warps
            mbar_init(&bars[BAR_PROD_TAKE + i], 1);
        }
        mbar_init(&bars[BAR_XROWS], 1);
        mbar_init(&bars[BAR_DISP_DONE], 1);
        mbar_init(&bars[BAR_WG], 1);
        mbar_init(&bars[BAR_REMOTE], 1);
        for (int i = 0; i < GATE_STAGES; ++i) { mbar_init(&bars[BAR_GFULL + i], 1); mbar_init(&bars[BAR_GEMPTY + i], 1); }
        mbar_init(&bars[BAR_GACC], 1);
        fence_mbar_init();
    }
    if (warp == 0 && (tid & 31) == 0) {
        tma_prefetch_desc(&p.tm_a0); tma_prefetch_desc(&p.tm_b0);
        tma_prefetch_desc(&p.tm_a1); tma_prefetch_desc(&p.tm_b1);
    }
    if (warp == 3 && (tid & 31) == 0 && (p.phase_mask & 3u) == 3u && (!PAIR || (blockIdx.x & 1) == 0)) {
        // Warm L2 with the weight tile this pair will most likely claim first (item id = pair index: the first wave is
        // claimed in arrival order), pipeline depth only: HBM is idle during the router and the first tile's loads are
        // then L2 hits.  A wrong guess costs nothing -- the tile is needed by some pair of the first wave anyway.
        const int id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
        if (id < p.total_items) {
            int cur = 0;
            while (id >= p.blocks[cur + 1].start) ++cur;
            const TileBlock blk = p.blocks[cur];
            const int local = id - blk.start;
            const bool cross = PAIR && blk.pkt2 >= 0;
            const int m_items = (PAIR && !cross) ? (p.TCM + 1) / 2 : p.TCM;
            const int nt = local / m_items, le = blk.pkt % p.nLx;
            const CUtensorMap* tb = blk.kind == 0 ? &p.tm_b0 : &p.tm_b1;
            const int b0 = (blk.kind == 0 ? le * 2 * p.P : (le * 2 + 1) * p.H) + nt * BLOCK_N;
            const int nk_w = (blk.kind == 0 ? p.H : p.P) / BLOCK_K;
            constexpr int step = BLOCK_N / PipeCfg<PAIR>::B_ROWS_DIV;
            for (int kb = 0; kb < min(nk_w, PipeCfg<PAIR>::STAGES); ++kb)
                for (int r = 0; r < BLOCK_N; r += step) tma_prefetch_l2_2d(tb, kb * BLOCK_K, b0 + r);
        }
    }
    if (warp == 2 && ((p.phase_mask & 2u) || p.tc_gate)) { if (PAIR) tmem_alloc_pair(tmem_ptr, TMEM_COLS); else tmem_alloc(tmem_ptr, TMEM_COLS); }
    tcgen05_fence_before();
}

// warp roles of the expert-FFN phase (entered per warp as soon as that warp is free; no block-wide sync on entry)
template <bool PAIR>
__device__ __forceinline__ void ffn_roles(const FmParams& p, uint8_t* smem, uint32_t crank) {
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BARS);
    const int tid = threadIdx.x, warp = tid >> 5;
    tcgen05_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM_PTR);
    if (warp == 0) ffn_producer<PAIR>(p, smem, bars, crank);
    else if (warp == 1) { if (crank == 0) ffn_mma<PAIR>(p, smem, bars, tmem_base); }
    else if (warp == 2) ffn_publisher<PAIR>(p, smem, bars, crank);
    else if (warp == 3) { if (crank == 0) ffn_scheduler<PAIR>(p, smem, bars); }
    else if (warp >= EPI_WARP0) ffn_epilogue<PAIR>(p, smem, bars, tmem_base, crank);
}

template <bool PAIR>
__device__ __forceinline__ void ffn_teardown(const FmParams& p, uint8_t* smem) {
    const int tid = threadIdx.x, warp = tid >> 5;
    tcgen05_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();   // nobody leaves while the partner may still touch its smem/TMEM
    if (warp == 2) {
        tcgen05_fence_after();
        const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM_PTR);
        if (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS); else tmem_dealloc(tmem_base, TMEM_COLS);
    }
    if (tid == 0) trace_stamp(p, 5);
}

// ============================================================================================================
// Phase C: combine (gather path: k > 2 or FM_FUSED_COMBINE=0; the default for k <= 2 is the fused GEMM1 epilogue +
// finish_fused below).  For token t with picks (e_j, slot_j):
//   k > 1: out[t,c] = bf16-accumulate over kept j of rne( p~_j * rne( y_j[c] / mCw ) )   (processor.cuh:110-169)
//   k = 1: out[t,:] = y_0 (no scaling), zeros if dropped                                  (processor.cuh:170-203)
// Deterministic gather (no atomics, no zero-fill pass); for k == 2 it equals the reference's atomicAdd result
// exactly because bf16 addition commutes and 0 + a is exact.
// ============================================================================================================
template <int KMAX, int PIECES>
__device__ __forceinline__ void combine_rows(const FmParams& p, int t0, int n_tok, const int* c_e, const int* c_s,
                                             const float* c_w, const float* c_m) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int H = p.H, k = p.k;
    for (int ti = warp; ti < n_tok; ti += NUM_WARPS) {
        const __nv_bfloat16* yrow[KMAX];
        float pw[KMAX];
        bool keep[KMAX];
        const float mcw = c_m[ti];
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
            keep[j] = false;
            yrow[j] = nullptr;
            pw[j] = 0.0f;
            if (j < k) {
                const int s = c_s[ti * k + j];
                pw[j] = c_w[ti * k + j];
                keep[j] = s < p.EC;
                yrow[j] = p.ret_y + ((size_t)c_e[ti * k + j] * p.pEC + (keep[j] ? s : 0)) * H;
            }
        }
        __nv_bfloat16* orow = p.out + (size_t)(t0 + ti) * H;
        for (int hg = 0; hg < H; hg += PIECES * 256) {
            uint4 yv[KMAX][PIECES];   // every load of this column group is issued before the arithmetic
#pragma unroll
            for (int j = 0; j < KMAX; ++j)
#pragma unroll
                for (int i = 0; i < PIECES; ++i) {
                    const int h = hg + i * 256 + lane * 8;
                    if (j < k && keep[j] && h < H) yv[j][i] = ld_global_v4(yrow[j] + h);
                }
#pragma unroll
            for (int i = 0; i < PIECES; ++i) {
                const int h = hg + i * 256 + lane * 8;
                if (h >= H) continue;
                float acc[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) acc[q] = 0.0f;
#pragma unroll
                for (int j = 0; j < KMAX; ++j) {
                    if (j < k && keep[j]) {
                        float y[8];
                        unpack8(yv[j][i], y);
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float qv = rne_bf16(__fdividef(y[q], mcw));
                            const float term = rne_bf16(pw[j] * qv);
                            acc[q] = rne_bf16(acc[q] + term);
                        }
                    }
                }
                uint4 o;
                o.x = pack_bf16x2(acc[0], acc[1]); o.y = pack_bf16x2(acc[2], acc[3]);
                o.z = pack_bf16x2(acc[4], acc[5]); o.w = pack_bf16x2(acc[6], acc[7]);
                st_global_v4(orow + h, o);
            }
        }
    }
}

// fused path: the output rows were accumulated by the GEMM1 epilogues; wait until every expert (local or remote) has
// reported all of its contributions, then (W > 1) move my rows from the symmetric accumulator to the caller's tensor
__device__ __forceinline__ void finish_fused(const FmParams& p, int t0, int n_tok) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // Contributions of experts on THIS GPU need no flag when the rows are left where they were accumulated (out == the
    // accumulation target): they are complete when the kernel is, and nobody reads them before.  Only the experts on other
    // ranks -- whose adds arrive over NVLink at their own pace -- must have reported; with a separate caller tensor (the
    // copy below) the local ones must have, too.
    const bool need_local = p.out_acc != p.out;
    for (int e = tid; e < p.E; e += NUM_THREADS) {
        if (!need_local && e / p.nLx == p.rank) continue;
        SpinGuard g;
        while ((ld_acquire_sys_u64(p.done_flag + e) >> 32) != p.epoch)
            g.tick(p.dbg, p.timeout_ns, FM_TRAP_RET_FLAG, e, 0xD0E, 0);
    }
    __syncthreads();
    if (tid == 0) trace_stamp(p, 14);   // every expert's contributions to this rank's tokens are in
    if (p.out_acc != p.out) {
        for (int ti = warp; ti < n_tok; ti += NUM_WARPS) {
            const __nv_bfloat16* src = p.out_acc + (size_t)(t0 + ti) * p.H;
            __nv_bfloat16* dst = p.out + (size_t)(t0 + ti) * p.H;
            for (int hg = 0; hg < p.H; hg += 1024) {
                uint4 v[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int h = hg + i * 256 + lane * 8;
                    if (h < p.H) v[i] = ld_global_v4(src + h);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int h = hg + i * 256 + lane * 8;
                    if (h < p.H) st_global_v4(dst + h, v[i]);
                }
            }
        }
    }
}

__device__ __forceinline__ void combine_phase(const FmParams& p, uint8_t* smem, int t0, int n_tok) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int H = p.H, k = p.k;
    // the pipeline stage area is free again: stage this chunk's routing records, and let one thread per (token, pick)
    // poll its return flag so the waits overlap instead of chaining per token
    int* c_e = reinterpret_cast<int*>(smem);
    int* c_s = c_e + G_SEL_MAX;
    float* c_w = reinterpret_cast<float*>(c_s + G_SEL_MAX);
    float* c_m = c_w + G_SEL_MAX;
    const int n = n_tok * k;
    for (int i = tid; i < n; i += NUM_THREADS) {
        const size_t gi = (size_t)t0 * k + i;
        const int e = p.topk_idx[gi];
        const int s = p.slot[gi];
        c_e[i] = e;
        c_s[i] = s;
        c_w[i] = __bfloat162float(p.topk_w[gi]);
        if (s < p.EC) {
            const unsigned long long* fl = p.ret_flag + (size_t)e * p.TCM + (s / BLOCK_M);
            SpinGuard g;
            while ((ld_acquire_sys_u64(fl) >> 32) != p.epoch)
                g.tick(p.dbg, p.timeout_ns, FM_TRAP_RET_FLAG, e, s, t0 + i / k);
        }
    }
    for (int i = tid; i < n_tok; i += NUM_THREADS) c_m[i] = p.mcw[t0 + i];
    __syncthreads();
    if (k == 1) {
        for (int ti = warp; ti < n_tok; ti += NUM_WARPS) {
            const bool keep = c_s[ti] < p.EC;
            const __nv_bfloat16* yrow = p.ret_y + ((size_t)c_e[ti] * p.pEC + (keep ? c_s[ti] : 0)) * H;
            __nv_bfloat16* orow = p.out + (size_t)(t0 + ti) * H;
            for (int h = lane * 8; h < H; h += 256) {
                uint4 v = make_uint4(0u, 0u, 0u, 0u);
                if (keep) v = ld_global_v4(yrow + h);
                st_global_v4(orow + h, v);
            }
        }
    } else if (k == 2) {
        combine_rows<2, 4>(p, t0, n_tok, c_e, c_s, c_w, c_m);
    } else {
        combine_rows<8, 1>(p, t0, n_tok, c_e, c_s, c_w, c_m);
    }
}

// ============================================================================================================
template <bool PAIR>
__global__ void __launch_bounds__(NUM_THREADS, 1) fm_moe_forward_kernel(const __grid_constant__ FmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int t0 = blockIdx.x * p.tpc;
    const int n_tok = max(0, min(p.tpc, p.S - t0));
    const uint32_t crank = PAIR ? cluster_ctarank() : 0u;

    if (tid == 0) trace_stamp(p, 0);
    ffn_setup<PAIR>(p, smem);   // mbarriers + TMEM for the later phases (visible to everyone after the next block sync)
    if (p.phase_mask & 1u) {
        // per-launch reset of the work counters (reference clearState, moe.cuh:21-70); consumed only after the grid barrier
        if (blockIdx.x == 0) {
            for (int i = tid; i < p.num_pkts * p.TCM; i += NUM_THREADS) {
                p.g0_done[i] = 0u;
                p.g1_done[i] = 0u;
            }
            for (int i = tid; i < p.num_pkts; i += NUM_THREADS) p.pkt_done[i] = 0u;
            // the arrival counters of the NEXT epoch's parity: nobody reads them any more (launch epoch-1 is over) and no
            // peer can write them yet (a rank starts forward epoch+1 only after this launch has returned all its rows)
            unsigned int* next_rows = p.recv_rows + (size_t)((p.epoch + 1u) & 1u) * p.num_pkts * p.TCM;
            for (int i = tid; i < p.num_pkts * p.TCM; i += NUM_THREADS) next_rows[i] = 0u;
            if (p.aux != nullptr) {   // the loss buffers of the next launch (reference clearState, moe.cuh:49-54)
                float* next_aux = p.aux + (size_t)((p.epoch + 1u) & 1u) * (2 * p.E + 1);
                for (int i = tid; i < 2 * p.E + 1; i += NUM_THREADS) next_aux[i] = 0.0f;
            }
            if (tid == 0) *p.claim = 0u;
        }
        if (p.dense) gate_phase_dense(p, t0, n_tok); else gate_phase<PAIR>(p, smem, t0, n_tok, crank);
        if (tid == 0) trace_stamp(p, 1);
        grid_barrier(p);   // also a cluster-wide sync: the partner CTA's barriers are initialised before any remote arrive
        if (tid == 0) trace_stamp(p, 2);
    } else {
        if (blockIdx.x == 0 && tid == 0) *p.claim = 0u;   // debug re-run of later phases on the previous routing
        if (PAIR) cluster_sync_all(); else __syncthreads();
    }

    // From here the warps specialise.  Warps 0, 1, 3 (TMA producer, MMA issuer, tile scheduler) enter their FFN roles at
    // once -- the scheduler claims its first tile and spins on the packet flag while warps 2, 4-7 dispatch this CTA's rows;
    // warps 4-7 then become the epilogue.
    const bool disp_warp = (warp == 2) || (warp >= EPI_WARP0);
    if ((p.phase_mask & 1u) && disp_warp) {
        if (!p.dense) dispatch_phase(p, smem, t0, n_tok);
        else if (warp == 2 && (tid & 31) == 0)   // nothing to copy: GEMM0's TMA reads x in place; release the producer
            mbar_arrive(reinterpret_cast<uint64_t*>(smem + OFF_BARS) + BAR_DISP_DONE);
        if (warp == 2 && (tid & 31) == 0) trace_stamp(p, 3);
    }
    if (p.phase_mask & 2u) {
        if (tid == EPI_WARP0 * 32) trace_stamp(p, 4);
        ffn_roles<PAIR>(p, smem, crank);
        ffn_teardown<PAIR>(p, smem);
    } else if (p.tc_gate && (p.phase_mask & 1u)) {
        ffn_teardown<PAIR>(p, smem);   // (router-only debug launch: the tensor-core router allocated TMEM)
    }

    if (p.phase_mask & 4u) {
        __syncthreads();
        if (p.fused) finish_fused(p, t0, n_tok);
        else combine_phase(p, smem, t0, n_tok);
        __syncthreads();
        if (tid == 0) trace_stamp(p, 6);
    }
}

}  // namespace fm
