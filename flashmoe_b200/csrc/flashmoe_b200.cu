// flashmoe_b200.cu -- host runtime + C-ABI (include/flashmoe_b200.h) around the fused sm_100a kernel.
//
// Replaces the used slice of the reference's host runtime: bootstrap.cuh:278-512 (symmetric heap + bookkeeping
// allocation, peer pointer tables), moe.cuh:146-205 (launch) and python_bindings.cu:17-151 (argument checks) --
// without NVSHMEM (peer mapping is CUDA IPC or caller-provided pointers), without per-call weight copies
// (python_bindings.cu:76-120 re-uploads every weight on every call) and without exit() on errors.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "fm_kernel.cuh"

// ---- compile-time configuration surface: csrc/flashmoe_config.json -> -DFM_CFG_* (build script) -------------
#ifndef FM_CFG_CAPACITY_FACTOR
#define FM_CFG_CAPACITY_FACTOR 1
#define FM_CFG_DROP_TOKENS 1
#define FM_CFG_EXPERT_TOP_K 2
#define FM_CFG_GLOBAL_BATCH 256
#define FM_CFG_IS_TRAINING 0
#define FM_CFG_HIDDEN_ACT 0
#define FM_CFG_HIDDEN_SIZE 1024
#define FM_CFG_INTERMEDIATE_SIZE 4096
#define FM_CFG_MINI_BATCH 1
#define FM_CFG_MOE_FREQUENCY 1
#define FM_CFG_NUM_EXPERTS 8
#define FM_CFG_NUM_LAYERS 1
#define FM_CFG_SEQUENCE_LEN 4096
#define FM_CFG_TORCH_DTYPE 2
#define FM_CFG_VOCAB_SIZE 32000
#endif

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define FM_CUDA(expr)                                                                                         \
    do {                                                                                                      \
        cudaError_t _e = (expr);                                                                              \
        if (_e != cudaSuccess)                                                                                \
            return fail(FM_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// 2-D row-major bf16 tensor [rows, cols], tile box [box_rows, 64 cols], 128-byte swizzle (matches the UMMA smem
// descriptors built in fm_ptx.cuh), out-of-bounds elements read as zero.
int make_tmap(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (fn == nullptr) return fail(FM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {cols * 2};
    const cuuint32_t box[2] = {(cuuint32_t)fm::BLOCK_K, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(FM_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d (base=%p rows=%llu cols=%llu)", (int)r,
                    base, (unsigned long long)rows, (unsigned long long)cols);
    return FM_OK;
}

}  // namespace

struct fm_ctx {
    fm_config_t cfg;
    fm_dims_t d;
    int device = 0;
    int grid = 0;
    int tpc = 0;
    int TN0 = 0, TN1 = 0, num_pkts = 0, num_blocks = 0, total_items = 0;
    bool coop = true;    // cooperative launch attribute (validates co-residency of the persistent grid)
    bool pair = false;   // cta_group::2: two CTAs (one cluster) per 256-row tile
    uint32_t epoch = 0;
    unsigned long long bar_count = 0;
    // in-kernel waits give up after this long (fm_set_timeout_ms): generous by default so that ordinary rank skew (a peer
    // still loading data, compiling, paused in a debugger) is not turned into a trap -- see fm_ptx.cuh SpinGuard
    unsigned long long timeout_ns = 120ull * 1000ull * 1000ull * 1000ull;
    uint64_t launches = 0;
    // device buffers
    int* topk_idx = nullptr;
    __nv_bfloat16* topk_w = nullptr;
    float* mcw = nullptr;
    int* slot = nullptr;
    int* counts = nullptr;
    __nv_bfloat16* gate_out = nullptr;
    int* chunk_counts = nullptr;
    unsigned int* ctrl = nullptr;  // [0] unused, [1] claim, [2..3] grid barrier (u64)
    unsigned int* g0_done = nullptr;
    unsigned int* g1_done = nullptr;
    int* recv_cnt = nullptr;
    fm::TileBlock* blocks = nullptr;
    __nv_bfloat16* hidden = nullptr;
    // host-buffer path (fm_host_submit / fm_host_wait): FM_HOST_SLOTS staging pairs, three streams, so the H2D copy of
    // step i+1 and the D2H copy of step i-1 run under the kernel of step i (PCIe is full duplex; steps are independent)
    __nv_bfloat16* x_stage[FM_HOST_SLOTS] = {};
    __nv_bfloat16* out_stage[FM_HOST_SLOTS] = {};
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[FM_HOST_SLOTS] = {}, ev_kernel[FM_HOST_SLOTS] = {}, ev_d2h[FM_HOST_SLOTS] = {};
    bool host_ready = false;
    uint64_t host_submitted = 0, host_waited = 0;
    // symmetric slab
    void* symm = nullptr;
    bool symm_external = false;
    size_t symm_bytes = 0, off_recv_x = 0, off_ret_y = 0, off_recv_flag = 0, off_ret_flag = 0;
    size_t off_recv_meta = 0, off_out_acc = 0, off_done_flag = 0, off_recv_rows = 0;
    bool fused = false;   // GEMM1 epilogue adds straight into the source rank's output (no return buffer / gather)
    bool dense = false;   // E == 1: GEMM0 reads x in place, no router GEMV, no dispatch copy (reference fffn.cuh:31-167)
    float* aux = nullptr; // is_training: [2][2E+1] {gML, gMeC, loss} by epoch parity
    const void* cached_x = nullptr;
    bool tc_gate = false;               // router logits on the tensor cores (E <= 256)
    const void* cached_gx = nullptr;
    const void* cached_gw = nullptr;
    CUtensorMap tm_gx, tm_gw;
    unsigned int* pkt_done = nullptr;
    void* peer_base[FM_MAX_WORLD] = {};
    bool peer_opened[FM_MAX_WORLD] = {};
    bool attached = false;
    fm::DebugRecord* dbg_host = nullptr;
    fm::DebugRecord* dbg_dev = nullptr;
    unsigned long long* trace = nullptr;
    bool trace_on = false;
    // tensor-map cache (re-encoded only when the caller's weight pointer changes)
    const void* cached_expert_w = nullptr;
    CUtensorMap tm_a0, tm_b0, tm_a1, tm_b1;
    bool tm_static_ready = false;
};

namespace {

int validate_config(const fm_config_t& c, int world, fm_dims_t* d) {
    if (c.torch_dtype != 2) return fail(FM_EINVAL, "torch_dtype=%d: this build computes in bf16 only (2)", c.torch_dtype);
    if (c.is_training != 0 && c.is_training != 1) return fail(FM_EINVAL, "is_training must be 0 or 1");
    if (c.hidden_act != 0 && c.hidden_act != 1) return fail(FM_EINVAL, "hidden_act must be 0 (relu) or 1 (gelu)");
    if (c.drop_tokens != 0 && c.drop_tokens != 1) return fail(FM_EINVAL, "drop_tokens must be 0 or 1");
    if (c.capacity_factor < 1) return fail(FM_EINVAL, "capacity_factor must be >= 1");
    if (c.hidden_size <= 0 || c.hidden_size % 64) return fail(FM_EINVAL, "hidden_size must be a positive multiple of 64");
    if (c.intermediate_size <= 0 || c.intermediate_size % 64)
        return fail(FM_EINVAL, "intermediate_size must be a positive multiple of 64");
    if (c.hidden_size > 32768) return fail(FM_EINVAL, "hidden_size > 32768 is not supported (row staging)");
    if (c.mini_batch < 1 || c.sequence_len < 1) return fail(FM_EINVAL, "mini_batch and sequence_len must be >= 1");
    const long long S = (long long)c.sequence_len * c.mini_batch;
    if (S % 128) return fail(FM_EINVAL, "S = sequence_len*mini_batch = %lld must be a multiple of 128", S);
    if (S > (1ll << 24)) return fail(FM_EINVAL, "S = %lld too large", S);
    if (c.num_experts < 1 || c.num_experts > 1024) return fail(FM_EINVAL, "num_experts must be in [1, 1024]");
    if (c.expert_top_k < 1 || c.expert_top_k > c.num_experts || c.expert_top_k > 8)
        return fail(FM_EINVAL, "expert_top_k must be in [1, min(num_experts, 8)]");
    if (world < 1 || world > FM_MAX_WORLD) return fail(FM_EINVAL, "world size %d not in [1, %d]", world, FM_MAX_WORLD);
    if (c.num_experts % world) return fail(FM_EINVAL, "num_experts=%d not divisible by world=%d", c.num_experts, world);
    d->S = (int)S;
    d->H = c.hidden_size;
    d->E = c.num_experts;
    d->P = c.intermediate_size;
    d->PX = ceil_div(c.num_experts, 64) * 64;
    d->element_size = 2;
    d->k = c.expert_top_k;
    const long long ec = (long long)(c.drop_tokens ? ceil_div((int)S, c.num_experts) : (int)S) * c.capacity_factor *
                         c.expert_top_k;
    if (ec > (1ll << 24)) return fail(FM_EINVAL, "expert capacity %lld too large", ec);
    d->EC = (int)ec;
    d->pEC = ceil_div(d->EC, 128) * 128;
    d->TCM = d->pEC / 128;
    d->world = world;
    d->num_local_experts = c.num_experts / world;
    return FM_OK;
}

template <typename T>
int dev_alloc(T** p, size_t count, bool zero = true) {
    void* q = nullptr;
    const size_t bytes = count * sizeof(T);
    cudaError_t e = cudaMalloc(&q, bytes ? bytes : 16);
    if (e != cudaSuccess) return fail(FM_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    if (zero) {
        e = cudaMemset(q, 0, bytes ? bytes : 16);
        if (e != cudaSuccess) return fail(FM_ECUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    }
    *p = static_cast<T*>(q);
    return FM_OK;
}

// The FFN work list: runs of work items (all tiles of one GEMM of one packet, or of a packet pair), claimed in this
// order by the CTAs' schedulers, followed by a sentinel {kind -1, start = total items}.
// Sources in the order own rank, rank+1, ... (local rows need no NVLink hop, so they are ready first).
// With CTA pairs a work item is a 256-row tile made of two 128-row halves that share the B operand (same local expert):
//   * world even and an odd number of row blocks per packet: halves = the SAME row block of the packets of two
//     different source ranks ("cross-source pairing": no half is wasted -- with 128 experts on 8 GPUs every packet has
//     exactly one);
//   * otherwise:  halves = two consecutive row blocks of one packet (with an even number of row blocks this wastes
//     nothing and keeps the local packets -- whose rows are ready first -- free of any remote dependency).
// Orders:
//   one rank:    all GEMM0, then all GEMM1 (measured best on config B);
//   2-3 ranks:   GEMM0 local, GEMM0 remote, GEMM1 remote, GEMM1 local (the remote rows land while the local packets
//                run; the outputs of remote packets cross NVLink as reductions and their done flags have a link round
//                trip ahead of them, while the local adds, which nobody else waits for, come last);
//   4+ ranks:    GEMM0 local, GEMM1 local, then the remote units with GEMM1 one source behind GEMM0 -- the local
//                packets are the only work available until the remote rows have crossed NVLink (~50 us at 8 GPUs),
//                and starting the remote units' GEMM1 early spreads the return traffic (reductions over NVLink at
//                ~350 GB/s per GPU, which would otherwise pile up behind the last tiles) over the whole phase.
std::vector<fm::TileBlock> build_work_list(int world, int rank, int nLx, int TCM, int TN0, int TN1, bool pair) {
    const bool xpair = pair && world >= 2 && (world % 2) == 0 && (TCM % 2) == 1;
    struct Unit { int pkt, pkt2; };
    std::vector<Unit> loc, rem;   // units of this rank's own packets / of the other ranks' packets, in source order
    for (int j = 0; j < world; j += xpair ? 2 : 1)
        for (int le = 0; le < nLx; ++le) {
            const Unit u = {((rank + j) % world) * nLx + le, xpair ? ((rank + j + 1) % world) * nLx + le : -1};
            (j == 0 ? loc : rem).push_back(u);
        }
    std::vector<fm::TileBlock> blocks;
    int start = 0;
    auto push = [&](int kind, const Unit& u) {
        blocks.push_back({kind, u.pkt, start, u.pkt2});
        const int row_items = (pair && u.pkt2 < 0) ? (TCM + 1) / 2 : TCM;
        start += row_items * (kind == 0 ? TN0 : TN1);
    };
    if (world >= 4) {
        for (const Unit& u : loc) push(0, u);
        for (const Unit& u : loc) push(1, u);
        // remote units grouped by source rank (nLx units per source, or per source pair): GEMM1 one source behind GEMM0
        const size_t per_src = (size_t)nLx;
        for (size_t g0 = 0; g0 < rem.size(); g0 += per_src) {
            for (size_t i = g0; i < std::min(g0 + per_src, rem.size()); ++i) push(0, rem[i]);
            if (g0 >= per_src)
                for (size_t i = g0 - per_src; i < g0; ++i) push(1, rem[i]);
        }
        for (size_t i = rem.size() >= per_src ? rem.size() - per_src : 0; i < rem.size(); ++i) push(1, rem[i]);
    } else {
        for (const Unit& u : loc) push(0, u);
        for (const Unit& u : rem) push(0, u);
        for (const Unit& u : rem) push(1, u);
        for (const Unit& u : loc) push(1, u);
    }
    blocks.push_back({-1, 0, start, -1});
    return blocks;
}

void set_peer_pointers(const fm_ctx* c, fm::FmParams& p) {
    for (int r = 0; r < c->d.world; ++r) {
        char* b = static_cast<char*>(c->peer_base[r]);
        p.peer_recv_x[r] = reinterpret_cast<__nv_bfloat16*>(b + c->off_recv_x);
        p.peer_ret_y[r] = reinterpret_cast<__nv_bfloat16*>(b + c->off_ret_y);
        p.peer_recv_flag[r] = reinterpret_cast<unsigned long long*>(b + c->off_recv_flag);
        p.peer_recv_rows[r] = reinterpret_cast<unsigned int*>(b + c->off_recv_rows);
        p.peer_ret_flag[r] = reinterpret_cast<unsigned long long*>(b + c->off_ret_flag);
        p.peer_recv_meta[r] = reinterpret_cast<uint4*>(b + c->off_recv_meta);
        p.peer_done_flag[r] = reinterpret_cast<unsigned long long*>(b + c->off_done_flag);
        p.peer_out_acc[r] = reinterpret_cast<__nv_bfloat16*>(b + c->off_out_acc);
    }
}

int check_kernel_status(fm_ctx* c) {
    if (c->dbg_host != nullptr && c->dbg_host->code != 0) {
        static const char* names[] = {"none", "smem-full mbarrier", "smem-empty mbarrier", "tmem-full mbarrier",
                                      "tmem-empty mbarrier", "sched-full mbarrier", "sched-empty mbarrier",
                                      "grid barrier", "dispatch flag (packet never arrived)", "GEMM0 row-block counter",
                                      "return flag (expert output never arrived)",
                                      "dispatch row acknowledgement (rows of a packet never arrived)", "publisher mbarrier"};
        const fm::DebugRecord r = *c->dbg_host;
        const char* nm = r.code < sizeof(names) / sizeof(names[0]) ? names[r.code] : "unknown";
        return fail(FM_EKERNEL,
                    "kernel wait timed out on %s: block %u thread %u info=(%u,%u,%u) waited %.1f ms (rank %d, launch %llu)",
                    nm, r.block, r.thread, r.info0, r.info1, r.info2, (double)r.waited_ns * 1e-6, c->d.rank,
                    (unsigned long long)c->launches);
    }
    return FM_OK;
}

int launch(fm_ctx* c, const void* x, const void* gate_w, const void* expert_w, const void* bias_up,
           const void* bias_down, void* out, cudaStream_t stream, uint32_t phase_mask) {
    if (c == nullptr) return fail(FM_EINVAL, "null context");
    if (x == nullptr || gate_w == nullptr || expert_w == nullptr || out == nullptr)
        return fail(FM_EINVAL, "x, gate_w, expert_w and out must be non-null device pointers");
    {   // TMA tensor maps, cp.async.bulk row copies and the 16-byte vector accesses all need 16-byte aligned bases
        const void* ptrs[] = {x, gate_w, expert_w, bias_up, bias_down, out};
        const char* names[] = {"x", "gate_w", "expert_w", "bias_up", "bias_down", "out"};
        for (int i = 0; i < 6; ++i)
            if (reinterpret_cast<uintptr_t>(ptrs[i]) % 16)
                return fail(FM_EINVAL, "%s must be 16-byte aligned (got %p)", names[i], ptrs[i]);
    }
    if (!c->attached) return fail(FM_ESTATE, "peers not attached: call fm_symm_attach_ipc/ptrs before fm_moe_forward");
    if ((phase_mask & 1u) == 0u && c->d.world != 1) return fail(FM_EINVAL, "partial-phase launches are single-rank only");
    if ((phase_mask & 1u) == 0u && c->epoch == 0) return fail(FM_ESTATE, "no previous routing to reuse");
    FM_CUDA(cudaSetDevice(c->device));
    const fm_dims_t& d = c->d;
    const int nLx = d.num_local_experts;
    int rc;
    if (c->dense && c->cached_x != x) {   // E == 1: the A operand of GEMM0 is the caller's x itself
        if ((rc = make_tmap(&c->tm_a0, x, (uint64_t)d.S, d.H, fm::BLOCK_M))) return rc;
        c->cached_x = x;
    }
    if (c->tc_gate) {
        // router on tensor cores: x as [S, H] in 32-row boxes, Wg_eff = the [H, E] tensor read flat as [E, H]
        // (python_bindings.cu:93-99, moe.cuh:107-109) in boxes of E_pad rows (a CTA pair stages half each); rows past E
        // read as zero
        if (c->cached_gx != x) {
            if ((rc = make_tmap(&c->tm_gx, x, (uint64_t)d.S, d.H, 32))) return rc;
            c->cached_gx = x;
        }
        if (c->cached_gw != gate_w) {
            const uint32_t e_pad = (uint32_t)((d.E + 15) / 16 * 16);
            if ((rc = make_tmap(&c->tm_gw, gate_w, (uint64_t)d.E, d.H, c->pair ? e_pad / 2 : e_pad))) return rc;
            c->cached_gw = gate_w;
        }
    }
    if (!c->tm_static_ready) {
        if (!c->dense && (rc = make_tmap(&c->tm_a0, static_cast<char*>(c->symm) + c->off_recv_x, (uint64_t)c->num_pkts * d.pEC, d.H,
                                         fm::BLOCK_M)))
            return rc;
        if ((rc = make_tmap(&c->tm_a1, c->hidden, (uint64_t)c->num_pkts * d.pEC, d.P, fm::BLOCK_M))) return rc;
        c->tm_static_ready = true;
    }
    if (c->cached_expert_w != expert_w) {
        // expert_weights [nLx, 2, P, H]: [i,0] is W_up [P,H]; [i,1] is the same P*H block viewed as W_down [H,P]
        // (python_bindings.cu:104-119).  One tensor map per GEMM over the whole tensor with a per-expert row stride
        // of 2*P (resp. 2*H) rows is not expressible in 2-D, so rows are addressed as [nLx*2*P, H] / [nLx*2*H, P]:
        // expert i's W_up starts at row i*2*P, its W_down at row (i*2+1)*H of the [.,P] view.
        // in pair mode each CTA of the pair stages half of the B tile's rows
        const uint32_t b_box = (uint32_t)fm::BLOCK_N / (c->pair ? 2u : 1u);
        if ((rc = make_tmap(&c->tm_b0, expert_w, (uint64_t)nLx * 2 * d.P, d.H, b_box))) return rc;
        if ((rc = make_tmap(&c->tm_b1, expert_w, (uint64_t)nLx * 2 * d.H, d.P, b_box))) return rc;
        c->cached_expert_w = expert_w;
    }
    fm::FmParams p;
    memset(&p, 0, sizeof(p));
    p.tm_a0 = c->tm_a0; p.tm_b0 = c->tm_b0; p.tm_a1 = c->tm_a1; p.tm_b1 = c->tm_b1;
    if (c->tc_gate) { p.tm_gx = c->tm_gx; p.tm_gw = c->tm_gw; }
    p.tc_gate = c->tc_gate ? 1 : 0;
    p.S = d.S; p.H = d.H; p.P = d.P; p.E = d.E; p.k = d.k; p.W = d.world; p.rank = d.rank; p.nLx = nLx;
    p.EC = d.EC; p.pEC = d.pEC; p.TCM = d.TCM; p.act = c->cfg.hidden_act;
    p.TN0 = c->TN0; p.TN1 = c->TN1; p.tpc = c->tpc; p.num_pkts = c->num_pkts; p.num_blocks = c->num_blocks;
    p.total_items = c->total_items;
    // the epoch and the grid-barrier target advance only when the launch has been accepted (see below): a failed launch
    // must not leave the host ahead of the device counter and of the peers
    const uint32_t epoch = c->epoch + ((phase_mask & 1u) ? 1u : 0u);
    const unsigned long long bar_count = c->bar_count + ((phase_mask & 1u) ? (unsigned long long)c->grid : 0ull);
    p.epoch = epoch;
    p.phase_mask = phase_mask;
    p.bar_target = bar_count;
    p.timeout_ns = c->timeout_ns;
    p.x = static_cast<const __nv_bfloat16*>(x);
    p.wg = static_cast<const __nv_bfloat16*>(gate_w);
    p.b_up = static_cast<const __nv_bfloat16*>(bias_up);
    p.b_down = static_cast<const __nv_bfloat16*>(bias_down);
    p.out = static_cast<__nv_bfloat16*>(out);
    p.topk_idx = c->topk_idx; p.topk_w = c->topk_w; p.mcw = c->mcw; p.slot = c->slot; p.counts = c->counts;
    p.gate_out = c->gate_out; p.chunk_counts = c->chunk_counts;
    p.claim = c->ctrl + 1;
    p.grid_bar = reinterpret_cast<unsigned long long*>(c->ctrl + 2);
    p.g0_done = c->g0_done; p.g1_done = c->g1_done; p.recv_cnt = c->recv_cnt; p.blocks = c->blocks;
    p.hidden = c->hidden;
    char* sb = static_cast<char*>(c->symm);
    p.recv_x = reinterpret_cast<__nv_bfloat16*>(sb + c->off_recv_x);
    p.ret_y = reinterpret_cast<__nv_bfloat16*>(sb + c->off_ret_y);
    p.recv_flag = reinterpret_cast<unsigned long long*>(sb + c->off_recv_flag);
    p.recv_rows = reinterpret_cast<unsigned int*>(sb + c->off_recv_rows);
    p.ret_flag = reinterpret_cast<unsigned long long*>(sb + c->off_ret_flag);
    set_peer_pointers(c, p);
    p.fused = c->fused ? 1 : 0;
    p.pkt_done = c->pkt_done;
    p.recv_meta = reinterpret_cast<uint4*>(sb + c->off_recv_meta);
    p.done_flag = reinterpret_cast<unsigned long long*>(sb + c->off_done_flag);
    // single rank: accumulate straight into the caller's tensor; otherwise into the peer-mapped accumulator
    p.out_acc = d.world == 1 ? p.out : reinterpret_cast<__nv_bfloat16*>(sb + c->off_out_acc);
    if (d.world == 1) p.peer_out_acc[0] = p.out;
    p.aux = c->aux;
    p.dense = c->dense ? 1 : 0;
    p.dbg = c->dbg_dev;
    p.trace = c->trace_on ? c->trace : nullptr;

    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(c->grid);
    lc.blockDim = dim3(fm::NUM_THREADS);
    lc.dynamicSmemBytes = (size_t)fm::SMEM_BYTES;
    lc.stream = stream;
    cudaLaunchAttribute attrs[2];
    int na = 0;
    if (c->coop) {
        attrs[na].id = cudaLaunchAttributeCooperative;   // all CTAs co-resident: in-kernel spin waits + grid barrier
        attrs[na].val.cooperative = 1;
        ++na;
    }
    if (c->pair) {
        attrs[na].id = cudaLaunchAttributeClusterDimension;
        attrs[na].val.clusterDim.x = 2;
        attrs[na].val.clusterDim.y = 1;
        attrs[na].val.clusterDim.z = 1;
        ++na;
    }
    lc.attrs = attrs;
    lc.numAttrs = na;
    if (c->pair) FM_CUDA(cudaLaunchKernelEx(&lc, fm::fm_moe_forward_kernel<true>, p));
    else FM_CUDA(cudaLaunchKernelEx(&lc, fm::fm_moe_forward_kernel<false>, p));
    c->epoch = epoch;
    c->bar_count = bar_count;
    c->launches += 1;
    return FM_OK;
}

}  // namespace

// =================================================================================================================
extern "C" {

FM_API const char* fm_last_error(void) { return g_err.c_str(); }
FM_API const char* fm_version(void) { return "flashmoe_b200 0.1.0 (sm_100a, tcgen05/TMEM/TMA)"; }

FM_API int fm_compiled_config(fm_config_t* out) {
    if (out == nullptr) return fail(FM_EINVAL, "null output");
    out->capacity_factor = FM_CFG_CAPACITY_FACTOR;
    out->drop_tokens = FM_CFG_DROP_TOKENS;
    out->expert_top_k = FM_CFG_EXPERT_TOP_K;
    out->global_batch = FM_CFG_GLOBAL_BATCH;
    out->is_training = FM_CFG_IS_TRAINING;
    out->hidden_act = FM_CFG_HIDDEN_ACT;
    out->hidden_size = FM_CFG_HIDDEN_SIZE;
    out->intermediate_size = FM_CFG_INTERMEDIATE_SIZE;
    out->mini_batch = FM_CFG_MINI_BATCH;
    out->moe_frequency = FM_CFG_MOE_FREQUENCY;
    out->num_experts = FM_CFG_NUM_EXPERTS;
    out->num_layers = FM_CFG_NUM_LAYERS;
    out->sequence_len = FM_CFG_SEQUENCE_LEN;
    out->torch_dtype = FM_CFG_TORCH_DTYPE;
    out->vocab_size = FM_CFG_VOCAB_SIZE;
    return FM_OK;
}

FM_API int fm_create(const fm_config_t* cfg, int rank, int world, int device, fm_ctx_t** out) {
    if (out == nullptr) return fail(FM_EINVAL, "null output");
    *out = nullptr;
    fm_config_t c;
    if (cfg != nullptr) c = *cfg;
    else fm_compiled_config(&c);
    fm_dims_t d;
    memset(&d, 0, sizeof(d));
    int rc = validate_config(c, world, &d);
    if (rc) return rc;
    if (rank < 0 || rank >= world) return fail(FM_EINVAL, "rank %d not in [0, %d)", rank, world);
    d.rank = rank;

    int ndev = 0;
    FM_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(FM_EINVAL, "device %d not in [0, %d)", device, ndev);
    FM_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    FM_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(FM_ECUDA, "device %d is sm_%d%d; this library contains sm_100a code only (tcgen05/TMEM/TMA)", device,
                    prop.major, prop.minor);
    int coop = 0;
    FM_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
    if (!coop) return fail(FM_ECUDA, "device does not support cooperative launch");
    d.num_sms = prop.multiProcessorCount;
    d.smem_bytes = fm::SMEM_BYTES;
    d.grid = prop.multiProcessorCount;

    FM_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(&fm::fm_moe_forward_kernel<false>),
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, fm::SMEM_BYTES));
    FM_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(&fm::fm_moe_forward_kernel<true>),
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, fm::SMEM_BYTES));
    int occ = 0;
    FM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fm::fm_moe_forward_kernel<false>, fm::NUM_THREADS,
                                                          (size_t)fm::SMEM_BYTES));
    if (occ < 1) return fail(FM_ECUDA, "kernel does not fit on an SM (smem %d B)", fm::SMEM_BYTES);

    fm_ctx* ctx = new fm_ctx();
    ctx->cfg = c;
    ctx->d = d;
    ctx->device = device;
    // environment overrides of the defaults below: tests use them to cross-check the alternative paths
    auto env_int = [](const char* name, int dflt) {
        const char* v = getenv(name);
        return (v != nullptr && *v) ? atoi(v) : dflt;
    };
    ctx->grid = d.num_sms;  // one persistent CTA per SM; all co-resident (spin waits + grid barrier)
    ctx->pair = env_int("FM_PAIR", 1) != 0;   // default: CTA pairs (measured +9 % on config B)
    // fused GEMM1 -> combine (REDG into the token's output row): only for k <= 2, where bf16 accumulation is
    // order-independent (0 + a exact, a + b commutative) and therefore bit-identical to the deterministic gather;
    // k > 2 keeps the gather so results do not depend on arrival order
    ctx->fused = env_int("FM_FUSED_COMBINE", 1) != 0 && d.k <= 2;
    ctx->dense = d.E == 1 && world == 1 && env_int("FM_DENSE_E1", 1) != 0;
    // router logits by tcgen05.mma instead of the CUDA-core GEMV (2*S*H*E flops: 4.3 GFLOP per rank at E = 128,
    // d_model 2048, 8192 tokens -- ~0.2 ms on the CUDA cores); one accumulator holds <= 256 experts
    // Default: from 17 experts up.  Measured on one B200: E = 128, d_model 2048, 56 tokens per CTA: router 29 us instead
    // of 433 us; E = 8, d_model 1024, 28 tokens per CTA (config B): a wash (the GEMV is latency-, not flop-bound there).
    ctx->tc_gate = !ctx->dense && d.E <= 256 && env_int("FM_TC_GATE", d.E > 16 ? 1 : 0) != 0;
    if (ctx->pair && (ctx->grid & 1)) ctx->grid -= 1;  // CTA pairs need an even grid
    ctx->d.grid = ctx->grid;
    ctx->tpc = ceil_div(d.S, ctx->grid);
    if ((long long)ctx->tpc * d.k > fm::G_SEL_MAX) {
        delete ctx;
        return fail(FM_EINVAL, "tokens-per-CTA * k = %d exceeds the router scratch (%d)", ctx->tpc * d.k, fm::G_SEL_MAX);
    }
    const int nLx = d.num_local_experts;
    // The persistent grid spins on flags, counters and one grid barrier, so every CTA must be resident: the launch is
    // cooperative (the driver then refuses to start it unless the whole grid fits, also next to other work on the GPU).
    // One exception: Nsight Compute cannot replay a cooperative launch that also has cluster dimensions (the driver
    // reports LaunchFailed), so under a CUDA injection profiler -- or with FM_COOP=0 -- the attribute is dropped and
    // co-residency rests on the cudaOccupancyMaxActiveClusters check below plus exclusive use of the GPU.
    const bool under_profiler = getenv("CUDA_INJECTION64_PATH") != nullptr || getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR") != nullptr ||
                                getenv("NSIGHT_CUDA_DEBUGGER") != nullptr;
    ctx->coop = env_int("FM_COOP", (ctx->pair && under_profiler) ? 0 : 1) != 0;
    if (ctx->pair) {
        cudaLaunchConfig_t oc = {};
        oc.gridDim = dim3(ctx->grid);
        oc.blockDim = dim3(fm::NUM_THREADS);
        oc.dynamicSmemBytes = (size_t)fm::SMEM_BYTES;
        cudaLaunchAttribute oa[1];
        oa[0].id = cudaLaunchAttributeClusterDimension;
        oa[0].val.clusterDim.x = 2; oa[0].val.clusterDim.y = 1; oa[0].val.clusterDim.z = 1;
        oc.attrs = oa;
        oc.numAttrs = 1;
        int max_clusters = 0;
        cudaError_t oe = cudaOccupancyMaxActiveClusters(&max_clusters, fm::fm_moe_forward_kernel<true>, &oc);
        if (oe != cudaSuccess || max_clusters * 2 < ctx->grid) {
            const int got = max_clusters;
            delete ctx;
            return fail(FM_ECUDA, "the persistent grid of %d CTA pairs cannot be co-resident (max active clusters %d, %s)",
                        d.num_sms / 2, got, cudaGetErrorString(oe));
        }
    }
    ctx->TN0 = ceil_div(d.P, fm::BLOCK_N);
    ctx->TN1 = ceil_div(d.H, fm::BLOCK_N);
    ctx->num_pkts = world * nLx;
    std::vector<fm::TileBlock> blocks = build_work_list(world, rank, nLx, d.TCM, ctx->TN0, ctx->TN1, ctx->pair);
    ctx->num_blocks = (int)blocks.size() - 1;
    ctx->total_items = blocks.back().start;

#define FM_TRY(expr)          \
    do {                      \
        rc = (expr);          \
        if (rc) {             \
            fm_destroy(ctx);  \
            return rc;        \
        }                     \
    } while (0)
#define FM_TRY_CUDA(expr)                                                                             \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            fm_destroy(ctx);                                                                          \
            return fail(FM_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));                    \
        }                                                                                             \
    } while (0)

    FM_TRY(dev_alloc(&ctx->topk_idx, (size_t)d.S * d.k));
    FM_TRY(dev_alloc(&ctx->topk_w, (size_t)d.S * d.k));
    FM_TRY(dev_alloc(&ctx->mcw, (size_t)d.S));
    FM_TRY(dev_alloc(&ctx->slot, (size_t)d.S * d.k));
    FM_TRY(dev_alloc(&ctx->counts, (size_t)d.E));
    FM_TRY(dev_alloc(&ctx->gate_out, (size_t)d.S * d.E));
    FM_TRY(dev_alloc(&ctx->chunk_counts, (size_t)ctx->grid * d.E));
    FM_TRY(dev_alloc(&ctx->ctrl, 8));
    FM_TRY(dev_alloc(&ctx->g0_done, (size_t)ctx->num_pkts * d.TCM));
    FM_TRY(dev_alloc(&ctx->g1_done, (size_t)ctx->num_pkts * d.TCM));
    FM_TRY(dev_alloc(&ctx->recv_cnt, (size_t)ctx->num_pkts));
    FM_TRY(dev_alloc(&ctx->pkt_done, (size_t)ctx->num_pkts));
    FM_TRY(dev_alloc(&ctx->blocks, blocks.size(), false));
    FM_TRY_CUDA(cudaMemcpy(ctx->blocks, blocks.data(), blocks.size() * sizeof(fm::TileBlock), cudaMemcpyHostToDevice));
    FM_TRY(dev_alloc(&ctx->hidden, (size_t)ctx->num_pkts * d.pEC * d.P));
    FM_TRY(dev_alloc(&ctx->trace, (size_t)ctx->grid * fm::TRACE_SLOTS));
    if (c.is_training) FM_TRY(dev_alloc(&ctx->aux, (size_t)2 * (2 * d.E + 1)));

    // symmetric slab: [recv_x | ret_y | recv_flag | ret_flag]  (reference heap + flags, bootstrap.cuh:348-362)
    size_t off = 0;
    // the return buffer + per-row-block return flags exist only on the gather-combine path (the fused path adds
    // straight into the token's output row)
    ctx->off_recv_x = off; off = align_up(off + (size_t)ctx->num_pkts * d.pEC * d.H * 2, 1024);
    ctx->off_ret_y = off;  off = align_up(off + (ctx->fused ? 0 : (size_t)d.E * d.pEC * d.H * 2), 1024);
    ctx->off_recv_flag = off; off = align_up(off + (size_t)ctx->num_pkts * 8, 1024);
    ctx->off_recv_rows = off; off = align_up(off + (size_t)2 * ctx->num_pkts * d.TCM * 4, 1024);
    ctx->off_ret_flag = off;  off = align_up(off + (ctx->fused ? 0 : (size_t)d.E * d.TCM * 8), 1024);
    ctx->off_recv_meta = off; off = align_up(off + (size_t)ctx->num_pkts * d.pEC * 16, 1024);
    ctx->off_done_flag = off; off = align_up(off + (size_t)d.E * 8, 1024);
    ctx->off_out_acc = off;   off = align_up(off + (world > 1 ? (size_t)d.S * d.H * 2 : 0), 1024);
    ctx->symm_bytes = off;
    {
        void* q = nullptr;
        cudaError_t e = cudaMalloc(&q, ctx->symm_bytes);
        if (e != cudaSuccess) {
            fm_destroy(ctx);
            return fail(FM_ENOMEM, "cudaMalloc(symmetric slab, %zu bytes) failed: %s", ctx->symm_bytes, cudaGetErrorString(e));
        }
        ctx->symm = q;
        FM_TRY_CUDA(cudaMemset(q, 0, ctx->symm_bytes));
    }
    FM_TRY_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ctx->dbg_host), sizeof(fm::DebugRecord), cudaHostAllocMapped));
    memset(ctx->dbg_host, 0, sizeof(fm::DebugRecord));
    FM_TRY_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->dbg_dev), ctx->dbg_host, 0));
    FM_TRY_CUDA(cudaDeviceSynchronize());
    if (world == 1) {
        ctx->peer_base[0] = ctx->symm;
        ctx->attached = true;
    }
#undef FM_TRY
#undef FM_TRY_CUDA
    *out = ctx;
    return FM_OK;
}

FM_API int fm_destroy(fm_ctx_t* ctx) {
    if (ctx == nullptr) return FM_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < ctx->d.world; ++r)
        if (ctx->peer_opened[r] && ctx->peer_base[r] != nullptr) cudaIpcCloseMemHandle(ctx->peer_base[r]);
    void* bufs[] = {ctx->topk_idx, ctx->topk_w, ctx->mcw, ctx->slot, ctx->counts, ctx->gate_out, ctx->chunk_counts,
                    ctx->ctrl, ctx->g0_done, ctx->g1_done, ctx->pkt_done, ctx->recv_cnt, ctx->blocks, ctx->hidden, ctx->trace,
                    ctx->aux};
    for (void* b : bufs)
        if (b != nullptr) cudaFree(b);
    for (int i = 0; i < FM_HOST_SLOTS; ++i) {
        if (ctx->x_stage[i] != nullptr) cudaFree(ctx->x_stage[i]);
        if (ctx->out_stage[i] != nullptr) cudaFree(ctx->out_stage[i]);
        if (ctx->ev_h2d[i] != nullptr) cudaEventDestroy(ctx->ev_h2d[i]);
        if (ctx->ev_kernel[i] != nullptr) cudaEventDestroy(ctx->ev_kernel[i]);
        if (ctx->ev_d2h[i] != nullptr) cudaEventDestroy(ctx->ev_d2h[i]);
    }
    if (ctx->s_h2d != nullptr) cudaStreamDestroy(ctx->s_h2d);
    if (ctx->s_d2h != nullptr) cudaStreamDestroy(ctx->s_d2h);
    if (ctx->symm != nullptr && !ctx->symm_external) cudaFree(ctx->symm);
    if (ctx->dbg_host != nullptr) cudaFreeHost(ctx->dbg_host);
    delete ctx;
    return FM_OK;
}

FM_API int fm_get_dims(const fm_ctx_t* ctx, fm_dims_t* out) {
    if (ctx == nullptr || out == nullptr) return fail(FM_EINVAL, "null argument");
    *out = ctx->d;
    return FM_OK;
}

FM_API int fm_num_local_experts(const fm_ctx_t* ctx) {
    if (ctx == nullptr) return fail(FM_EINVAL, "null context");
    return ctx->d.num_local_experts;
}

FM_API int fm_symm_size(const fm_ctx_t* ctx, size_t* bytes) {
    if (ctx == nullptr || bytes == nullptr) return fail(FM_EINVAL, "null argument");
    *bytes = ctx->symm_bytes;
    return FM_OK;
}

FM_API int fm_symm_local_ptr(const fm_ctx_t* ctx, void** base) {
    if (ctx == nullptr || base == nullptr) return fail(FM_EINVAL, "null argument");
    *base = ctx->symm;
    return FM_OK;
}

FM_API int fm_output_buffer(const fm_ctx_t* ctx, void** ptr, size_t* bytes) {
    if (ctx == nullptr || ptr == nullptr || bytes == nullptr) return fail(FM_EINVAL, "null argument");
    const bool has = ctx->d.world > 1;   // the accumulation target peers add into; single rank: the caller's tensor
    *ptr = has ? static_cast<char*>(ctx->symm) + ctx->off_out_acc : nullptr;
    *bytes = has ? (size_t)ctx->d.S * ctx->d.H * 2 : 0;
    return FM_OK;
}

FM_API int fm_symm_use_external(fm_ctx_t* ctx, void* base, size_t bytes) {
    if (ctx == nullptr || base == nullptr) return fail(FM_EINVAL, "null argument");
    if (ctx->attached && ctx->d.world > 1) return fail(FM_ESTATE, "already attached");
    if (bytes < ctx->symm_bytes) return fail(FM_EINVAL, "external slab too small: %zu < %zu", bytes, ctx->symm_bytes);
    if (reinterpret_cast<uintptr_t>(base) % 1024) return fail(FM_EINVAL, "external slab must be 1 KiB aligned");
    FM_CUDA(cudaSetDevice(ctx->device));
    if (ctx->symm != nullptr && !ctx->symm_external) FM_CUDA(cudaFree(ctx->symm));
    ctx->symm = base;
    ctx->symm_external = true;
    ctx->tm_static_ready = false;
    if (ctx->d.world == 1) ctx->peer_base[0] = base;
    return FM_OK;
}

FM_API int fm_symm_export(fm_ctx_t* ctx, void* handle_out) {
    if (ctx == nullptr || handle_out == nullptr) return fail(FM_EINVAL, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == FM_IPC_HANDLE_BYTES, "IPC handle size");
    FM_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    FM_CUDA(cudaIpcGetMemHandle(&h, ctx->symm));
    memcpy(handle_out, &h, sizeof(h));
    return FM_OK;
}

FM_API int fm_symm_attach_ipc(fm_ctx_t* ctx, const void* all_handles) {
    if (ctx == nullptr || all_handles == nullptr) return fail(FM_EINVAL, "null argument");
    if (ctx->attached && ctx->d.world > 1) return fail(FM_ESTATE, "already attached");
    FM_CUDA(cudaSetDevice(ctx->device));
    const char* hs = static_cast<const char*>(all_handles);
    for (int r = 0; r < ctx->d.world; ++r) {
        if (r == ctx->d.rank) {
            ctx->peer_base[r] = ctx->symm;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, hs + (size_t)r * FM_IPC_HANDLE_BYTES, sizeof(h));
        void* ptr = nullptr;
        FM_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        ctx->peer_base[r] = ptr;
        ctx->peer_opened[r] = true;
    }
    ctx->attached = true;
    return FM_OK;
}

FM_API int fm_symm_attach_ptrs(fm_ctx_t* ctx, void* const* peer_bases) {
    if (ctx == nullptr || peer_bases == nullptr) return fail(FM_EINVAL, "null argument");
    for (int r = 0; r < ctx->d.world; ++r) {
        if (peer_bases[r] == nullptr) return fail(FM_EINVAL, "peer base %d is null", r);
        ctx->peer_base[r] = (r == ctx->d.rank) ? ctx->symm : peer_bases[r];
    }
    ctx->attached = true;
    return FM_OK;
}

FM_API int fm_moe_forward(fm_ctx_t* ctx, const void* x, const void* gate_w, const void* expert_w, const void* bias_up,
                          const void* bias_down, void* out, void* stream) {
    return launch(ctx, x, gate_w, expert_w, bias_up, bias_down, out, static_cast<cudaStream_t>(stream), 7u);
}

FM_API int fm_debug_forward(fm_ctx_t* ctx, const void* x, const void* gate_w, const void* expert_w,
                            const void* bias_up, const void* bias_down, void* out, void* stream, uint32_t phase_mask) {
    if (phase_mask == 0 || phase_mask > 7u) return fail(FM_EINVAL, "phase_mask must be in [1, 7]");
    return launch(ctx, x, gate_w, expert_w, bias_up, bias_down, out, static_cast<cudaStream_t>(stream), phase_mask);
}

// ---- host-buffer entry points -----------------------------------------------------------------------------------
static int host_setup(fm_ctx* c) {
    if (c->host_ready) return FM_OK;
    const size_t elems = (size_t)c->d.S * c->d.H;
    int rc;
    for (int i = 0; i < FM_HOST_SLOTS; ++i) {
        if ((rc = dev_alloc(&c->x_stage[i], elems, false))) return rc;
        if ((rc = dev_alloc(&c->out_stage[i], elems, false))) return rc;
        FM_CUDA(cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming));
        FM_CUDA(cudaEventCreateWithFlags(&c->ev_kernel[i], cudaEventDisableTiming));
        FM_CUDA(cudaEventCreateWithFlags(&c->ev_d2h[i], cudaEventDisableTiming));
    }
    FM_CUDA(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    FM_CUDA(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
    c->host_ready = true;
    return FM_OK;
}

FM_API int fm_host_submit(fm_ctx_t* ctx, const void* x_host, const void* gate_w, const void* expert_w, const void* bias_up,
                          const void* bias_down, void* out_host, void* stream, uint64_t* ticket) {
    if (ctx == nullptr || x_host == nullptr || out_host == nullptr || ticket == nullptr) return fail(FM_EINVAL, "null argument");
    FM_CUDA(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = host_setup(ctx))) return rc;
    if (ctx->host_submitted - ctx->host_waited >= FM_HOST_SLOTS)
        return fail(FM_ESTATE, "%d steps in flight: call fm_host_wait on the oldest ticket first", FM_HOST_SLOTS);
    const size_t bytes = (size_t)ctx->d.S * ctx->d.H * 2;
    const int slot = (int)(ctx->host_submitted % FM_HOST_SLOTS);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // x_stage[slot] was last read by the kernel of step (submitted - SLOTS): the H2D copy waits for that kernel
    // (out_stage[slot]'s previous D2H has been waited for on the host already, see the in-flight bound above)
    if (ctx->host_submitted >= FM_HOST_SLOTS) FM_CUDA(cudaStreamWaitEvent(ctx->s_h2d, ctx->ev_kernel[slot], 0));
    FM_CUDA(cudaMemcpyAsync(ctx->x_stage[slot], x_host, bytes, cudaMemcpyHostToDevice, ctx->s_h2d));
    FM_CUDA(cudaEventRecord(ctx->ev_h2d[slot], ctx->s_h2d));
    FM_CUDA(cudaStreamWaitEvent(s, ctx->ev_h2d[slot], 0));
    if ((rc = launch(ctx, ctx->x_stage[slot], gate_w, expert_w, bias_up, bias_down, ctx->out_stage[slot], s, 7u))) return rc;
    FM_CUDA(cudaEventRecord(ctx->ev_kernel[slot], s));
    FM_CUDA(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_kernel[slot], 0));
    FM_CUDA(cudaMemcpyAsync(out_host, ctx->out_stage[slot], bytes, cudaMemcpyDeviceToHost, ctx->s_d2h));
    FM_CUDA(cudaEventRecord(ctx->ev_d2h[slot], ctx->s_d2h));
    *ticket = ctx->host_submitted++;
    return FM_OK;
}

FM_API int fm_host_wait(fm_ctx_t* ctx, uint64_t ticket) {
    if (ctx == nullptr) return fail(FM_EINVAL, "null context");
    if (ticket >= ctx->host_submitted) return fail(FM_EINVAL, "ticket %llu was never issued", (unsigned long long)ticket);
    if (ticket < ctx->host_waited) return FM_OK;   // already complete
    if (ticket != ctx->host_waited) return fail(FM_ESTATE, "tickets must be waited for in submission order (oldest is %llu)",
                                                (unsigned long long)ctx->host_waited);
    FM_CUDA(cudaSetDevice(ctx->device));
    cudaError_t e = cudaEventSynchronize(ctx->ev_d2h[ticket % FM_HOST_SLOTS]);
    int rc;
    if ((rc = check_kernel_status(ctx))) return rc;
    if (e != cudaSuccess) return fail(FM_ECUDA, "cudaEventSynchronize failed: %s", cudaGetErrorString(e));
    ctx->host_waited = ticket + 1;
    return FM_OK;
}

FM_API int fm_moe_forward_host(fm_ctx_t* ctx, const void* x_host, const void* gate_w, const void* expert_w,
                               const void* bias_up, const void* bias_down, void* out_host, void* stream) {
    if (ctx == nullptr) return fail(FM_EINVAL, "null context");
    int rc;
    while (ctx->host_waited < ctx->host_submitted)   // drain earlier asynchronous steps first
        if ((rc = fm_host_wait(ctx, ctx->host_waited))) return rc;
    uint64_t t = 0;
    if ((rc = fm_host_submit(ctx, x_host, gate_w, expert_w, bias_up, bias_down, out_host, stream, &t))) return rc;
    return fm_host_wait(ctx, t);
}

FM_API int fm_check(fm_ctx_t* ctx) {
    if (ctx == nullptr) return fail(FM_EINVAL, "null context");
    return check_kernel_status(ctx);
}

FM_API int fm_set_timeout_ms(fm_ctx_t* ctx, uint32_t ms) {
    if (ctx == nullptr) return fail(FM_EINVAL, "null context");
    ctx->timeout_ns = (unsigned long long)ms * 1000000ull;
    return FM_OK;
}

FM_API int fm_set_trace(fm_ctx_t* ctx, int enable) {
    if (ctx == nullptr) return fail(FM_EINVAL, "null context");
    ctx->trace_on = enable != 0;
    return FM_OK;
}

FM_API uint64_t fm_launch_count(const fm_ctx_t* ctx) { return ctx ? ctx->launches : 0; }

static int buffer_desc(const fm_ctx_t* c, int which, const void** ptr, size_t* bytes) {
    const fm_dims_t& d = c->d;
    const char* sb = static_cast<const char*>(c->symm);
    switch (which) {
        case FM_BUF_TOPK_IDX: *ptr = c->topk_idx; *bytes = (size_t)d.S * d.k * 4; break;
        case FM_BUF_TOPK_W: *ptr = c->topk_w; *bytes = (size_t)d.S * d.k * 2; break;
        case FM_BUF_MCW: *ptr = c->mcw; *bytes = (size_t)d.S * 4; break;
        case FM_BUF_SLOT: *ptr = c->slot; *bytes = (size_t)d.S * d.k * 4; break;
        case FM_BUF_COUNTS: *ptr = c->counts; *bytes = (size_t)d.E * 4; break;
        case FM_BUF_RECV_X: *ptr = sb + c->off_recv_x; *bytes = (size_t)c->num_pkts * d.pEC * d.H * 2; break;
        case FM_BUF_HIDDEN: *ptr = c->hidden; *bytes = (size_t)c->num_pkts * d.pEC * d.P * 2; break;
        case FM_BUF_RET_Y:
            if (c->fused) return fail(FM_EINVAL, "the return buffer does not exist on the fused-combine path (FM_FUSED_COMBINE=0 keeps it)");
            *ptr = sb + c->off_ret_y; *bytes = (size_t)d.E * d.pEC * d.H * 2; break;
        case FM_BUF_GATE_OUT: *ptr = c->gate_out; *bytes = (size_t)d.S * d.E * 2; break;
        case FM_BUF_RECV_CNT: *ptr = c->recv_cnt; *bytes = (size_t)c->num_pkts * 4; break;
        case FM_BUF_TRACE: *ptr = c->trace; *bytes = (size_t)c->grid * fm::TRACE_SLOTS * 8; break;
        case FM_BUF_AUX_LOSS:
            if (c->aux == nullptr) return fail(FM_EINVAL, "the auxiliary loss exists only with is_training = 1");
            *ptr = c->aux + (size_t)(c->epoch & 1u) * (2 * d.E + 1); *bytes = (size_t)(2 * d.E + 1) * 4; break;
        default: return fail(FM_EINVAL, "unknown buffer id %d", which);
    }
    return FM_OK;
}

FM_API int fm_buffer_bytes(const fm_ctx_t* ctx, int which, size_t* bytes) {
    if (ctx == nullptr || bytes == nullptr) return fail(FM_EINVAL, "null argument");
    const void* p = nullptr;
    return buffer_desc(ctx, which, &p, bytes);
}

FM_API int fm_read_buffer(fm_ctx_t* ctx, int which, void* host_dst, size_t bytes) {
    if (ctx == nullptr || host_dst == nullptr) return fail(FM_EINVAL, "null argument");
    const void* p = nullptr;
    size_t n = 0;
    int rc = buffer_desc(ctx, which, &p, &n);
    if (rc) return rc;
    if (bytes != n) return fail(FM_EINVAL, "buffer %d holds %zu bytes, caller asked for %zu", which, n, bytes);
    FM_CUDA(cudaSetDevice(ctx->device));
    cudaError_t e = cudaDeviceSynchronize();
    if ((rc = check_kernel_status(ctx))) return rc;
    if (e != cudaSuccess) return fail(FM_ECUDA, "cudaDeviceSynchronize failed: %s", cudaGetErrorString(e));
    FM_CUDA(cudaMemcpy(host_dst, p, n, cudaMemcpyDeviceToHost));
    return FM_OK;
}

}  // extern "C"
