// tmac_b200.cu -- host side of libtmac_b200.so: context, resident-weight registry, kcfg registry,
// pointer-domain handling and the C ABI declared in include/tmac_b200.h.
//
// Mirrors, for the hot path only:
//   * the generated dispatchers qgemm_lut_int8 / preprocessor_int8 (deploy/compile.py:60-67),
//   * TMAC::TMACGeMMWrapper::{llama_cpp_init, llama_cpp_compute, get_kcfg}
//     (include/t-mac/tmac_gemm_wrapper.h:173-255),
//   * the ggml hook (3rdparty/llama.cpp/ggml/src/ggml-tmac.cpp).
// There is no CPU fallback anywhere in this file: every compute entry point launches CUDA
// kernels or fails with -1.
#include "../../include/tmac_b200.h"

#include <algorithm>
#include <atomic>
#include <functional>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sys/mman.h>
#include <map>
#include <mutex>
#include <shared_mutex>
#include <set>
#include <string>
#include <vector>

#include "tmac_kernels.cuh"
#include "tmac_prefill.cuh"
#include "tmac_prefill16.cuh"
#include "tmac_seq.cuh"
#include "tmac_chain.cuh"
#include "tmac_layout.h"
#include "tmac_gguf.h"

using namespace tmac_b200;

namespace {

thread_local std::string t_err;
int fail(const std::string &m) { t_err = m; return -1; }
#define CUDA_OK(expr)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) return fail(std::string(#expr) + ": " + cudaGetErrorString(e_));    \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t n) {
        if (n <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = std::max(n, (size_t)4096);
        if (cudaMalloc(&p, want) != cudaSuccess) return -1;
        cap = want;
        return 0;
    }
};
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t n) {
        if (n <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = std::max(n, (size_t)65536);
        if (cudaMallocHost(&p, want) != cudaSuccess) return -1;
        cap = want;
        return 0;
    }
};

struct Resident {
    tmac_b200_kcfg cfg{};
    StreamLayout L{};
    unsigned char *d = nullptr;          // stream layout in HBM, then the fp16 prefill tile's row exponents (int [nrsb * rsb] at rexp_off)
    size_t rexp_off = 0, alloc = 0;      // offset of the row exponents, bytes allocated at d
    const unsigned char *host_a = nullptr;  // alias key: reference-layout host range
    size_t host_a_bytes = 0;
    int row0 = 0;                        // first row of the full tensor held here (row shards)
    void *reserved = nullptr;            // address range reserved (PROT_NONE, no memory) to serve as the host alias key
    size_t reserved_bytes = 0;
    float *host_scales = nullptr;        // scales in the reference's run-time order, owned here (tmac_tensor_extra::scales)
    int64_t id = 0;                      // its handle
};

// A LUT that lives in CALLER host memory (the reference's workspace, ref:ggml.c:12566-12576) and its device-resident copy.
// ggml writes the LUT once per mat-vec (task_init) and then calls task_compute once per weight tile with the same pointers
// (ref:ggml.c:12662-12691): the copy is keyed by the host QLUT pointer AND compared with the bytes the call passes, so a caller that
// rewrites the table is never served stale data, and the first tile call computes the whole tensor once (`res`), later tile
// calls of the same (LUT bytes, tensor) copy their rows out.
struct HostLut {
    const void *hq = nullptr;
    std::vector<unsigned char> copy;     // the bytes the device copy was made from: QLUT || LUT_Scales || LUT_Biases (empty = invalid)
    size_t qb = 0, sb = 0;
    int N = 0;
    DevBuf dq, dls, dlb;
    bool sym = false;
    int64_t res_id = 0;                  // tensor whose full result `res` holds (0 = none)
    int res_dtype = 0;
    PinBuf res;                          // [N][Mout] in page-locked host memory, written by the kernel itself
    uint64_t stamp = 0;
};

struct Context {
    bool inited = false;
    int device = 0, sms = 148;
    cudaStream_t own = nullptr, user = nullptr;
    bool use_user = false;
    int float_type = TMAC_B200_F32;
    int lut_mode = 0;                    // 0 auto, 1 general, 2 symmetric
    int use_pdl = 1;
    int cs_override = 0, wpc_override = 0, pdl_late = -1, minb_override = 0, nbuf_override = 0;
    int last_launch[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int use_fused = 1;
    int seq_impl = 2;                    // decode sequences: 0 = stream-K sequence kernel (tmac_seq.cuh), 1 = resident gemv3 chain (tmac_chain.cuh), 2 = chain when the sequence qualifies
    int seq_smem_kb = 200;               // decode sequences: shared-memory budget; the rest of the 228 KB stays L1 (descriptor / polling loads, spills)
    int seq_grid = 0;                    // decode sequences: grid override (tests: CTA-boundary placements); 0 = one CTA per SM
    int use_prefill16 = 1;               // fp16-operand prefill tile for N >= 64 (tmac_prefill16.cuh); 0 = the exact int8 tile for every N >= prefill_min_n
    int pf_streamk = 0;                  // stream-K over all SMs when a prefill call has fewer tiles than SMs (measured slower: B delivery from L2 is the bound)
    int use_prefill = 1, prefill_min_n = 32;   // N >= prefill_min_n: tcgen05 int8 tile (W2 g128 act64)                   // tmac_b200_gemv builds the LUT inside the GEMV when the grouping allows
    int npeer = 0; void *peer_out[7] = {};   // one-shot: peer output vectors of the next N = 1 launch (tmac_b200_peer_outputs)
    int64_t next_hint = 0;               // one-shot: tensor whose blocks the next launch prefetches into L2
    std::map<int64_t, Resident> res;
    int64_t next_handle = 1;
    std::vector<tmac_b200_kcfg> kcfgs;
    HostLut hluts[4];
    uint64_t hlut_clock = 0;
    std::set<const void *> sym_qluts;    // device QLUT buffers last written by our preprocessor
    std::vector<std::pair<std::vector<const void *>, void *>> ptr_tables;   // grouped-launch pointer tables
    // workspaces
    DevBuf d_b, d_qlut, d_ls, d_lb, d_c, d_cbits, d_trace, d_tiles, d_pf_scratch, d_pf_flags, d_pf_texp;
    int trace = 0, trace_ctas = 0, trace_seq = 0;
    int chain_flags = 0;                 // resident chain (tmac_chain.cuh): bit 0 = grid-barrier form (comparison); default: data flow
    PinBuf h_in, h_out;
    cudaEvent_t stage_ev = nullptr;      // last H2D that read h_in
    bool stage_pending = false;
    cudaStream_t stream() const { return use_user ? user : own; }
};

Context g;
std::shared_mutex g_mu;     // exclusive for everything that launches or mutates; shared for the read-only tile fast path
std::map<int64_t, GgufFile *> g_gguf;    // open GGUF files (tmac_b200_gguf_*)
int64_t g_next_gguf = 1;

std::map<int64_t, cudaGraphExec_t> g_graphs;   // tmac_b200_graph_*
int64_t g_next_graph = 1;

// decode sequences (tmac_b200_seq_*)
struct SeqOpHost { int64_t handle; const void *x_ext; int in_op, in_off; void *C; int out_f16; int npeer = 0; void *peer[7] = {}; };
struct Sequence {
    std::vector<SeqOpHost> ops;
    bool built = false;
    int grid = 0, pb = 0, qch = 0, agq = 0, bits = 0;
    seq_fn fn = nullptr;
    size_t smem = 0;
    SeqParams params{};
    int impl = 0;                         // 1: chain_kernel
    chain_fn cfn = nullptr;
    ChainParams cparams{};
    void *d_cops = nullptr, *d_bar = nullptr, *d_cint = nullptr;
    void *d_ops = nullptr, *d_ctas = nullptr, *d_lut = nullptr, *d_y = nullptr, *d_xchg = nullptr, *d_epochs = nullptr, *d_err = nullptr, *d_trace = nullptr;
    void release() {
        for (void *q : {d_ops, d_ctas, d_lut, d_y, d_xchg, d_epochs, d_err, d_trace, d_cops, d_bar, d_cint}) if (q) cudaFree(q);
        d_cops = d_bar = d_cint = nullptr;
        d_ops = d_ctas = d_lut = d_y = d_xchg = d_epochs = d_err = d_trace = nullptr; built = false;
    }
};
std::map<int64_t, Sequence> g_seqs;
int64_t g_next_seq = 1;

bool is_device_ptr(const void *p) {
    if (!p) return false;
    // ggml calls in once per weight tile with pointers into the same few host buffers: remember which 4 KB pages were ORDINARY
    // HOST memory (a page of host address space never becomes device memory; one that gets page-locked later is still valid to
    // treat as pageable), so that cudaPointerGetAttributes (~0.5 us) is not paid 4 times per tile
    static thread_local uintptr_t host_pages[64];
    const uintptr_t page = (uintptr_t)p >> 12, slot = page & 63;
    if (host_pages[slot] == page) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type == cudaMemoryTypeUnregistered) host_pages[slot] = page;
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// The entry whose device copy was made from exactly these host bytes (memcmp of ~17 KB: ~0.1 us), or null.
HostLut *hlut_find(const void *hq, const void *ls, const void *lb, size_t qb, size_t sb) {
    for (HostLut &e : g.hluts)
        if (e.hq == hq && e.qb == qb && e.sb == sb && e.copy.size() == qb + 2 * sb && !std::memcmp(e.copy.data(), hq, qb) &&
            !std::memcmp(e.copy.data() + qb, ls, sb) && !std::memcmp(e.copy.data() + qb + sb, lb, sb)) { e.stamp = ++g.hlut_clock; return &e; }
    return nullptr;
}
HostLut *hlut_slot(const void *hq) {     // the entry of this host pointer, else the least recently used one
    HostLut *best = &g.hluts[0];
    for (HostLut &e : g.hluts) {
        if (e.hq == hq) { best = &e; break; }
        if (e.stamp < best->stamp) best = &e;
    }
    best->hq = hq; best->copy.clear(); best->res_id = 0; best->stamp = ++g.hlut_clock;
    return best;
}

// 0 = ordinary host memory, 1 = page-locked host memory the device can address (dev = its device alias), 2 = device / managed
int ptr_kind(const void *p, void **dev = nullptr) {
    if (!p) return 0;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return 0; }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return 2;
    if (a.type == cudaMemoryTypeHost && a.devicePointer) { if (dev) *dev = a.devicePointer; return 1; }
    return 0;
}

int ensure_init() {
    if (g.inited) {   // the CUDA current device is per host thread (ggml worker threads enter here too)
        static thread_local int t_dev = -1;
        if (t_dev != g.device) { if (cudaSetDevice(g.device) != cudaSuccess) { cudaGetLastError(); return fail("cudaSetDevice failed"); } t_dev = g.device; }
        return 0;
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return fail("no CUDA device: libtmac_b200 has no CPU fallback"); }
    int dev = 0;
    if (const char *e = getenv("TMAC_B200_DEVICE")) dev = atoi(e);
    else { int cur = 0; if (cudaGetDevice(&cur) == cudaSuccess) dev = cur; }
    CUDA_OK(cudaSetDevice(dev));
    g.device = dev;
    cudaDeviceProp prop;
    CUDA_OK(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) return fail("libtmac_b200 is built for sm_100a only (found sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + ")");
    g.sms = prop.multiProcessorCount;
    CUDA_OK(cudaStreamCreate(&g.own));   // blocking stream: ordered after the legacy default stream (safe default for torch/ggml callers)
    if (const char *e = getenv("TMAC_B200_LUT_MODE")) g.lut_mode = atoi(e);
    if (const char *e = getenv("TMAC_B200_PDL")) g.use_pdl = atoi(e);
    if (const char *e = getenv("TMAC_B200_TRACE")) g.trace = atoi(e);
    if (const char *e = getenv("TMAC_B200_CS")) g.cs_override = atoi(e);
    if (const char *e = getenv("TMAC_B200_PDL_LATE")) g.pdl_late = atoi(e);
    if (const char *e = getenv("TMAC_B200_MINB")) g.minb_override = atoi(e);
    if (const char *e = getenv("TMAC_B200_FUSED")) g.use_fused = atoi(e);
    if (const char *e = getenv("TMAC_B200_PREFILL")) g.use_prefill = atoi(e);
    if (const char *e = getenv("TMAC_B200_PREFILL16")) g.use_prefill16 = atoi(e);
    if (const char *e = getenv("TMAC_B200_PREFILL_MIN_N")) g.prefill_min_n = atoi(e);
    if (const char *e = getenv("TMAC_B200_WPC")) g.wpc_override = atoi(e);
    if (const char *e = getenv("TMAC_B200_NBUF")) g.nbuf_override = atoi(e);
    g.inited = true;
    return 0;
}

// ---- kernel dispatch ---------------------------------------------------------------------
typedef void (*gemv3_fn)(const Gemv3Params, const uint32_t, const uint32_t);
template <int PB, bool SYM, int MINB> gemv3_fn pick3_qa(int qch, int agq) {
    switch (qch * 16 + agq) {
        case 8 * 16 + 8: return gemv3_kernel<PB, SYM, 8, 8, MINB>;
        case 8 * 16 + 4: return gemv3_kernel<PB, SYM, 8, 4, MINB>;
        case 8 * 16 + 2: return gemv3_kernel<PB, SYM, 8, 2, MINB>;
        case 8 * 16 + 0: return gemv3_kernel<PB, SYM, 8, 0, MINB>;
        case 4 * 16 + 4: return gemv3_kernel<PB, SYM, 4, 4, MINB>;
        case 4 * 16 + 2: return gemv3_kernel<PB, SYM, 4, 2, MINB>;
        case 4 * 16 + 0: return gemv3_kernel<PB, SYM, 4, 0, MINB>;
        case 2 * 16 + 2: return gemv3_kernel<PB, SYM, 2, 2, MINB>;
        case 2 * 16 + 0: return gemv3_kernel<PB, SYM, 2, 0, MINB>;
    }
    return nullptr;
}
template <int MINB> gemv3_fn pick_gemv3_m(int pb, bool sym, int qch, int agq) {
    if (pb == 4) return sym ? pick3_qa<4, true, MINB>(qch, agq) : pick3_qa<4, false, MINB>(qch, agq);
    if (pb == 2) return sym ? pick3_qa<2, true, MINB>(qch, agq) : pick3_qa<2, false, MINB>(qch, agq);
    if (pb == 1) return sym ? pick3_qa<1, true, MINB>(qch, agq) : pick3_qa<1, false, MINB>(qch, agq);
    return nullptr;
}
gemv3_fn pick_gemv3(int pb, bool sym, int qch, int agq, int minb) {
    return minb == 3 ? pick_gemv3_m<3>(pb, sym, qch, agq) : pick_gemv3_m<4>(pb, sym, qch, agq);
}
// fused-LUT instantiations (symmetric by construction, activation group inside the chunk)
template <int PB, int MINB> gemv3_fn pick3_fused_qa(int qch, int agq) {
    switch (qch * 16 + agq) {
        case 8 * 16 + 8: return gemv3_kernel<PB, true, 8, 8, MINB, true>;
        case 8 * 16 + 4: return gemv3_kernel<PB, true, 8, 4, MINB, true>;
        case 8 * 16 + 2: return gemv3_kernel<PB, true, 8, 2, MINB, true>;
        case 8 * 16 + 0: return gemv3_kernel<PB, true, 8, 0, MINB, true>;     // integer path (one activation group = K)
        case 4 * 16 + 4: return gemv3_kernel<PB, true, 4, 4, MINB, true>;
        case 4 * 16 + 2: return gemv3_kernel<PB, true, 4, 2, MINB, true>;
        case 4 * 16 + 0: return gemv3_kernel<PB, true, 4, 0, MINB, true>;
        case 2 * 16 + 2: return gemv3_kernel<PB, true, 2, 2, MINB, true>;
        case 2 * 16 + 0: return gemv3_kernel<PB, true, 2, 0, MINB, true>;
    }
    return nullptr;
}
template <int MINB> gemv3_fn pick_fused_m(int pb, int qch, int agq) {
    if (pb == 4) return pick3_fused_qa<4, MINB>(qch, agq);
    if (pb == 2) return pick3_fused_qa<2, MINB>(qch, agq);
    if (pb == 1) return pick3_fused_qa<1, MINB>(qch, agq);
    return nullptr;
}
gemv3_fn pick_gemv3_fused(int pb, int qch, int agq, int minb) {
    return minb == 3 ? pick_fused_m<3>(pb, qch, agq) : pick_fused_m<4>(pb, qch, agq);
}

int ilog2(int v) { int s = 0; while ((1 << (s + 1)) <= v) ++s; return s; }

// Decomposition of one launch: cluster size CS (K slices of a super-block), warps per CTA, chunks
// per warp.  Minimises the work of the busiest SM (CTAs are spread round-robin over SMs), then
// prefers more warps in flight.
void choose_decomposition(int nrsb, int nchunk, int N, int *cs_out, int *wpc_out, int *bpw_out) {
    double best_cost = 1e30; int bcs = 1, bwpc = 1, bbpw = nchunk;
    for (int cs : {1, 2, 4, 8})
        for (int wpc = 1; wpc <= kG3MaxWarps; ++wpc) {
            if (cs * wpc > nchunk && !(cs == 1 && wpc == 1)) { if (cs * (wpc - 1) >= nchunk) continue; }
            const int bpw = (nchunk + cs * wpc - 1) / (cs * wpc);
            if ((cs - 1) * wpc * bpw >= nchunk) continue;              // an entirely idle CTA
            const long ctas = (long)nrsb * cs * N;
            const int res = std::max(1, std::min(32, 2048 / (wpc * 32)));   // resident CTAs per SM (threads)
            const long per_sm = (ctas + g.sms - 1) / g.sms;
            const long waves = (per_sm + res - 1) / res;
            double cost = (double)per_sm * wpc * bpw;                  // chunk-slots on the busiest SM
            cost *= 1.0 + 0.15 * (waves - 1);                          // later waves lose the overlap
            cost += 0.02 * bpw * wpc + 0.2 * bpw;                      // prefer short per-warp chains ...
            cost += 0.5 * std::max(0L, 8 - per_sm * wpc);              // ... and at least 8 warps per SM
            if (cost < best_cost) { best_cost = cost; bcs = cs; bwpc = wpc; bbpw = bpw; }
        }
    *cs_out = bcs; *wpc_out = bwpc; *bpw_out = bbpw;
}

// Production launch: clusters + DSMEM reduction + PDL (gemv3_kernel).
struct BatchPtrs { int n = 0; const unsigned char *const *W = nullptr; const int8_t *const *q = nullptr; const float *const *ls = nullptr,
                   *const *lb = nullptr; void *const *C = nullptr; };

int launch_gemv3(const Resident &R, int row_begin, int row_end, int N, const int8_t *qlut, const float *ls, const float *lb, void *C,
                 int ldc, int c_row0, int out_f16, bool sym, const BatchPtrs *batch = nullptr, const void *fused_act = nullptr,
                 int act_f16 = 0) {
    const StreamLayout &L = R.L;
    if (row_begin < 0 || row_end > L.Mout || row_begin >= row_end) return fail("qgemm_lut: bad row range");
    const int rsb0 = row_begin / L.rsb, rsb1 = (row_end + L.rsb - 1) / L.rsb, nrsb = rsb1 - rsb0;
    const bool int_path = L.one_scale && L.act_group_size == L.K;
    Gemv3Params p{};
    p.W = R.d + (size_t)rsb0 * L.rsb_stride;
    p.Wnext = nullptr;
    if (g.next_hint) {
        auto it = g.res.find(g.next_hint);
        if (it != g.res.end() && it->second.L.total == L.total && it->second.L.blk == L.blk) p.Wnext = it->second.d + (size_t)rsb0 * L.rsb_stride;
        g.next_hint = 0;
    }
    p.qlut = qlut; p.lut_scales = ls; p.lut_biases = lb; p.C = C;
    p.K = L.K; p.ldc = ldc; p.row_begin = row_begin; p.row_end = row_end; p.c_row0 = c_row0; p.bits = L.bits;
    p.nrsb = nrsb; p.rsb0 = rsb0; p.nchunk = L.nchunk;
    p.ags = L.act_group_size;
    const int agq = int_path ? 0 : std::min(L.act_group_size, L.ck) / 16;
    p.zp = L.zp; p.one_scale = L.one_scale; p.sd = L.sd; p.out_f16 = out_f16;
    p.blk_bytes = (int)L.blk; p.scale0 = L.scale0; p.rsb_stride = L.rsb_stride;
    if (g.npeer) {
        if (N != 1 || batch) { g.npeer = 0; return fail("peer outputs: N = 1, single-tensor launches only"); }
        p.npeer = g.npeer;
        for (int q = 0; q < g.npeer; ++q) p.Cpeer[q] = g.peer_out[q];
        g.npeer = 0;
    }
    p.pdl_late = (g.pdl_late >= 0) ? g.pdl_late : (fused_act ? 0 : 1);   // measured: fused launches prefer the early trigger
    const int nb = batch ? batch->n : 0;
    if (batch) { p.nbatch = nb; p.Wv = batch->W; p.qlutv = batch->q; p.lsv = batch->ls; p.lbv = batch->lb; p.Cv = batch->C; }
    choose_decomposition(nrsb, L.nchunk, N * std::max(1, nb), &p.cs, &p.wpc, &p.bpw);
    // Measured on B200 (profiles/): a lone launch per tensor is latency bound and prefers fewer, fatter
    // CTAs with more registers (ILP); grouped / batched launches are ALU-pipe bound and prefer more CTAs.
    const bool lone = (N * std::max(1, nb) == 1);
    // 85-register variant (more ILP) for lone launches and for grouped W1/W2 launches (shared memory caps residency at 3
    // CTAs per SM anyway; measured +6 %); grouped W3/W4 launches measured better with the 64-register variant.
    int minb = (lone || L.pb != 4) ? 3 : 4;
    if (lone && p.cs == 8 && p.wpc == 4 && p.bpw == 1) { p.cs = 4; p.wpc = 8; }
    if (!lone && (long)nrsb * N * std::max(1, nb) >= 4L * g.sms) {   // machine already full of whole super-blocks: no K split
        p.cs = 1; p.wpc = std::min(kG3MaxWarps, L.nchunk); p.bpw = (L.nchunk + p.wpc - 1) / p.wpc;
    }
    if (g.minb_override > 0) minb = g.minb_override;
    if (g.cs_override > 0) { p.cs = g.cs_override; }
    if (g.wpc_override > 0) { p.wpc = std::min(g.wpc_override, kG3MaxWarps); }
    if (g.cs_override > 0 || g.wpc_override > 0) p.bpw = (L.nchunk + p.cs * p.wpc - 1) / (p.cs * p.wpc);
    g.last_launch[0] = p.cs; g.last_launch[1] = p.wpc; g.last_launch[2] = p.bpw; g.last_launch[3] = minb;
    g.last_launch[4] = nrsb * p.cs; g.last_launch[5] = L.pb; g.last_launch[6] = sym ? 1 : 0; g.last_launch[7] = std::max(1, nb);
    if (g.trace) {   // ring of 8 launches
        const size_t per = (size_t)nrsb * p.cs * 8;
        if (g.d_trace.ensure(per * 8 * sizeof(long long))) return fail("out of device memory (trace)");
        p.trace = (long long *)g.d_trace.p + per * (size_t)(g.trace_seq++ % 8);
        g.trace_ctas = nrsb * p.cs;
    }
    if (fused_act) { p.act = fused_act; p.act_f16 = act_f16; sym = true; }
    gemv3_fn fn = fused_act ? pick_gemv3_fused(L.pb, L.qch, agq, minb) : pick_gemv3(L.pb, sym, L.qch, agq, minb);
    if (!fn) return fail("qgemm_lut: unsupported chunking (qch=" + std::to_string(L.qch) + ", agq=" + std::to_string(agq) + ")");
    p.nbuf = (p.bpw > 1) ? 2 : 1;
    if (g.nbuf_override > 0) p.nbuf = std::min(p.nbuf, g.nbuf_override);
    const size_t wregion = std::max((size_t)p.wpc * (p.nbuf * L.blk + (size_t)L.qch * 4 * (sym ? 8 : 16)), (size_t)p.wpc * L.rsb * 4);
    size_t smem = (size_t)p.cs * L.rsb * 4 + ((wregion + 15) & ~(size_t)15) + (size_t)p.wpc * 16;   // + warp-private mbarriers
    if (fused_act && int_path) { p.ioff = (int)smem; smem += (size_t)(L.K / 32 + kG3MaxWarps + 4 + 8) * 4; }   // row scan: block sums, warp maxima, bias, cluster maxima
    if (smem > 48 * 1024) CUDA_OK(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint32_t wtx, wty;
    plane_weight_regs(L.bits, sym, &wtx, &wty);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(nrsb * p.cs, N, std::max(1, nb));
    cfg.blockDim = dim3(p.wpc * 32, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = g.stream();
    cudaLaunchAttribute attr[2];
    int na = 0;
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
    ++na;
    if (p.cs > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = p.cs; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        ++na;
    }
    cfg.attrs = attr; cfg.numAttrs = na;
    CUDA_OK(cudaLaunchKernelEx(&cfg, fn, p, wtx, wty));
    return 0;
}

// Prefill tile on tcgen05 (tmac_prefill.cuh).  Returns 1 if the shape is not covered (caller falls back to the GEMV
// kernel per activation row), 0 on launch, -1 on error.
int launch_prefill(const Resident &R, int N, const int8_t *qlut, const float *ls, const float *lb, void *C, int ldc, int out_f16, bool sym) {
    const StreamLayout &L = R.L;
    if (!g.use_prefill || N < g.prefill_min_n || !sym) return 1;
    if (L.pb != 2 || L.qch != 8 || L.act_group_size != 64 || L.one_scale || L.ck != 128) return 1;
    const size_t rawsz = (L.blk + 127) & ~(size_t)127;
    if (g.use_prefill16 && N >= 64) {   // fp path: scales folded into fp16 operands, fp32 accumulation over K in TMEM (tmac_prefill16.cuh)
        const int nmain = L.K / 64, nextra = (L.nchunk + 31) / 32, ntile16 = (N + kP16NT - 1) / kP16NT;
        const size_t smem16 = (size_t)kP16NA * kP16SubA + (size_t)kP16NB * kP16SubB + 2 * rawsz + (2 * kP16NA + 2 * kP16NB + 2) * 8 + 1024;
        if (smem16 <= 227 * 1024) {
            if (g.d_tiles.ensure((size_t)ntile16 * (nmain + nextra) * kP16BBytes)) return fail("out of device memory (LUT tiles)");
            if (g.d_pf_texp.ensure((size_t)N * sizeof(int))) return fail("out of device memory (token exponents)");
            {   // programmatic dependent launches: the exponent scan starts under the preprocessor's tail, the tiling kernel loads its
                // LUT entries while the exponents are being computed (each waits on griddepcontrol before it reads its inputs)
                cudaLaunchConfig_t lc{};
                lc.blockDim = dim3(256); lc.stream = g.stream();
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                at[0].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
                lc.attrs = at; lc.numAttrs = 1;
                lc.gridDim = dim3((N + 7) / 8);
                CUDA_OK(cudaLaunchKernelEx(&lc, p16_token_exp_kernel, ls, lb, (int *)g.d_pf_texp.p, N, nmain));
                lc.gridDim = dim3(nmain + nextra, ntile16);
                CUDA_OK(cudaLaunchKernelEx(&lc, lut_tile16_kernel, qlut, ls, lb, (const int *)g.d_pf_texp.p, (unsigned char *)g.d_tiles.p,
                                           N, (int)L.K, nmain, nextra));
            }
            Prefill16Params q{};
            q.W = R.d; q.C = C; q.N = N; q.K = L.K; q.Mout = L.Mout; q.ldc = ldc; q.out_f16 = out_f16;
            q.nchunk = L.nchunk; q.zp = L.zp; q.sd = L.sd; q.blk_bytes = (int)L.blk; q.nmain = nmain; q.nextra = nextra;
            q.rsb_stride = L.rsb_stride; q.tiles = (const unsigned char *)g.d_tiles.p;
            q.nrsb = L.nrsb; q.ntiles = L.nrsb * ntile16;
            q.texp = (const int *)g.d_pf_texp.p; q.rexp = reinterpret_cast<const int *>(R.d + R.rexp_off);
            // fewer tiles than SMs (e.g. 86 at N = 256): stream-K over all SMs, partial tiles through `scratch`
            q.streamk = (g.pf_streamk && q.ntiles < g.sms && (long)q.ntiles * (nmain + nextra) >= 2L * g.sms) ? 1 : 0;
            const int grid = q.streamk ? g.sms : q.ntiles;
            if (q.streamk) {
                const size_t sb = (size_t)grid * kP16NT * 128 * sizeof(float);
                if (g.d_pf_scratch.ensure(sb)) return fail("out of device memory (stream-K scratch)");
                if (g.d_pf_flags.cap < (size_t)grid * sizeof(int)) {
                    if (g.d_pf_flags.ensure((size_t)grid * sizeof(int))) return fail("out of device memory (stream-K flags)");
                    CUDA_OK(cudaMemsetAsync(g.d_pf_flags.p, 0, g.d_pf_flags.cap, g.stream()));
                }
                q.scratch = (float *)g.d_pf_scratch.p; q.flags = (int *)g.d_pf_flags.p;
            }
            CUDA_OK(cudaFuncSetAttribute((const void *)prefill16_w2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16));
            prefill16_w2_kernel<<<dim3(grid), kP16Threads, smem16, g.stream()>>>(q);
            CUDA_OK(cudaGetLastError());
            g.last_launch[0] = 16; g.last_launch[1] = kP16Threads / 32; g.last_launch[2] = L.nchunk; g.last_launch[3] = q.streamk; g.last_launch[4] = grid;
            g.last_launch[5] = L.pb; g.last_launch[6] = 1; g.last_launch[7] = -N;
            return 0;
        }
    }
    const size_t smem = (size_t)kPfStages * (kPfStageBytes + kPfRec) + 2 * rawsz + 256 * 8 + (2 * kPfStages + 4) * 8 + 1024;
    if (smem > 225 * 1024) return 1;
    const int nag = L.K / 64, ntile = (N + kPfNT - 1) / kPfNT;
    if (g.d_tiles.ensure((size_t)ntile * nag * kPfRec)) return fail("out of device memory (LUT tiles)");
    lut_tile_kernel<<<dim3(nag, ntile), 128, 0, g.stream()>>>(qlut, ls, lb, (unsigned char *)g.d_tiles.p, N, L.K);
    CUDA_OK(cudaGetLastError());
    PrefillParams p{};
    p.W = R.d; p.qlut = qlut; p.lut_scales = ls; p.lut_biases = lb; p.C = C;
    p.lut_tiles = (const unsigned char *)g.d_tiles.p;
    p.N = N; p.K = L.K; p.Mout = L.Mout; p.ldc = ldc; p.out_f16 = out_f16;
    p.nchunk = L.nchunk; p.zp = L.zp; p.sd = L.sd; p.blk_bytes = (int)L.blk; p.rsb_stride = L.rsb_stride;
    if (g.trace) {
        if (g.d_trace.ensure(8192)) return fail("out of device memory (trace)");
        CUDA_OK(cudaMemsetAsync(g.d_trace.p, 0, 3 * 32 * 4 * sizeof(long long), g.stream()));
        p.dbg = (long long *)g.d_trace.p; g.trace_ctas = 12;   // 96 rows of 4 = 48 rows of 8
    }
    CUDA_OK(cudaFuncSetAttribute((const void *)prefill_w2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(L.nrsb, ntile);
    prefill_w2_kernel<<<grid, kPfThreads2, smem, g.stream()>>>(p);
    CUDA_OK(cudaGetLastError());
    g.last_launch[0] = 1; g.last_launch[1] = kPfThreads2 / 32; g.last_launch[2] = L.nchunk; g.last_launch[3] = 1; g.last_launch[4] = L.nrsb;
    g.last_launch[5] = L.pb; g.last_launch[6] = 1; g.last_launch[7] = -N;   // batch < 0 marks the tcgen05 prefill tile
    return 0;
}

// Launch qgemm_lut over rows [row_begin,row_end) (relative to the resident tensor): the tcgen05 tile for whole-tensor batches,
// else gemv3_kernel.  All pointers are device pointers; C is [N][ldc] with C[n][row - c_row0].
int launch_gemv(const Resident &R, int row_begin, int row_end, int N, const int8_t *qlut, const float *ls,
                const float *lb, void *C, int ldc, int c_row0, int out_f16, bool sym, int32_t *cbits_unused) {
    (void)cbits_unused;
    if (row_begin == 0 && row_end == R.L.Mout && c_row0 == 0 && ldc == R.L.Mout) {
        const int rc = launch_prefill(R, N, qlut, ls, lb, C, ldc, out_f16, sym);
        if (rc <= 0) return rc;
    }
    return launch_gemv3(R, row_begin, row_end, N, qlut, ls, lb, C, ldc, c_row0, out_f16, sym);
}

int launch_preprocessor(int K, int N, int ags, int dtype, const void *B, float *ls, float *lb, int8_t *qlut) {
    if (ags <= 0 || ags > K) ags = K;
    if (K % 32 || ags % 32 || K % ags) return fail("preprocessor: K and act_group_size must be multiples of 32, K % act_group_size == 0");
    const int nag = K / ags;
    int agb = (ags == K) ? 1 : std::max(1, 1024 / ags);
    const int gx = (nag + agb - 1) / agb;
    const int ng = agb * (ags / 4);
    const size_t smem = (size_t)agb * 4 + (size_t)ng * 4 + (size_t)(ng / 8 + 1) * 4;
    if (smem > 200 * 1024) return fail("preprocessor: activation group too large");
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(gx, N, 1);
    cfg.blockDim = dim3(kPreThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = g.stream();
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (dtype == TMAC_B200_F16) {
        if (smem > 48 * 1024) CUDA_OK(cudaFuncSetAttribute((const void *)preprocessor_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_OK(cudaLaunchKernelEx(&cfg, preprocessor_kernel<__half>, (const __half *)B, ls, lb, qlut, K, ags, agb));
    } else {
        if (smem > 48 * 1024) CUDA_OK(cudaFuncSetAttribute((const void *)preprocessor_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_OK(cudaLaunchKernelEx(&cfg, preprocessor_kernel<float>, (const float *)B, ls, lb, qlut, K, ags, agb));
    }
    CUDA_OK(cudaGetLastError());
    if (g.sym_qluts.size() > 4096) g.sym_qluts.clear();
    g.sym_qluts.insert(qlut);
    return 0;
}

bool host_lut_symmetric(const int8_t *q, size_t groups) {
    for (size_t g2 = 0; g2 < groups; ++g2) {
        const int8_t *t = q + g2 * 16;
        for (int i = 0; i < 8; ++i)
            if ((int)t[15 - i] != -(int)t[i]) return false;
    }
    return true;
}

int validate_cfg(const tmac_b200_kcfg &c) {
    if (c.bits < 1 || c.bits > 4) return fail("kcfg: bits must be 1..4");
    if (c.M <= 0 || c.K <= 0 || c.K % 32) return fail("kcfg: bad M/K");
    if (c.bm <= 0 || (c.M * c.bits) % c.bm || c.bm % 32 || c.bm % c.bits) return fail("kcfg: bm must divide M*bits and be a multiple of 32 and of bits");
    if (c.kfactor <= 0 || (c.K / 4) % c.kfactor) return fail("kcfg: kfactor must divide K/4");
    if (c.simd_n_in != 16 || c.simd_n_out != 8) return fail("kcfg: only simd_n_in=16, simd_n_out=8 (the reference's only instantiation)");
    if (!c.one_scale && (c.group_size <= 0 || c.K % c.group_size || c.group_size % 32)) return fail("kcfg: group_size must be a positive multiple of 32 that divides K");
    return 0;
}

int64_t register_resident(const tmac_b200_kcfg &cfg, const PlainWeights &P, const void *host_alias, size_t alias_bytes, int row0) {
    StreamLayout L;
    bool fp16_ok = true;
    if (!cfg.one_scale) {
        fp16_ok = all_fp16_exact(P.scales.data(), P.scales.size()) && (P.zeros.empty() || all_fp16_exact(P.zeros.data(), P.zeros.size()));
        if (getenv("TMAC_B200_SCALES_F32")) fp16_ok = false;
    }
    if (!make_layout(P.Mout, cfg.K, cfg.bits, cfg.group_size, cfg.act_group_size, cfg.zero_point, cfg.one_scale, fp16_ok ? 2 : 4, &L))
        return fail("unsupported shape / grouping for the stream layout");
    if (cfg.one_scale) L.scale0 = P.scales.empty() ? 0.f : P.scales[0];
    Resident R;
    R.rexp_off = (L.total + 15) & ~(size_t)15;
    R.alloc = R.rexp_off + (size_t)L.nrsb * L.rsb * sizeof(int);
    std::vector<uint8_t> host(R.alloc, 0);
    encode_stream(P, L, host.data());
    if (!cfg.one_scale) {                // per-row exponents of the fp16 prefill tile (tmac_prefill16.cuh, p16_exp); padding rows 0
        const int ng = cfg.K / cfg.group_size;
        int *rexp = reinterpret_cast<int *>(host.data() + R.rexp_off);
        for (int r = 0; r < P.Mout; ++r)
            rexp[r] = p16_row_exp(P.scales.data() + (size_t)r * ng, P.zeros.empty() ? nullptr : P.zeros.data() + (size_t)r * ng, ng);
    }
    R.cfg = cfg; R.L = L; R.row0 = row0;
    if (cudaMalloc((void **)&R.d, R.alloc) != cudaSuccess) { cudaGetLastError(); return fail("out of device memory for resident weights"); }
    if (cudaMemcpy(R.d, host.data(), R.alloc, cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(R.d); return fail("weight upload failed"); }
    R.host_a = (const unsigned char *)host_alias;
    R.host_a_bytes = alias_bytes;
    const int64_t h = g.next_handle++;
    R.id = h;
    g.res[h] = R;
    return h;
}

Resident *find_by_alias(const void *A, size_t *offset) {
    const unsigned char *a = (const unsigned char *)A;
    for (auto &kv : g.res) {
        Resident &R = kv.second;
        if (R.host_a && a >= R.host_a && a < R.host_a + R.host_a_bytes) { *offset = (size_t)(a - R.host_a); return &R; }
        if (a == R.d) { *offset = 0; return &R; }
    }
    return nullptr;
}

const tmac_b200_kcfg *find_kcfg_locked(int m_times_bits, int k, int bits) {
    const tmac_b200_kcfg *tile_match = nullptr;
    for (const auto &c : g.kcfgs) {
        if (c.K != k || c.bits != bits) continue;
        if (c.M * c.bits == m_times_bits) return &c;
        if (m_times_bits % c.bm == 0 && m_times_bits < c.M * c.bits && !tile_match) tile_match = &c;
    }
    return tile_match;
}

// Stage helpers for host pointers ---------------------------------------------------------
// h_in is written by the host at call time and read by an async H2D: before reusing it wait for
// the previous call's copy; after enqueuing this call's copies record the event again.
void stage_wait() {
    if (g.stage_pending) { cudaEventSynchronize(g.stage_ev); g.stage_pending = false; }
}
void stage_mark() {
    if (!g.stage_ev) cudaEventCreateWithFlags(&g.stage_ev, cudaEventDisableTiming);
    cudaEventRecord(g.stage_ev, g.stream());
    g.stage_pending = true;
}
int h2d(DevBuf &dst, PinBuf &pin, size_t pin_off, const void *src, size_t bytes) {
    if (dst.ensure(bytes)) return fail("out of device memory");
    std::memcpy((char *)pin.p + pin_off, src, bytes);
    CUDA_OK(cudaMemcpyAsync(dst.p, (char *)pin.p + pin_off, bytes, cudaMemcpyHostToDevice, g.stream()));
    return 0;
}

size_t esize(int dtype) { return dtype == TMAC_B200_F16 ? 2 : 4; }

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int tmac_b200_init(int device) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (!g.inited && device >= 0) {
        if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail("cudaSetDevice failed"); }
    }
    return ensure_init();
}

void tmac_b200_shutdown(void) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (!g.inited) return;
    cudaStreamSynchronize(g.stream());
    for (auto &kv : g_seqs) kv.second.release();
    g_seqs.clear();
    for (auto &kv : g_graphs) cudaGraphExecDestroy(kv.second);
    g_graphs.clear();
    for (auto &e : g.ptr_tables) if (e.second) cudaFree(e.second);
    g.ptr_tables.clear();
    for (auto &kv : g_gguf) delete kv.second;
    g_gguf.clear();
    for (auto &kv : g.res) {
        cudaFree(kv.second.d);
        if (kv.second.reserved) munmap(kv.second.reserved, kv.second.reserved_bytes);
        std::free(kv.second.host_scales);
    }
    g.res.clear();
    for (DevBuf *b : {&g.d_b, &g.d_qlut, &g.d_ls, &g.d_lb, &g.d_c, &g.d_cbits, &g.d_trace, &g.d_tiles, &g.d_pf_scratch, &g.d_pf_flags, &g.d_pf_texp}) { if (b->p) cudaFree(b->p); b->p = nullptr; b->cap = 0; }
    for (HostLut &e : g.hluts) {
        for (DevBuf *b : {&e.dq, &e.dls, &e.dlb}) { if (b->p) cudaFree(b->p); b->p = nullptr; b->cap = 0; }
        if (e.res.p) cudaFreeHost(e.res.p);
        e = HostLut();
    }
    for (PinBuf *b : {&g.h_in, &g.h_out}) { if (b->p) cudaFreeHost(b->p); b->p = nullptr; b->cap = 0; }
    if (g.stage_ev) cudaEventDestroy(g.stage_ev);
    g.stage_ev = nullptr; g.stage_pending = false;
    if (g.own) cudaStreamDestroy(g.own);
    g.own = nullptr; g.sym_qluts.clear();
    g.user = nullptr; g.use_user = false; g.trace_ctas = 0; g.trace_seq = 0; g.next_hint = 0;
    g.inited = false;
}

const char *tmac_b200_last_error(void) { return t_err.c_str(); }
int tmac_b200_version(void) { return 100; }

int tmac_b200_set_stream(void *stream) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    g.user = (cudaStream_t)stream;
    g.use_user = stream != nullptr;
    return 0;
}

int tmac_b200_set_float_type(int dtype) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (dtype != TMAC_B200_F32 && dtype != TMAC_B200_F16) return fail("bad dtype");
    g.float_type = dtype;
    return 0;
}

int tmac_b200_register_kcfg(const tmac_b200_kcfg *cfg) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (!cfg) return fail("null kcfg");
    tmac_b200_kcfg c = *cfg;
    if (c.simd_n_in == 0) c.simd_n_in = 16;
    if (c.simd_n_out == 0) c.simd_n_out = 8;
    if (c.act_group_size <= 0 || c.act_group_size > c.K) c.act_group_size = c.K;
    if (validate_cfg(c)) return -1;
    for (auto &o : g.kcfgs)
        if (o.M == c.M && o.K == c.K && o.bits == c.bits) { o = c; return 0; }
    g.kcfgs.push_back(c);
    return 0;
}

void tmac_b200_clear_kcfg(void) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    g.kcfgs.clear();
}

int tmac_b200_find_kcfg(int m_times_bits, int k, int bits, tmac_b200_kcfg *out) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    const tmac_b200_kcfg *c = find_kcfg_locked(m_times_bits, k, bits);
    if (!c) return fail("no kcfg for m=" + std::to_string(m_times_bits) + " k=" + std::to_string(k) + " b=" + std::to_string(bits));
    if (out) *out = *c;
    return 0;
}

// Minimal INI reader for the reference's kcfg.ini (deploy/compile.py:156-165,203-204).
int tmac_b200_load_kcfg_file(const char *path) {
    FILE *f = path ? fopen(path, "r") : nullptr;
    if (!f) return fail(std::string("cannot open kcfg file ") + (path ? path : "(null)"));
    struct Sec { std::string name; std::map<std::string, long> kv; };
    std::vector<Sec> secs;
    char line[512];
    while (fgets(line, sizeof line, f)) {
        std::string s(line);
        size_t a = s.find_first_not_of(" \t\r\n");
        if (a == std::string::npos || s[a] == ';' || s[a] == '#') continue;
        size_t b = s.find_last_not_of(" \t\r\n");
        s = s.substr(a, b - a + 1);
        if (s.front() == '[' && s.back() == ']') { secs.push_back({s.substr(1, s.size() - 2), {}}); continue; }
        size_t eq = s.find('=');
        if (eq == std::string::npos || secs.empty()) continue;
        std::string k = s.substr(0, eq), v = s.substr(eq + 1);
        k.erase(k.find_last_not_of(" \t") + 1);
        v.erase(0, v.find_first_not_of(" \t"));
        secs.back().kv[k] = atol(v.c_str());
    }
    fclose(f);
    int count = 0;
    for (auto &s : secs) {
        int t, m, k, n, b;
        if (sscanf(s.name.c_str(), "qgemm_lut_t%d_int8_m%d_k%d_n%d_b%d", &t, &m, &k, &n, &b) != 5) continue;
        if (b < 1 || b > 4) continue;                    // not a section this library can serve (and m / b below)
        auto get = [&](const char *key, long dflt) { auto it = s.kv.find(key); return it == s.kv.end() ? dflt : it->second; };
        tmac_b200_kcfg c{};
        c.M = m / b; c.K = k; c.bits = b;
        c.bm = (int)get("bm", 0); c.kfactor = (int)get("kfactor", 16);
        c.simd_n_in = (int)get("simd_n_in", 16); c.simd_n_out = (int)get("simd_n_out", 8);
        c.group_size = (int)get("group_size", 128);
        const long lss = get("lut_scales_size", 0), ss = get("scales_size", 0);
        c.act_group_size = (int)get("act_group_size", lss > 0 ? (long)k * n / lss : 64);
        const long per_group = (long)c.M * (k / std::max(1, c.group_size));
        c.one_scale = (int)get("m_groups", ss > 0 && ss < c.M ? 1 : -1) > 0 ? 1 : 0;
        c.zero_point = (int)get("zero_point", (!c.one_scale && ss == 2 * per_group) ? 1 : 0);
        if (tmac_b200_register_kcfg(&c) == 0) ++count;
    }
    return count;
}

int64_t tmac_b200_upload_weights(const tmac_b200_kcfg *cfg_in, const void *A, const void *scales, int scales_dtype) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (!cfg_in || !A || !scales) return fail("upload_weights: null argument");
    if (is_device_ptr(A)) return fail("upload_weights: A must be a host pointer (reference layout)");
    tmac_b200_kcfg cfg = *cfg_in;
    if (cfg.simd_n_in == 0) cfg.simd_n_in = 16;
    if (cfg.simd_n_out == 0) cfg.simd_n_out = 8;
    if (cfg.act_group_size <= 0 || cfg.act_group_size > cfg.K) cfg.act_group_size = cfg.K;
    if (validate_cfg(cfg)) return -1;
    const size_t nsc = cfg.one_scale ? 1 : (size_t)cfg.M * (cfg.K / cfg.group_size) * (cfg.zero_point ? 2 : 1);
    std::vector<float> s32(nsc);
    if (scales_dtype == TMAC_B200_F16) {
        const uint16_t *h = (const uint16_t *)scales;
        for (size_t i = 0; i < nsc; ++i) s32[i] = f16_bits_to_f32(h[i]);
    } else
        std::memcpy(s32.data(), scales, nsc * 4);
    PlainWeights P;
    plain_from_reference((const uint8_t *)A, s32.data(), cfg.M, cfg.K, cfg.bits, cfg.bm, cfg.kfactor, cfg.group_size,
                         cfg.zero_point, cfg.one_scale, &P);
    return register_resident(cfg, P, A, (size_t)cfg.M * cfg.K * cfg.bits / 8, 0);
}

int64_t tmac_b200_upload_plain_rows(const tmac_b200_kcfg *cfg_in, const uint8_t *w, const float *scales, const float *zeros,
                                    int row0, int rows) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (!cfg_in || !w || !scales) return fail("upload_plain: null argument");
    tmac_b200_kcfg cfg = *cfg_in;
    if (cfg.simd_n_in == 0) cfg.simd_n_in = 16;
    if (cfg.simd_n_out == 0) cfg.simd_n_out = 8;
    if (cfg.act_group_size <= 0 || cfg.act_group_size > cfg.K) cfg.act_group_size = cfg.K;
    if (cfg.bits < 1 || cfg.bits > 4 || cfg.M <= 0 || cfg.K <= 0 || cfg.K % 32) return fail("upload_plain: bad shape");
    if (!cfg.one_scale && (cfg.group_size <= 0 || cfg.K % cfg.group_size || cfg.group_size % 32)) return fail("upload_plain: group_size must be a positive multiple of 32 that divides K");
    if (row0 < 0 || rows <= 0 || row0 + rows > cfg.M) return fail("upload_plain: bad row range");
    if (cfg.zero_point && !zeros && !cfg.one_scale) return fail("upload_plain: zero_point set but zeros == NULL");
    PlainWeights P;
    plain_from_w(w, cfg.M, cfg.K, cfg.bits, row0, rows, &P);
    if (cfg.one_scale) P.scales.assign(1, scales[0]);
    else {
        const int NG = cfg.K / cfg.group_size;
        P.scales.assign(scales + (size_t)row0 * NG, scales + (size_t)(row0 + rows) * NG);
        if (cfg.zero_point) P.zeros.assign(zeros + (size_t)row0 * NG, zeros + (size_t)(row0 + rows) * NG);
    }
    return register_resident(cfg, P, nullptr, 0, row0);
}

int64_t tmac_b200_upload_plain(const tmac_b200_kcfg *cfg, const uint8_t *w, const float *scales, const float *zeros) {
    if (!cfg) return fail("upload_plain: null kcfg");
    return tmac_b200_upload_plain_rows(cfg, w, scales, zeros, 0, cfg->M);
}

// GPTQ checkpoint tensors (safetensors: qweight, scales, qzeros) -> resident weights, the C form of
// unpack_gptqv2 + preprocess_weights + upload (model_utils.py:95-129, :262-271; convert_hf_to_gguf.py:300-320).
// cfg gives M, K, bits, group_size, bm, kfactor, act_group_size; zero_point is implied.
int64_t tmac_b200_upload_gptq(const tmac_b200_kcfg *cfg_in, const int32_t *qweight, const uint16_t *scales_f16, const int32_t *qzeros,
                              int gptq_v2) {
    if (!cfg_in || !qweight || !scales_f16 || !qzeros) return fail("upload_gptq: null argument");
    tmac_b200_kcfg cfg = *cfg_in;
    cfg.zero_point = 1; cfg.one_scale = 0;
    if (cfg.group_size <= 0 || cfg.K % cfg.group_size) return fail("upload_gptq: bad group_size");
    const size_t NG = (size_t)cfg.K / cfg.group_size;
    std::vector<uint8_t> w((size_t)cfg.M * cfg.K);
    std::vector<float> sc((size_t)cfg.M * NG), zr((size_t)cfg.M * NG);
    if (!unpack_gptq(qweight, scales_f16, qzeros, cfg.K, cfg.M, cfg.bits, cfg.group_size, gptq_v2 != 0, w.data(), sc.data(), zr.data()))
        return fail("upload_gptq: unsupported packing (bits must divide 32; K, M multiples of 32/bits)");
    return tmac_b200_upload_plain(&cfg, w.data(), sc.data(), zr.data());
}
// Host-only: the unpack step alone (CPU suite).  w [M][K], scales / zeros [M][K/group_size].
int tmac_b200_debug_unpack_gptq(const int32_t *qweight, const uint16_t *scales_f16, const int32_t *qzeros, int K, int M, int bits,
                                int group_size, int gptq_v2, uint8_t *w, float *scales, float *zeros) {
    if (!qweight || !scales_f16 || !qzeros || !w || !scales || !zeros) return fail("debug_unpack_gptq: null argument");
    if (!unpack_gptq(qweight, scales_f16, qzeros, K, M, bits, group_size, gptq_v2 != 0, w, scales, zeros)) return fail("debug_unpack_gptq: unsupported packing");
    return 0;
}

// Host-only converter-side quantisers (tmac_layout.h): fp weights -> codes + scales (+ zeros) in the T-MAC convention, ready for
// tmac_b200_upload_plain.  0 or -1.
int tmac_b200_quantize_bitdistiller(const float *w, int rows, int cols, int bits, int group_size, uint8_t *codes, float *scales, float *zeros) {
    if (!w || !codes || !scales || !zeros) return fail("quantize_bitdistiller: null argument");
    if (!quantize_bitdistiller(w, rows, cols, bits, group_size, codes, scales, zeros)) return fail("quantize_bitdistiller: bad shape / bits / group size");
    return 0;
}
int tmac_b200_quantize_bitnet(const float *w, int rows, int cols, uint8_t *codes, float *scale) {
    if (!w || !codes || !scale || rows <= 0 || cols <= 0) return fail("quantize_bitnet: bad argument");
    quantize_bitnet(w, (size_t)rows * cols, codes, scale);
    return 0;
}

// Host-only: run the reference-layout -> stream-layout transform without touching the GPU and
// return the stream bytes (used by the CPU test-suite to pin the layout).  dst may be NULL to
// query the size.  Returns the byte count or -1.
int64_t tmac_b200_debug_encode(const tmac_b200_kcfg *cfg_in, const void *A, const void *scales, void *dst, size_t cap,
                               int *layout_out /* int[12] */) {
    if (!cfg_in || !A || !scales) return fail("debug_encode: null argument");
    tmac_b200_kcfg cfg = *cfg_in;
    if (cfg.simd_n_in == 0) cfg.simd_n_in = 16;
    if (cfg.simd_n_out == 0) cfg.simd_n_out = 8;
    if (cfg.act_group_size <= 0 || cfg.act_group_size > cfg.K) cfg.act_group_size = cfg.K;
    if (validate_cfg(cfg)) return -1;
    PlainWeights P;
    plain_from_reference((const uint8_t *)A, (const float *)scales, cfg.M, cfg.K, cfg.bits, cfg.bm, cfg.kfactor, cfg.group_size,
                         cfg.zero_point, cfg.one_scale, &P);
    bool fp16_ok = true;
    if (!cfg.one_scale) fp16_ok = all_fp16_exact(P.scales.data(), P.scales.size()) && (P.zeros.empty() || all_fp16_exact(P.zeros.data(), P.zeros.size()));
    StreamLayout L;
    if (!make_layout(P.Mout, cfg.K, cfg.bits, cfg.group_size, cfg.act_group_size, cfg.zero_point, cfg.one_scale, fp16_ok ? 2 : 4, &L))
        return fail("unsupported shape / grouping for the stream layout");
    if (layout_out) {
        const int v[12] = {L.pb, L.rw, L.rsb, L.nrsb, L.ck, L.qch, L.nchunk, L.sd, L.zp, L.one_scale, (int)L.blk, (int)L.wbytes};
        std::memcpy(layout_out, v, sizeof v);
    }
    if (dst) {
        if (cap < L.total) return fail("debug_encode: destination too small");
        encode_stream(P, L, (uint8_t *)dst);
    }
    return (int64_t)L.total;
}

int tmac_b200_free_weights(int64_t handle) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g.res.find(handle);
    if (it == g.res.end()) return fail("bad handle");
    cudaStreamSynchronize(g.stream());
    for (HostLut &e : g.hluts) if (e.res_id == handle) e.res_id = 0;
    cudaFree(it->second.d);
    if (it->second.reserved) munmap(it->second.reserved, it->second.reserved_bytes);
    std::free(it->second.host_scales);
    g.res.erase(it);
    return 0;
}

size_t tmac_b200_weights_nbytes(int64_t handle) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g.res.find(handle);
    return it == g.res.end() ? 0 : it->second.L.total;
}

// Second resident copy of the same tensor in its own HBM allocation (benchmarks rotate through
// distinct buffers so that weights stream from HBM, not L2; multi-layer models with tied shapes).
int64_t tmac_b200_clone_weights(int64_t handle) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g.res.find(handle);
    if (it == g.res.end()) return fail("clone: bad handle");
    Resident R = it->second;
    R.host_a = nullptr; R.host_a_bytes = 0;
    R.reserved = nullptr; R.reserved_bytes = 0; R.host_scales = nullptr;   // owned by the original only (no double munmap / free)
    if (cudaMalloc((void **)&R.d, R.alloc) != cudaSuccess) { cudaGetLastError(); return fail("out of device memory for clone"); }
    if (cudaMemcpy(R.d, it->second.d, R.alloc, cudaMemcpyDeviceToDevice) != cudaSuccess) { cudaFree(R.d); return fail("clone copy failed"); }
    const int64_t h = g.next_handle++;
    R.id = h;
    g.res[h] = R;
    return h;
}

// ---- CUDA-graph helpers: capture a sequence of library calls (device pointers only; run the
// sequence once eagerly first so that every workspace is allocated) and replay it. -------------

int tmac_b200_graph_begin(void) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    CUDA_OK(cudaStreamBeginCapture(g.stream(), cudaStreamCaptureModeThreadLocal));
    return 0;
}
int64_t tmac_b200_graph_end(void) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    cudaGraph_t graph = nullptr;
    CUDA_OK(cudaStreamEndCapture(g.stream(), &graph));
    cudaGraphExec_t exec = nullptr;
    cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return fail(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
    const int64_t h = g_next_graph++;
    g_graphs[h] = exec;
    return h;
}
int tmac_b200_graph_launch(int64_t graph, int times) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_graphs.find(graph);
    if (it == g_graphs.end()) return fail("graph_launch: bad handle");
    for (int i = 0; i < times; ++i) CUDA_OK(cudaGraphLaunch(it->second, g.stream()));
    return 0;
}
int tmac_b200_graph_free(int64_t graph) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_graphs.find(graph);
    if (it == g_graphs.end()) return fail("graph_free: bad handle");
    cudaGraphExecDestroy(it->second);
    g_graphs.erase(it);
    return 0;
}
int tmac_b200_sync(void) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (!g.inited) return 0;
    CUDA_OK(cudaStreamSynchronize(g.stream()));
    return 0;
}

// Debug / reporting: {cluster size, warps per CTA, chunks per warp, min blocks variant, grid.x, PB, sym, batch}
// of the last qgemm_lut launch.
int tmac_b200_debug_last_launch(int *out8) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (!out8) return fail("null");
    std::memcpy(out8, g.last_launch, sizeof g.last_launch);
    return 0;
}

// One-shot hint: the tensor that will be multiplied next.  The next qgemm_lut launch prefetches its
// blocks into L2 (cp.async.bulk.prefetch.L2) while it computes, so that the HBM stream of launch
// i+1 overlaps launch i.  Ignored unless the tensor has the same stream geometry.
int tmac_b200_hint_next_weights(int64_t handle) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    g.next_hint = handle;
    return 0;
}

// Debug: per-CTA clock64 stamps of the last gemv3 launch ([ctas][8]); returns #ctas or -1.
int tmac_b200_debug_trace(long long *dst, int cap_ctas) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (!g.trace || !g.d_trace.p) return fail("trace disabled (TMAC_B200_TRACE=1)");
    CUDA_OK(cudaStreamSynchronize(g.stream()));
    const int n = std::min(cap_ctas, g.trace_ctas * 8);   // ring of 8 launches x ctas
    CUDA_OK(cudaMemcpy(dst, g.d_trace.p, (size_t)n * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    return g.trace_ctas;
}

// Tuning / A-B knobs at run time (same names as the TMAC_B200_* environment variables, lower case, without the prefix).
int tmac_b200_debug_set(const char *key, int value) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    const std::string k = key ? key : "";
    if (k == "seq_grid") g.seq_grid = value;
    else if (k == "seq_smem_kb") g.seq_smem_kb = value;
    else if (k == "seq_impl") g.seq_impl = value;
    else if (k == "trace") g.trace = value;
    else if (k == "chain_flags") g.chain_flags = value;

    else if (k == "fused") g.use_fused = value;
    else if (k == "prefill") g.use_prefill = value;
    else if (k == "prefill16") g.use_prefill16 = value;
    else if (k == "pf_streamk") g.pf_streamk = value;
    else if (k == "prefill_min_n") g.prefill_min_n = value;
    else if (k == "pdl") g.use_pdl = value;
    else if (k == "pdl_late") g.pdl_late = value;
    else if (k == "cs") g.cs_override = value;
    else if (k == "wpc") g.wpc_override = value;
    else if (k == "minb") g.minb_override = value;
    else if (k == "nbuf") g.nbuf_override = value;
    else return fail("tmac_b200_debug_set: unknown key '" + k + "'");
    return 0;
}

int tmac_b200_set_lut_mode(int mode) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    g.lut_mode = mode;
    return 0;
}

int tmac_b200_preprocessor(int K, int N, int act_group_size, int dtype, const void *B, void *LUT_Scales, void *LUT_Biases, void *QLUT) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (!B || !LUT_Scales || !LUT_Biases || !QLUT || N <= 0) return fail("preprocessor: null/empty argument");
    const int ags = (act_group_size <= 0 || act_group_size > K) ? K : act_group_size;
    if (K % 32 || ags % 32 || K % ags) return fail("preprocessor: bad K / act_group_size");
    const int nag = K / ags;
    const bool dev_in = is_device_ptr(B), dev_out = is_device_ptr(QLUT);
    if (dev_out != is_device_ptr(LUT_Scales) || dev_out != is_device_ptr(LUT_Biases)) return fail("preprocessor: outputs must live in one memory domain");
    const void *dB = B;
    if (!dev_in) {
        const size_t bytes = (size_t)N * K * esize(dtype);
        stage_wait();
        if (g.h_in.ensure(bytes)) return fail("out of pinned memory");
        if (h2d(g.d_b, g.h_in, 0, B, bytes)) return -1;
        stage_mark();
        dB = g.d_b.p;
    }
    float *dls = (float *)LUT_Scales, *dlb = (float *)LUT_Biases;
    int8_t *dq = (int8_t *)QLUT;
    const size_t qb = (size_t)N * K * 4, sb = (size_t)N * nag * 4;
    HostLut *hl = nullptr;
    if (!dev_out) {          // the LUT goes to the caller's host workspace AND stays on the device for the compute calls that follow
        hl = hlut_slot(QLUT);
        if (hl->dq.ensure(qb) || hl->dls.ensure(sb) || hl->dlb.ensure(sb)) return fail("out of device memory");
        dls = (float *)hl->dls.p; dlb = (float *)hl->dlb.p; dq = (int8_t *)hl->dq.p;
    }
    if (launch_preprocessor(K, N, ags, dtype, dB, dls, dlb, dq)) return -1;
    if (!dev_out) {
        if (g.h_out.ensure(qb + 2 * sb)) return fail("out of pinned memory");
        char *ho = (char *)g.h_out.p;
        CUDA_OK(cudaMemcpyAsync(ho, dq, qb, cudaMemcpyDeviceToHost, g.stream()));
        CUDA_OK(cudaMemcpyAsync(ho + qb, dls, sb, cudaMemcpyDeviceToHost, g.stream()));
        CUDA_OK(cudaMemcpyAsync(ho + qb + sb, dlb, sb, cudaMemcpyDeviceToHost, g.stream()));
        CUDA_OK(cudaStreamSynchronize(g.stream()));
        std::memcpy(QLUT, ho, qb);
        std::memcpy(LUT_Scales, ho + qb, sb);
        std::memcpy(LUT_Biases, ho + qb + sb, sb);
        hl->copy.assign((const unsigned char *)ho, (const unsigned char *)ho + qb + 2 * sb);
        hl->qb = qb; hl->sb = sb; hl->N = N; hl->sym = true; hl->res_id = 0;
    }
    return 0;
}

static int qgemm_impl(Resident &R, int row0, int rows, int N, int dtype, const void *QLUT, const void *LUT_Scales,
                      const void *LUT_Biases, void *C) {
    const StreamLayout &L = R.L;
    if (N <= 0 || rows <= 0) return fail("qgemm_lut: empty problem");
    if (!QLUT || !LUT_Scales || !LUT_Biases || !C) return fail("qgemm_lut: null argument");
    const int nag = L.K / L.act_group_size;
    const size_t qb = (size_t)N * L.K * 4, sb = (size_t)N * nag * 4;
    const bool dev_lut = is_device_ptr(QLUT);
    if (dev_lut != is_device_ptr(LUT_Scales) || dev_lut != is_device_ptr(LUT_Biases)) return fail("qgemm_lut: LUT inputs must live in one memory domain");
    const bool dev_c = is_device_ptr(C);
    const int8_t *dq = (const int8_t *)QLUT;
    const float *dls = (const float *)LUT_Scales, *dlb = (const float *)LUT_Biases;
    bool sym;
    HostLut *hl = nullptr;
    if (!dev_lut) {
        // device-resident copy keyed by (host pointer, content hash): written by the preprocessor call that filled this host
        // workspace, or uploaded here once when the caller brings a table of its own
        hl = hlut_find(QLUT, LUT_Scales, LUT_Biases, qb, sb);
        if (!hl) {
            hl = hlut_slot(QLUT);
            stage_wait();
            if (g.h_in.ensure(qb + 2 * sb)) return fail("out of pinned memory");
            if (h2d(hl->dq, g.h_in, 0, QLUT, qb) || h2d(hl->dls, g.h_in, qb, LUT_Scales, sb) || h2d(hl->dlb, g.h_in, qb + sb, LUT_Biases, sb)) return -1;
            stage_mark();
            hl->copy.resize(qb + 2 * sb);
            std::memcpy(hl->copy.data(), QLUT, qb); std::memcpy(hl->copy.data() + qb, LUT_Scales, sb); std::memcpy(hl->copy.data() + qb + sb, LUT_Biases, sb);
            hl->qb = qb; hl->sb = sb; hl->N = N; hl->res_id = 0;
            hl->sym = host_lut_symmetric((const int8_t *)QLUT, (size_t)N * L.K / 4);
        }
        sym = hl->sym;
        dq = (const int8_t *)hl->dq.p; dls = (const float *)hl->dls.p; dlb = (const float *)hl->dlb.p;
    } else
        sym = g.sym_qluts.count(QLUT) != 0;
    if (g.lut_mode == 1) sym = false;
    if (g.lut_mode == 2) sym = true;
    const size_t es = esize(dtype);
    if (hl && !dev_c) {
        // host LUT, host output (the reference's callers): the whole tensor is computed ONCE per (LUT bytes, tensor) straight
        // into page-locked host memory; this call and the later tile calls of the same mat-vec copy their rows out
        const bool hit = hl->res_id == R.id && hl->res_dtype == dtype && hl->N == N;
        if (!hit) {
            const size_t full = (size_t)N * L.Mout * es;
            if (hl->res.ensure(full)) return fail("out of pinned memory");
            if (launch_gemv(R, 0, L.Mout, N, dq, dls, dlb, hl->res.p, L.Mout, 0, dtype == TMAC_B200_F16, sym, nullptr)) return -1;
            CUDA_OK(cudaStreamSynchronize(g.stream()));
            hl->res_id = R.id; hl->res_dtype = dtype; hl->N = N;
        }
        for (int n = 0; n < N; ++n)
            std::memcpy((char *)C + (size_t)n * rows * es, (const char *)hl->res.p + ((size_t)n * L.Mout + row0) * es, (size_t)rows * es);
        return 0;
    }
    void *dC = C;
    const size_t cb = (size_t)N * rows * es;
    if (!dev_c) {
        if (g.d_c.ensure(cb)) return fail("out of device memory");
        dC = g.d_c.p;
    }
    if (launch_gemv(R, row0, row0 + rows, N, dq, dls, dlb, dC, rows, row0, dtype == TMAC_B200_F16, sym, nullptr)) return -1;
    if (!dev_c) {
        if (g.h_out.ensure(cb)) return fail("out of pinned memory");
        CUDA_OK(cudaMemcpyAsync(g.h_out.p, dC, cb, cudaMemcpyDeviceToHost, g.stream()));
        CUDA_OK(cudaStreamSynchronize(g.stream()));
        std::memcpy(C, g.h_out.p, cb);
    }
    return 0;
}

int tmac_b200_qgemm_lut(int64_t handle, int row0, int rows, int N, int dtype, const void *QLUT, const void *LUT_Scales,
                        const void *LUT_Biases, void *C) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    auto it = g.res.find(handle);
    if (it == g.res.end()) return fail("qgemm_lut: bad weight handle");
    return qgemm_impl(it->second, row0, rows, N, dtype, QLUT, LUT_Scales, LUT_Biases, C);
}

// Grouped launch: `count` qgemm_lut problems with identical geometry (same M, K, bits, grouping;
// e.g. the q/k/v or gate/up projections of a layer, the experts of an MoE layer, or any set of
// GEMVs whose LUTs are already available) in ONE kernel launch.  Device pointers only.
// QLUT[i], LUT_Scales[i], LUT_Biases[i], C[i] are per-problem device pointers (host arrays of pointers).
int tmac_b200_qgemm_lut_grouped(const int64_t *handles, int count, int N, int dtype, const void *const *QLUT,
                                const void *const *LUT_Scales, const void *const *LUT_Biases, void *const *C) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (!handles || count <= 0 || count > 65535 || !QLUT || !LUT_Scales || !LUT_Biases || !C) return fail("grouped: bad arguments");
    std::vector<const Resident *> rs(count);
    for (int i = 0; i < count; ++i) {
        auto it = g.res.find(handles[i]);
        if (it == g.res.end()) return fail("grouped: bad weight handle");
        rs[i] = &it->second;
        const StreamLayout &a = rs[0]->L, &b = rs[i]->L;
        if (a.Mout != b.Mout || a.K != b.K || a.bits != b.bits || a.blk != b.blk || a.nchunk != b.nchunk || a.zp != b.zp ||
            a.one_scale != b.one_scale || a.sd != b.sd || a.act_group_size != b.act_group_size || a.scale0 != b.scale0)
            return fail("grouped: all tensors must share one geometry");
        if (!is_device_ptr(QLUT[i]) || !is_device_ptr(C[i])) return fail("grouped: device pointers only");
    }
    bool sym = true;
    for (int i = 0; i < count; ++i) sym = sym && g.sym_qluts.count(QLUT[i]) != 0;
    if (g.lut_mode == 1) sym = false;
    if (g.lut_mode == 2) sym = true;
    // pointer tables: one device allocation per distinct call signature (stable under graph capture)
    std::vector<const void *> tab(5 * (size_t)count);
    for (int i = 0; i < count; ++i) {
        tab[i] = rs[i]->d; tab[count + i] = QLUT[i]; tab[2 * count + i] = LUT_Scales[i]; tab[3 * count + i] = LUT_Biases[i]; tab[4 * count + i] = C[i];
    }
    void *dtab = nullptr;
    for (auto &e : g.ptr_tables)
        if (e.first == tab) { dtab = e.second; break; }
    if (!dtab) {
        if (cudaMalloc(&dtab, tab.size() * sizeof(void *)) != cudaSuccess) { cudaGetLastError(); return fail("out of device memory (pointer table)"); }
        CUDA_OK(cudaMemcpy(dtab, tab.data(), tab.size() * sizeof(void *), cudaMemcpyHostToDevice));
        if (g.ptr_tables.size() >= 256) {          // bounded: evict the oldest table (its launches are complete or enqueued before this sync)
            cudaStreamSynchronize(g.stream());
            cudaFree(g.ptr_tables.front().second);
            g.ptr_tables.erase(g.ptr_tables.begin());
        }
        g.ptr_tables.emplace_back(tab, dtab);
    }
    const void **dt = (const void **)dtab;
    BatchPtrs bp;
    bp.n = count;
    bp.W = (const unsigned char *const *)dt; bp.q = (const int8_t *const *)(dt + count);
    bp.ls = (const float *const *)(dt + 2 * count); bp.lb = (const float *const *)(dt + 3 * count); bp.C = (void *const *)(dt + 4 * count);
    const StreamLayout &L = rs[0]->L;
    return launch_gemv3(*rs[0], 0, L.Mout, N, nullptr, nullptr, nullptr, nullptr, L.Mout, 0, dtype == TMAC_B200_F16, sym, &bp);
}

/* q/k/v or gate/up in ONE launch with the LUT built inside it: `count` tensors of one geometry applied to the SAME activation
 * rows B [N][K] (device), outputs C[i] [N][Mout] (device).  The one-call form of preprocessor + tmac_b200_qgemm_lut_grouped. */
int tmac_b200_gemv_grouped(const int64_t *handles, int count, int N, int dtype, const void *B, void *const *C) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (!handles || count <= 0 || count > 65535 || !B || !C || N <= 0) return fail("gemv_grouped: bad arguments");
    if (!is_device_ptr(B)) return fail("gemv_grouped: device pointers only");
    std::vector<const Resident *> rs(count);
    for (int i = 0; i < count; ++i) {
        auto it = g.res.find(handles[i]);
        if (it == g.res.end()) return fail("gemv_grouped: bad weight handle");
        rs[i] = &it->second;
        const StreamLayout &a = rs[0]->L, &b = rs[i]->L;
        if (a.Mout != b.Mout || a.K != b.K || a.bits != b.bits || a.blk != b.blk || a.nchunk != b.nchunk || a.zp != b.zp ||
            a.one_scale != b.one_scale || a.sd != b.sd || a.act_group_size != b.act_group_size || a.scale0 != b.scale0)
            return fail("gemv_grouped: all tensors must share one geometry");
        if (!is_device_ptr(C[i])) return fail("gemv_grouped: device pointers only");
    }
    const StreamLayout &L = rs[0]->L;
    const bool int_path = L.one_scale && L.act_group_size == L.K;
    if (!(int_path || L.act_group_size <= L.ck)) return fail("gemv_grouped: the activation group must lie inside a chunk (or be the whole row)");
    std::vector<const void *> tab(5 * (size_t)count, nullptr);
    for (int i = 0; i < count; ++i) { tab[i] = rs[i]->d; tab[4 * count + i] = C[i]; }
    void *dtab = nullptr;
    for (auto &e : g.ptr_tables)
        if (e.first == tab) { dtab = e.second; break; }
    if (!dtab) {
        if (cudaMalloc(&dtab, tab.size() * sizeof(void *)) != cudaSuccess) { cudaGetLastError(); return fail("out of device memory (pointer table)"); }
        CUDA_OK(cudaMemcpy(dtab, tab.data(), tab.size() * sizeof(void *), cudaMemcpyHostToDevice));
        if (g.ptr_tables.size() >= 256) {
            cudaStreamSynchronize(g.stream());
            cudaFree(g.ptr_tables.front().second);
            g.ptr_tables.erase(g.ptr_tables.begin());
        }
        g.ptr_tables.emplace_back(tab, dtab);
    }
    const void **dt = (const void **)dtab;
    BatchPtrs bp;
    bp.n = count;
    bp.W = (const unsigned char *const *)dt; bp.q = (const int8_t *const *)(dt + count);
    bp.ls = (const float *const *)(dt + 2 * count); bp.lb = (const float *const *)(dt + 3 * count); bp.C = (void *const *)(dt + 4 * count);
    return launch_gemv3(*rs[0], 0, L.Mout, N, nullptr, nullptr, nullptr, nullptr, L.Mout, 0, dtype == TMAC_B200_F16, true, &bp, B, dtype == TMAC_B200_F16);
}

int tmac_b200_gemv(int64_t handle, int N, int dtype, const void *B, void *C) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    auto it = g.res.find(handle);
    if (it == g.res.end()) return fail("gemv: bad weight handle");
    Resident &R = it->second;
    const StreamLayout &L = R.L;
    if (!B || !C || N <= 0) return fail("gemv: null/empty argument");
    const int nag = L.K / L.act_group_size;
    const size_t qb = (size_t)N * L.K * 4, sb = (size_t)N * nag * 4;
    const size_t bb = (size_t)N * L.K * esize(dtype), cb = (size_t)N * L.Mout * esize(dtype);
    void *pinB = nullptr, *pinC = nullptr;
    const int kind_b = ptr_kind(B, &pinB), kind_c = ptr_kind(C, &pinC);
    const bool dev_b = kind_b == 2, dev_c = kind_c == 2;
    const bool int_path = L.one_scale && L.act_group_size == L.K;
    const bool prefill_shape = g.use_prefill && N >= g.prefill_min_n && L.pb == 2 && L.qch == 8 && L.act_group_size == 64 && !L.one_scale;
    const bool can_fuse = g.use_fused && (int_path || L.act_group_size <= L.ck) && g.lut_mode != 1 && !prefill_shape;
    auto launch_compute = [&](const void *dB, void *dC) -> int {
        if (can_fuse)   // one launch: the GEMV builds each chunk's LUT slice itself (bit-identical tables)
            return launch_gemv3(R, 0, L.Mout, N, nullptr, nullptr, nullptr, dC, L.Mout, 0, dtype == TMAC_B200_F16, true, nullptr, dB,
                                dtype == TMAC_B200_F16);
        if (g.d_qlut.ensure(qb) || g.d_ls.ensure(sb) || g.d_lb.ensure(sb)) return fail("out of device memory");
        if (launch_preprocessor(L.K, N, L.act_group_size, dtype, dB, (float *)g.d_ls.p, (float *)g.d_lb.p, (int8_t *)g.d_qlut.p)) return -1;
        return launch_gemv(R, 0, L.Mout, N, (const int8_t *)g.d_qlut.p, (const float *)g.d_ls.p, (const float *)g.d_lb.p, dC, L.Mout, 0,
                           dtype == TMAC_B200_F16, g.lut_mode != 1, nullptr);
    };
    // The (small) output is stored by the kernel straight into page-locked host memory the device can address -- the
    // caller's own buffer when it is page-locked, else our staging buffer -- instead of a device buffer + D2H copy.
    void *dC = C;
    if (kind_c == 1) dC = pinC;
    else if (kind_c == 0) { if (g.h_out.ensure(cb)) return fail("out of pinned memory"); dC = g.h_out.p; }

    const void *dB = B;
    if (!dev_b) {
        stage_wait();
        if (kind_b == 1 && !dev_c) {
            // page-locked caller buffer as the copy source itself -- only when this call synchronises before returning (host
            // output); with a device output the call returns early and the caller may overwrite B at once: stage it instead
            if (g.d_b.ensure(bb)) return fail("out of device memory");
            CUDA_OK(cudaMemcpyAsync(g.d_b.p, pinB, bb, cudaMemcpyHostToDevice, g.stream()));
        } else {
            if (g.h_in.ensure(bb)) return fail("out of pinned memory");
            if (h2d(g.d_b, g.h_in, 0, B, bb)) return -1;
            stage_mark();
        }
        dB = g.d_b.p;
    }
    if (launch_compute(dB, dC)) return -1;
    if (!dev_c) {
        CUDA_OK(cudaStreamSynchronize(g.stream()));
        if (kind_c == 0) std::memcpy(C, g.h_out.p, cb);
    }
    return 0;
}

// ---- multi-GPU row sharding without a collective launch (SURVEY 8e) --------------------------------------------------
// Rows shard naturally (ref:ggml.c:12636-12691: tiles are independent given the replicated activation row), so the
// "all-gather" of a sharded GEMV is every rank storing its finished rows into every rank's output vector.  The next
// N = 1 launch (tmac_b200_gemv / tmac_b200_qgemm_lut) stores its rows, besides C, at ptrs[q] + the same index as C --
// device pointers into PEER memory (cudaIpcOpenMemHandle), each already offset to this shard's first row.  One-shot.
int tmac_b200_peer_outputs(void *const *ptrs, int count) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (count < 0 || count > 7 || (count && !ptrs)) return fail("peer_outputs: 0..7 peers");
    g.npeer = count;
    for (int q = 0; q < count; ++q) g.peer_out[q] = ptrs[q];
    return 0;
}
// One tiny launch: all launches this rank enqueued before it are complete, and so are the peers' up to their matching call --
// the flag / barrier per fused group of a row-sharded model (peer stores into `flags` of every rank; see peer_barrier_kernel).
// flags: this rank's (world + 1) x u32 array inside an ipc allocation; peer_flags[q]: rank q's array as mapped here.
int tmac_b200_peer_barrier(void *flags, void *const *peer_flags, int rank, int world) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (!flags || !peer_flags || world < 1 || world > 8 || rank < 0 || rank >= world) return fail("peer_barrier: bad arguments");
    // the pointer table lives in device memory (stable under graph capture): cached per (flags) key
    static std::map<void *, void *> tables;
    void *&dt = tables[flags];
    if (!dt) {
        if (cudaMalloc(&dt, 10 * sizeof(void *)) != cudaSuccess) { cudaGetLastError(); dt = nullptr; return fail("peer_barrier: out of device memory"); }
        void *host[9] = {};
        for (int q = 0; q < world; ++q) host[q] = peer_flags[q];
        CUDA_OK(cudaMemcpy(dt, host, sizeof host, cudaMemcpyHostToDevice));
    }
    peer_barrier_kernel<<<1, 32, 0, g.stream()>>>((unsigned *)flags, (unsigned *const *)dt, rank, world, (int *)((void **)dt + 8));
    CUDA_OK(cudaGetLastError());
    return 0;
}

// Device allocations that other processes of the node can map: alloc returns the pointer and a 64-byte handle to send to the
// peers; open maps a peer's allocation (peer access is enabled on demand); close / free undo them.
void *tmac_b200_ipc_alloc(size_t bytes, void *handle64) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return nullptr;
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); fail("ipc_alloc: out of device memory"); return nullptr; }
    cudaMemset(p, 0, bytes);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    if (cudaIpcGetMemHandle((cudaIpcMemHandle_t *)handle64, p) != cudaSuccess) { cudaGetLastError(); cudaFree(p); fail("cudaIpcGetMemHandle failed"); return nullptr; }
    return p;
}
void *tmac_b200_ipc_open(const void *handle64) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return nullptr;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle64, sizeof h);
    void *p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); fail(std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); return nullptr; }
    return p;
}
int tmac_b200_ipc_close(void *peer_ptr) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    CUDA_OK(cudaIpcCloseMemHandle(peer_ptr));
    return 0;
}
int tmac_b200_ipc_free(void *ptr) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (g.inited) cudaStreamSynchronize(g.stream());
    CUDA_OK(cudaFree(ptr));
    return 0;
}

// ---- decode sequences: a chain of dependent GEMVs in ONE persistent launch (tmac_seq.cuh) ---------------------------
// The reference runs a token step as ggml's graph loop over mul_mat nodes on a persistent thread pool
// (3rdparty/llama.cpp/ggml/src/ggml.c:12562-12706 per node); a sequence is that loop for the quantised linears.

int64_t tmac_b200_seq_create(void) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    const int64_t h = g_next_seq++;
    g_seqs[h];
    return h;
}

int tmac_b200_seq_add_gemv(int64_t seq, int64_t handle, const void *x, int in_op, int in_offset, void *C, int dtype) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end()) return fail("seq_add_gemv: bad sequence");
    Sequence &S = it->second;
    if (S.built) return fail("seq_add_gemv: sequence already built");
    auto rt = g.res.find(handle);
    if (rt == g.res.end()) return fail("seq_add_gemv: bad weight handle");
    const StreamLayout &L = rt->second.L;
    if (x) {
        if (!is_device_ptr(x)) return fail("seq_add_gemv: the external input must be a device pointer");
        if ((uintptr_t)x % 16) return fail("seq_add_gemv: the external input must be 16-byte aligned");
    } else {
        if (in_op < 0 || in_op >= (int)S.ops.size()) return fail("seq_add_gemv: in_op must name an earlier op of the sequence");
        const StreamLayout &P = g.res.find(S.ops[in_op].handle)->second.L;
        if (in_offset < 0 || in_offset % 2 || in_offset + L.K > P.Mout) return fail("seq_add_gemv: [in_offset, in_offset + K) must lie inside the producer's output (even offset)");
    }
    if (C && !is_device_ptr(C)) return fail("seq_add_gemv: C must be a device pointer (or NULL)");
    S.ops.push_back({handle, x, x ? -1 : in_op, in_offset, C, dtype == TMAC_B200_F16});
    return (int)S.ops.size() - 1;
}

/* Multi-GPU row sharding inside a sequence (as tmac_b200_peer_outputs for single launches): op `op` also stores its finished rows
 * at ptrs[q][row] -- device pointers into PEER memory, each already offset to this shard's first row.  Before seq_build. */
int tmac_b200_seq_peer_outputs(int64_t seq, int op, void *const *ptrs, int count) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end()) return fail("seq_peer_outputs: bad sequence");
    Sequence &S = it->second;
    if (S.built) return fail("seq_peer_outputs: sequence already built");
    if (op < 0 || op >= (int)S.ops.size() || count < 0 || count > 7 || (count && !ptrs)) return fail("seq_peer_outputs: bad op / 0..7 peers");
    if (!S.ops[op].C) return fail("seq_peer_outputs: the op has no output vector");
    S.ops[op].npeer = count;
    for (int q = 0; q < count; ++q) S.ops[op].peer[q] = ptrs[q];
    return 0;
}

// Resident gemv3 chain (tmac_chain.cuh): 1 = built, 0 = the sequence does not qualify (caller falls back), -1 = error.
static int seq_build_chain(Sequence &S) {
    const int n = (int)S.ops.size();
    std::vector<ChainOp> ops(n);
    std::vector<size_t> coff(n, (size_t)-1), lloff(n, 0);
    size_t ctot = 0, max_blk = 0, lltot = 0;
    int max_nrsb = 0, pb = 0, qch = 0, agq = 0, bits = 0, rsbsz = 0;
    for (int i = 0; i < n; ++i) {
        const Resident &R = g.res.find(S.ops[i].handle)->second;
        const StreamLayout &L = R.L;
        if ((L.one_scale && L.act_group_size == L.K) || L.act_group_size > L.ck) return 0;
        const int a = std::min(L.act_group_size, L.ck) / 16;
        if (i == 0) { pb = L.pb; qch = L.qch; agq = a; bits = L.bits; rsbsz = L.rsb; }
        else if (pb != L.pb || qch != L.qch || agq != a || bits != L.bits) return 0;
        if (S.ops[i].x_ext) { if ((uintptr_t)S.ops[i].x_ext % 16) return 0; }
        else if (S.ops[i].in_off % ((g.chain_flags & kChainBarrier) ? 4 : 2) || S.ops[S.ops[i].in_op].out_f16) return 0;    // float4 loads (16-byte word pairs in data-flow mode) of an fp32 producer
        max_blk = std::max(max_blk, (L.blk + 127) & ~(size_t)127);
        max_nrsb = std::max(max_nrsb, L.nrsb);
        if (!S.ops[i].C) { coff[i] = ctot; ctot += ((size_t)L.nrsb * L.rsb * sizeof(float) + 255) & ~(size_t)255; }
        lloff[i] = lltot; lltot += ((size_t)L.nrsb * L.rsb * sizeof(uint2) + 255) & ~(size_t)255;
    }
    chain_fn fn = pick_chain(pb, qch, agq);
    if (!fn) return 0;
    const int grid = max_nrsb * kChainCS;
    const size_t smem = (size_t)(kChainCS + kChainWarps) * rsbsz * 4 + (size_t)kChainWarps * (2 * max_blk + (size_t)qch * 4 * 8) + kChainWarps * 16 + 32;
    if (smem > 48 * 1024 && cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return 0; }
    cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    {   // every cluster must be resident at once: the grid barrier spins
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kChainWarps * 32); cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kChainCS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, (const void *)fn, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
        if (nc < max_nrsb) return 0;
    }
    if (cudaMalloc(&S.d_cops, n * sizeof(ChainOp)) != cudaSuccess || cudaMalloc(&S.d_bar, 256) != cudaSuccess ||
        cudaMalloc(&S.d_epochs, grid * sizeof(unsigned)) != cudaSuccess || cudaMalloc(&S.d_err, sizeof(int)) != cudaSuccess ||
        cudaMalloc(&S.d_cint, std::max<size_t>(ctot, 256)) != cudaSuccess || cudaMalloc(&S.d_y, lltot) != cudaSuccess) { cudaGetLastError(); S.release(); return fail("seq_build: out of device memory"); }
    // (on the library's stream: the legacy default stream does not order against a non-blocking stream)
    CUDA_OK(cudaMemsetAsync(S.d_y, 0, lltot, g.stream()));     // epoch 0 never matches: launches publish epochs >= 1
    CUDA_OK(cudaMemsetAsync(S.d_bar, 0, 256, g.stream())); CUDA_OK(cudaMemsetAsync(S.d_epochs, 0, grid * sizeof(unsigned), g.stream()));
    CUDA_OK(cudaMemsetAsync(S.d_err, 0, sizeof(int), g.stream()));
    for (int i = 0; i < n; ++i) {
        const StreamLayout &L = g.res.find(S.ops[i].handle)->second.L;
        ChainOp &o = ops[i];
        o.W = g.res.find(S.ops[i].handle)->second.d;
        o.C = S.ops[i].C ? S.ops[i].C : (void *)((char *)S.d_cint + coff[i]);
        o.x = S.ops[i].x_ext ? (const float *)S.ops[i].x_ext : (const float *)ops[S.ops[i].in_op].C + S.ops[i].in_off;
        o.rsb_stride = L.rsb_stride; o.K = L.K; o.Mout = L.Mout; o.nrsb = L.nrsb; o.nchunk = L.nchunk;
        o.blk_bytes = (int)L.blk; o.bpw = (L.nchunk + kChainCS * kChainWarps - 1) / (kChainCS * kChainWarps);
        o.zp = L.zp; o.one_scale = L.one_scale; o.sd = L.sd; o.out_f16 = S.ops[i].out_f16; o.scale0 = L.scale0;
        o.in_op = S.ops[i].x_ext ? -1 : S.ops[i].in_op;
        o.npeer = S.ops[i].npeer; o.pad_ = 0;
        for (int q = 0; q < 7; ++q) o.Cpeer[q] = q < S.ops[i].npeer ? S.ops[i].peer[q] : nullptr;

        o.ll_out = (uint2 *)((char *)S.d_y + lloff[i]);
        o.ll_in = S.ops[i].x_ext ? nullptr : (const uint2 *)((char *)S.d_y + lloff[S.ops[i].in_op]) + S.ops[i].in_off;
    }
    CUDA_OK(cudaMemcpyAsync(S.d_cops, ops.data(), n * sizeof(ChainOp), cudaMemcpyHostToDevice, g.stream()));
    CUDA_OK(cudaStreamSynchronize(g.stream()));
    S.cparams.ops = (const ChainOp *)S.d_cops; S.cparams.nops = n; S.cparams.max_blk = (int)max_blk;
    S.cparams.bar = (unsigned *)S.d_bar; S.cparams.epochs = (unsigned *)S.d_epochs; S.cparams.err = (int *)S.d_err;
    S.cparams.flags = g.chain_flags; S.cparams.trace = nullptr;

    if (g.trace) {
        const size_t tb = (size_t)n * grid * (16 + 16 * kSeqWarps) * sizeof(long long);    // same size as the stream-K kernel's trace (seq_trace copies that much)
        if (cudaMalloc(&S.d_trace, tb) != cudaSuccess) { cudaGetLastError(); S.release(); return fail("seq_build: out of device memory (trace)"); }
        cudaMemsetAsync(S.d_trace, 0, tb, g.stream());
        S.cparams.trace = (long long *)S.d_trace;
    }
    S.cfn = fn; S.impl = 1; S.grid = grid; S.smem = smem; S.pb = pb; S.qch = qch; S.agq = agq; S.bits = bits;
    S.built = true;
    return 1;
}

int tmac_b200_seq_build(int64_t seq) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end()) return fail("seq_build: bad sequence");
    Sequence &S = it->second;
    if (S.built) return 0;
    if (S.ops.empty()) return fail("seq_build: empty sequence");
    for (auto &o : S.ops) if (g.res.find(o.handle) == g.res.end()) return fail("seq_build: a weight handle was freed");
    if (g.seq_impl >= 1 && g.seq_grid == 0) {
        const int rc = seq_build_chain(S);
        if (rc != 0) return rc < 0 ? -1 : 0;
        if (g.seq_impl == 1) return fail("seq_build: the sequence does not qualify for the resident chain kernel (fp path, one format, fp32 16-byte aligned inputs, clusters resident)");
    }
    for (auto &o : S.ops) if (o.npeer) return fail("seq_build: peer outputs need the resident chain kernel, and this sequence does not qualify for it");
    const int G = g.seq_grid > 0 ? std::min(g.seq_grid, g.sms) : g.sms;
    const int n = (int)S.ops.size();
    std::vector<SeqOp> ops(n);
    std::vector<size_t> yoff(n);
    size_t ytot = 0, red_b = 0, tab_b = 0, lsb_b = 0, slot_b = 0, yfin_b = 0, ltot = 0;
    int rsbmax = 0;
    std::vector<size_t> loff(n, (size_t)-1);       // LUT hand-over records of op i (only if an aligned consumer exists)
    const bool handover = getenv("TMAC_B200_SEQ_HANDOVER") ? atoi(getenv("TMAC_B200_SEQ_HANDOVER")) != 0 : true;
    for (int i = 0; i < n; ++i) {
        auto rt = g.res.find(S.ops[i].handle);
        if (rt == g.res.end()) return fail("seq_build: a weight handle was freed");
        const StreamLayout &L = rt->second.L;
        const bool int_path = L.one_scale && L.act_group_size == L.K;
        if (int_path || L.act_group_size > L.ck) return fail("seq_build: activation group must lie inside a chunk (fp path)");
        const int agq = std::min(L.act_group_size, L.ck) / 16;
        if (i == 0) { S.pb = L.pb; S.qch = L.qch; S.agq = agq; S.bits = L.bits; }
        else if (S.pb != L.pb || S.qch != L.qch || S.agq != agq || S.bits != L.bits) return fail("seq_build: all tensors of a sequence must share bits / grouping");
        const long total = (long)L.nrsb * L.nchunk;
        const long ge = std::min<long>(G, total);
        const int per = (int)((total + ge - 1) / ge);
        const int nseg = (per - 1 + L.nchunk - 1) / L.nchunk + 1;
        const int ntab = std::min(per, L.nchunk);
        const int nag = L.qch / agq;
        red_b = std::max(red_b, (size_t)nseg * kSeqWarps * L.rsb * 4);
        yfin_b = std::max(yfin_b, (size_t)nseg * L.rsb * 4);
        if (!S.ops[i].x_ext && handover) {   // consumer of an earlier op: can it take ready-made LUT records?
            const int src = S.ops[i].in_op;
            const StreamLayout &PL = g.res.find(S.ops[src].handle)->second.L;
            if (S.ops[i].in_off % L.act_group_size == 0 && PL.rsb % L.act_group_size == 0 && loff[src] == (size_t)-1) {
                loff[src] = ltot;
                const size_t rows = (size_t)PL.nrsb * PL.rsb;
                ltot += ((rows / 4 + rows / L.act_group_size) * sizeof(uint4) + 255) & ~(size_t)255;
            }
        }
        tab_b = std::max(tab_b, (size_t)ntab * L.qch * 4 * 8);
        lsb_b = std::max(lsb_b, (size_t)ntab * 2 * nag * 4);
        slot_b = std::max(slot_b, (L.blk + 127) & ~(size_t)127);
        rsbmax = std::max(rsbmax, L.rsb);
        yoff[i] = ytot;
        ytot += ((size_t)L.nrsb * L.rsb * sizeof(uint2) + 255) & ~(size_t)255;
    }
    const size_t budget = (size_t)std::max(64, std::min(227, g.seq_smem_kb)) * 1024;
    const size_t fixed = ((red_b + 15) & ~(size_t)15) + ((tab_b + 15) & ~(size_t)15) + ((lsb_b + 15) & ~(size_t)15) + ((yfin_b + 15) & ~(size_t)15) + 64 * 8 + (kSeqWarps + 1) * 4 + 64 + 2 * kSeqDescWords * 4;
    if (fixed + 4 * slot_b > budget) return fail("seq_build: shared-memory budget exceeded");
    const int nslots = (int)std::min<size_t>(64, (budget - fixed) / slot_b);
    S.fn = pick_seq(S.pb, S.qch, S.agq);
    if (!S.fn) return fail("seq_build: chunking not instantiated");
    S.grid = G;
    const size_t xper = (size_t)G * rsbmax * sizeof(uint2);
    if (cudaMalloc(&S.d_ops, n * sizeof(SeqOp)) != cudaSuccess || cudaMalloc(&S.d_ctas, (size_t)n * G * sizeof(SeqCta)) != cudaSuccess || cudaMalloc(&S.d_y, ytot) != cudaSuccess ||
        cudaMalloc(&S.d_xchg, xper * n) != cudaSuccess || cudaMalloc(&S.d_lut, std::max<size_t>(ltot, 256)) != cudaSuccess || cudaMalloc(&S.d_epochs, G * sizeof(unsigned)) != cudaSuccess ||
        cudaMalloc(&S.d_err, sizeof(int)) != cudaSuccess) { cudaGetLastError(); S.release(); return fail("seq_build: out of device memory"); }
    if (g.trace) {
        if (cudaMalloc(&S.d_trace, (size_t)n * G * (16 + 16 * kSeqWarps) * sizeof(long long)) != cudaSuccess) { cudaGetLastError(); S.release(); return fail("seq_build: out of device memory (trace)"); }
        cudaMemsetAsync(S.d_trace, 0, (size_t)n * G * (16 + 16 * kSeqWarps) * sizeof(long long), g.stream());
    }
    CUDA_OK(cudaMemsetAsync(S.d_y, 0, ytot, g.stream()));
    CUDA_OK(cudaMemsetAsync(S.d_lut, 0, std::max<size_t>(ltot, 256), g.stream()));
    CUDA_OK(cudaMemsetAsync(S.d_xchg, 0, xper * n, g.stream()));
    CUDA_OK(cudaMemsetAsync(S.d_epochs, 0, G * sizeof(unsigned), g.stream()));
    CUDA_OK(cudaMemsetAsync(S.d_err, 0, sizeof(int), g.stream()));
    for (int i = 0; i < n; ++i) {
        const Resident &R = g.res.find(S.ops[i].handle)->second;
        const StreamLayout &L = R.L;
        SeqOp &o = ops[i];
        o.W = R.d;
        o.x_ext = (const float *)S.ops[i].x_ext;
        o.x_ll = S.ops[i].x_ext ? nullptr : (const uint2 *)((char *)S.d_y + yoff[S.ops[i].in_op]) + S.ops[i].in_off;
        o.C = S.ops[i].C;
        o.y = (uint2 *)((char *)S.d_y + yoff[i]);
        o.xchg = (uint2 *)((char *)S.d_xchg + xper * i);
        o.rsb_stride = L.rsb_stride;
        o.K = L.K; o.Mout = L.Mout; o.nrsb = L.nrsb; o.nchunk = L.nchunk;
        o.blk_bytes = (int)L.blk; o.total = L.nrsb * L.nchunk;
        o.zp = L.zp; o.one_scale = L.one_scale; o.sd = L.sd; o.out_f16 = S.ops[i].out_f16;
        o.scale0 = L.scale0; o.geff = std::min(G, o.total);
        o.lut_out = o.ag_out = nullptr; o.lut_in = o.ag_in = nullptr;
        if (loff[i] != (size_t)-1) {
            o.lut_out = (uint4 *)((char *)S.d_lut + loff[i]);
            o.ag_out = o.lut_out + (size_t)L.nrsb * L.rsb / 4;
        }
        if (!S.ops[i].x_ext && handover) {
            const int src = S.ops[i].in_op;
            const StreamLayout &PL = g.res.find(S.ops[src].handle)->second.L;
            if (loff[src] != (size_t)-1 && S.ops[i].in_off % L.act_group_size == 0 && PL.rsb % L.act_group_size == 0) {
                const uint4 *base = (const uint4 *)((char *)S.d_lut + loff[src]);
                o.lut_in = base + S.ops[i].in_off / 4;
                o.ag_in = base + (size_t)PL.nrsb * PL.rsb / 4 + S.ops[i].in_off / L.act_group_size;
            }
        }
    }
    CUDA_OK(cudaMemcpy(S.d_ops, ops.data(), n * sizeof(SeqOp), cudaMemcpyHostToDevice));
    {   // per (op, CTA) shares: blocks [T*c/GE, T*(c+1)/GE) in (row super-block, chunk) order
        std::vector<SeqCta> ct((size_t)n * G);
        const int pmax = std::max(1, nslots / 2);
        for (int i = 0; i < n; ++i) {
            const long T = ops[i].total, GE = ops[i].geff, nc = ops[i].nchunk;
            auto first_block = [&](long c) { return T * c / GE; };
            for (int c = 0; c < G; ++c) {
                SeqCta &q = ct[(size_t)i * G + c];
                std::memset(&q, 0, sizeof q);
                q.fc = c;
                if (c >= GE) continue;
                const long b0 = first_block(c), b1 = first_block(c + 1);
                q.b0 = (int)b0; q.nb = (int)(b1 - b0);
                q.sb_first = (int)(b0 / nc); q.c0 = (int)(b0 % nc);
                q.nseg = (int)((b1 - 1) / nc - b0 / nc + 1);
                q.nck = (int)std::min<long>(q.nb, nc);
                q.npass = (q.nb + pmax - 1) / pmax;
                q.P = (q.nb + q.npass - 1) / q.npass;
                q.last_open = (b1 % nc) != 0;                     // my last super-block continues in CTA c + 1
                int fc = c;                                       // CTA that owns the first block of my first super-block
                while (fc > 0 && first_block(fc) > (long)q.sb_first * nc) --fc;
                q.fc = fc;
            }
        }
        CUDA_OK(cudaMemcpy(S.d_ctas, ct.data(), ct.size() * sizeof(SeqCta), cudaMemcpyHostToDevice));
    }
    SeqParams &P = S.params;
    P.ops = (const SeqOp *)S.d_ops; P.ctas = (const SeqCta *)S.d_ctas; P.nops = n; P.nslots = nslots; P.slot_bytes = (int)slot_b;
    size_t off = (size_t)nslots * slot_b;
    P.red_off = (int)off; off += (red_b + 15) & ~(size_t)15;
    P.tab_off = (int)off; off += (tab_b + 15) & ~(size_t)15;
    P.lsb_off = (int)off; off += (lsb_b + 15) & ~(size_t)15;
    P.bar_off = (int)off; off += (size_t)nslots * 8;
    P.prog_off = (int)off; off += (kSeqWarps + 1) * 4;   // + the producer's `issued` counter
    off = (off + 15) & ~(size_t)15;
    P.yfin_off = (int)off; off += (yfin_b + 15) & ~(size_t)15;
    P.desc_off = (int)off; off += 2 * kSeqDescWords * 4;
    P.epochs = (unsigned *)S.d_epochs; P.err = (int *)S.d_err; P.trace = (long long *)S.d_trace;
    S.smem = off;
    CUDA_OK(cudaFuncSetAttribute((const void *)S.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.smem));
    S.built = true;
    return 0;
}

int tmac_b200_seq_launch(int64_t seq) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end()) return fail("seq_launch: bad sequence");
    Sequence &S = it->second;
    if (!S.built) return fail("seq_launch: call tmac_b200_seq_build first");
    uint32_t wtx, wty;
    plane_weight_regs(S.bits, true, &wtx, &wty);
    if (S.impl == 1) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(S.grid); cfg.blockDim = dim3(kChainWarps * 32); cfg.dynamicSmemBytes = S.smem; cfg.stream = g.stream();
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kChainCS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        CUDA_OK(cudaLaunchKernelEx(&cfg, S.cfn, S.cparams, wtx, wty));
        return 0;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(S.grid, 1, 1);
    cfg.blockDim = dim3(kSeqThreads, 1, 1);
    cfg.dynamicSmemBytes = S.smem;
    cfg.stream = g.stream();
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;      // every CTA must be resident: CTAs wait for each other's rows
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    CUDA_OK(cudaLaunchKernelEx(&cfg, S.fn, S.params, wtx, wty));
    return 0;
}

/* Synchronises the stream and returns the sequence's error flag (0 = every wait completed). */
int tmac_b200_seq_status(int64_t seq) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end() || !it->second.built) return fail("seq_status: bad sequence");
    CUDA_OK(cudaStreamSynchronize(g.stream()));
    int e = 0;
    CUDA_OK(cudaMemcpy(&e, it->second.d_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (e) return fail("sequence kernel: a bounded wait expired (code " + std::to_string(e) + ")");
    return 0;
}

/* info[8] = {grid, ring slots, slot bytes, shared memory bytes, ops, planes/word, quads/chunk, quads/act group} */
int tmac_b200_seq_info(int64_t seq, int *out8) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end() || !it->second.built || !out8) return fail("seq_info: bad sequence");
    const Sequence &S = it->second;
    const int v[8] = {S.grid, S.impl == 1 ? -kChainCS : S.params.nslots, S.impl == 1 ? S.cparams.max_blk : S.params.slot_bytes, (int)S.smem, (int)S.ops.size(), S.pb, S.qch, S.agq};
    std::memcpy(out8, v, sizeof v);
    return 0;
}

/* Debug (knob "trace" set before seq_build): globaltimer stamps [ops][grid][8] of the last launch; returns grid. */
int tmac_b200_seq_trace(int64_t seq, long long *dst, size_t cap_bytes) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end() || !it->second.built || !it->second.d_trace) return fail("seq_trace: tracing was not enabled when the sequence was built");
    CUDA_OK(cudaStreamSynchronize(g.stream()));
    const size_t bytes = std::min(cap_bytes, it->second.ops.size() * (size_t)it->second.grid * (16 + 16 * kSeqWarps) * sizeof(long long));
    CUDA_OK(cudaMemcpy(dst, it->second.d_trace, bytes, cudaMemcpyDeviceToHost));
    return it->second.grid;
}

int tmac_b200_seq_free(int64_t seq) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_seqs.find(seq);
    if (it == g_seqs.end()) return fail("seq_free: bad sequence");
    if (g.inited) cudaStreamSynchronize(g.stream());
    it->second.release();
    g_seqs.erase(it);
    return 0;
}

int tmac_b200_cbits(int64_t handle, int N, const void *QLUT, int32_t *CBits) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    auto it = g.res.find(handle);
    if (it == g.res.end()) return fail("cbits: bad weight handle");
    Resident &R = it->second;
    const StreamLayout &L = R.L;
    if (!QLUT || !CBits || N <= 0) return fail("cbits: null/empty argument");
    const size_t qb = (size_t)N * L.K * 4, ob = (size_t)N * L.Mout * L.bits * 4;
    const int8_t *dq = (const int8_t *)QLUT;
    if (!is_device_ptr(QLUT)) {
        stage_wait();
        if (g.h_in.ensure(qb)) return fail("out of pinned memory");
        if (h2d(g.d_qlut, g.h_in, 0, QLUT, qb)) return -1;
        stage_mark();
        dq = (const int8_t *)g.d_qlut.p;
    }
    const bool dev_o = is_device_ptr(CBits);
    int32_t *dout = CBits;
    if (!dev_o) {
        if (g.d_cbits.ensure(ob)) return fail("out of device memory");
        dout = (int32_t *)g.d_cbits.p;
    }
    const long long total = (long long)N * L.Mout * L.bits;
    cbits_kernel<<<(unsigned)((total + 255) / 256), 256, 0, g.stream()>>>(R.d, dq, dout, L.Mout, L.K, L.bits, L.pb, L.qch, L.nchunk,
                                                                         L.rsb_stride, L.blk, N);
    CUDA_OK(cudaGetLastError());
    if (!dev_o) {
        CUDA_OK(cudaMemcpyAsync(CBits, dout, ob, cudaMemcpyDeviceToHost, g.stream()));
        CUDA_OK(cudaStreamSynchronize(g.stream()));
    }
    return 0;
}

// ---- reference dispatchers ---------------------------------------------------------------
int preprocessor_int8(int m, int k, int n, int b, void *B, void *LUT_Scales, void *LUT_Biases, void *QLUT) {
    int ags, dtype;
    {
        std::unique_lock<std::shared_mutex> lk(g_mu);
        const tmac_b200_kcfg *c = find_kcfg_locked(m, k, b);
        if (!c) return fail("preprocessor_int8: shape not configured (m=" + std::to_string(m) + ", k=" + std::to_string(k) + ", b=" + std::to_string(b) + ")");
        ags = c->act_group_size;
        dtype = g.float_type;
    }
    return tmac_b200_preprocessor(k, n, ags, dtype, B, LUT_Scales, LUT_Biases, QLUT);
}

int qgemm_lut_int8(int m, int k, int n, int b, void *A, void *LUT, void *Scales, void *LUT_Scales, void *LUT_Biases, void *C) {
    (void)Scales;  // the resident copy carries the scales that were uploaded together with A
    if (g.inited && b >= 1 && b <= 4 && m > 0 && m % b == 0 && !is_device_ptr(LUT) && !is_device_ptr(C)) {
        // read-only fast path (shared lock): a tile call of a mat-vec whose whole-tensor result is already in page-locked memory
        // (computed by an earlier tile call with the same LUT bytes) only copies its rows -- ggml's workers do this concurrently
        std::shared_lock<std::shared_mutex> rl(g_mu);
        size_t off = 0;
        Resident *R = find_by_alias(A, &off);
        if (R && R->cfg.K == k && R->cfg.bits == b) {
            const size_t tile_bytes = (size_t)(k / 4) * R->cfg.bm / 2;
            const int row0 = (int)(off / tile_bytes) * (R->cfg.bm / b), rows = m / b;
            const size_t qb = (size_t)n * k * 4, sb = (size_t)n * (k / R->L.act_group_size) * 4, es = esize(g.float_type);
            if (off % tile_bytes == 0 && row0 + rows <= R->L.Mout)
                for (HostLut &e : g.hluts)
                    if (e.hq == LUT && e.res_id == R->id && e.res_dtype == g.float_type && e.N == n && e.qb == qb && e.sb == sb &&
                        e.copy.size() == qb + 2 * sb && !std::memcmp(e.copy.data(), LUT, qb) && !std::memcmp(e.copy.data() + qb, LUT_Scales, sb) &&
                        !std::memcmp(e.copy.data() + qb + sb, LUT_Biases, sb)) {
                        for (int r = 0; r < n; ++r)
                            std::memcpy((char *)C + (size_t)r * rows * es, (const char *)e.res.p + ((size_t)r * R->L.Mout + row0) * es, (size_t)rows * es);
                        return 0;
                    }
        }
    }
    std::unique_lock<std::shared_mutex> lk(g_mu);
    if (ensure_init()) return -1;
    if (b < 1 || b > 4 || m <= 0 || m % b) return fail("qgemm_lut_int8: bad m/b");
    size_t off = 0;
    Resident *R = find_by_alias(A, &off);
    if (!R) return fail("qgemm_lut_int8: A is not a registered weight tensor (call tmac_b200_upload_weights / ggml_tmac_b200_transform_tensor at load time)");
    if (R->cfg.K != k || R->cfg.bits != b) return fail("qgemm_lut_int8: (k, b) do not match the registered tensor");
    const size_t tile_bytes = (size_t)(k / 4) * R->cfg.bm / 2;
    if (off % tile_bytes) return fail("qgemm_lut_int8: A is not at a tile boundary");
    const int row0 = (int)(off / tile_bytes) * (R->cfg.bm / b);
    const int rows = m / b;
    if (row0 + rows > R->L.Mout) return fail("qgemm_lut_int8: tile range exceeds the tensor");
    return qgemm_impl(*R, row0, rows, n, g.float_type, LUT, LUT_Scales, LUT_Biases, C);
}

// ---- ggml hook -----------------------------------------------------------------------------
void ggml_tmac_init(void) {
    if (tmac_b200_init(-1) != 0) { fprintf(stderr, "ggml_tmac_init: %s\n", tmac_b200_last_error()); return; }
    if (const char *f = getenv("TMAC_KCFG_FILE")) {   // tmac_gemm_wrapper.h:40-56
        if (tmac_b200_load_kcfg_file(f) < 0) fprintf(stderr, "ggml_tmac_init: %s\n", tmac_b200_last_error());
    }
}
void ggml_tmac_free(void) { tmac_b200_shutdown(); }

// ggml-tmac.cpp:267-275: ggml's n (output dim) / m (batch) are swapped relative to T-MAC.
void ggml_tmac_mul_mat_task_init(void *src1, void *qlut, void *lut_scales, void *lut_biases, int n, int k, int m, int bits) {
    if (preprocessor_int8(n * bits, k, m, bits, src1, lut_scales, lut_biases, qlut) != 0)
        fprintf(stderr, "ggml_tmac_mul_mat_task_init: %s\n", tmac_b200_last_error());
}
void ggml_tmac_mul_mat_task_compute(void *src0, void *scales, void *qlut, void *lut_scales, void *lut_biases, void *dst, int n, int k,
                                    int m, int bits) {
    if (qgemm_lut_int8(n * bits, k, m, bits, src0, qlut, scales, lut_scales, lut_biases, dst) != 0)
        fprintf(stderr, "ggml_tmac_mul_mat_task_compute: %s\n", tmac_b200_last_error());
}
// Caller emulation for measurements and tests: ggml_compute_forward_mul_mat's T-MAC branch (ref:ggml.c:12562-12706) for one
// activation row, in C++ so that no interpreter overhead sits between the hook calls.  Phase 1: ggml_tmac_mul_mat_task_init
// (one call).  Phase 2: per_tile = 0 -> one ggml_tmac_mul_mat_task_compute for the whole tensor (the TMAC_USE_TVM_THREADPOOL
// branch, :12610-12630); per_tile = 1 -> one call per weight tile of `tile_rows` rows from `threads` host threads that steal
// tiles through an atomic counter (:12632-12703).  All pointers are HOST pointers as in ggml.
int tmac_b200_debug_ggml_mul_mat(void *src0_qweights, void *src0_scales, void *src1_row, void *wdata, void *dst, int ne01, int ne00,
                                 int bits, int tile_rows, int per_tile, int threads) {
    if (!src0_qweights || !src1_row || !wdata || !dst || ne01 <= 0 || ne00 <= 0 || bits < 1 || bits > 4 || tile_rows <= 0 || ne01 % tile_rows)
        return fail("debug_ggml_mul_mat: bad arguments");
    tmac_b200_kcfg c;
    if (tmac_b200_find_kcfg(ne01 * bits, ne00, bits, &c)) return fail("debug_ggml_mul_mat: shape not configured");
    // workspace layout of ggml.c:12566-12576: qlut (K * 4 bytes) || lut_scales || lut_biases
    char *qlut = (char *)wdata;
    float *ls = (float *)(qlut + (size_t)ne00 * 4), *lb = ls + ne00 / c.act_group_size;
    ggml_tmac_mul_mat_task_init(src1_row, qlut, ls, lb, ne01, ne00, 1, bits);
    if (!per_tile) {
        ggml_tmac_mul_mat_task_compute(src0_qweights, src0_scales, qlut, ls, lb, dst, ne01, ne00, 1, bits);
        return 0;
    }
    const int n_tiles = ne01 / tile_rows;
    const size_t w_chunk = (size_t)ne00 * tile_rows * bits / 8;               // bytes of one tile in the permuted blob (:12636)
    const size_t s_chunk = c.one_scale ? 0 : (size_t)tile_rows * (ne00 / c.group_size) * (c.zero_point ? 2 : 1);
    // tile-stealing workers, parked between calls like ggml's thread pool (spawning threads per mat-vec would dominate)
    struct Pool {
        std::vector<std::thread> th;
        std::atomic<int> gen{0}, done{0}, next{0}, stop{0};
        std::function<void()> job;
        ~Pool() { stop = 1; gen++; for (auto &t : th) t.join(); }
    };
    static Pool pool;
    static std::mutex pool_mu;
    std::lock_guard<std::mutex> pl(pool_mu);
    const int extra = std::max(0, std::min(threads, 64) - 1);
    pool.next = 0; pool.done = 0;
    pool.job = [&, n_tiles, w_chunk, s_chunk]() {
        for (int t = pool.next.fetch_add(1); t < n_tiles; t = pool.next.fetch_add(1))
            ggml_tmac_mul_mat_task_compute((char *)src0_qweights + t * w_chunk, src0_scales ? (float *)src0_scales + t * s_chunk : nullptr, qlut, ls, lb,
                                           (float *)dst + (size_t)t * tile_rows, tile_rows, ne00, 1, bits);
    };
    while ((int)pool.th.size() < extra)
        pool.th.emplace_back([&p = pool, my = pool.gen.load()]() mutable {
            for (;;) {
                while (p.gen.load(std::memory_order_acquire) == my) std::this_thread::yield();
                my = p.gen.load();
                if (p.stop) return;
                p.job();
                p.done.fetch_add(1, std::memory_order_release);
            }
        });
    const int nworkers = (int)pool.th.size();
    pool.gen.fetch_add(1, std::memory_order_release);
    pool.job();
    while (pool.done.load(std::memory_order_acquire) < nworkers) std::this_thread::yield();
    return 0;
}

void ggml_tmac_set_n_threads(int n_threads) { (void)n_threads; /* CPU thread pool size is irrelevant on the GPU */ }

int ggml_tmac_get_type_bits(int type) {  // ggml-tmac.cpp:503-522; ids from ggml.h:359,391-396
    switch (type) {
        case 36: return 1;   // GGML_TYPE_I1
        case 37: return 2;   // GGML_TYPE_I2
        case 38: return 3;   // GGML_TYPE_I3
        case 39: return 4;   // GGML_TYPE_I4
        case 2: return 4;    // GGML_TYPE_Q4_0
        case 34: return 2;   // GGML_TYPE_TQ1_0
        case 35: return 2;   // GGML_TYPE_TQ2_0
        default: return 0;
    }
}

int ggml_tmac_b200_can_mul_mat(int src0_type, int src1_is_f32, int dst_is_f32, const char *src0_name) {
    // ggml-tmac.cpp:72-96,238-248 minus the backend check (weights live in HBM here): the pre-permuted I1..I4 types and
    // the block types the reference re-permutes at load time (Q4_0, TQ1_0, TQ2_0).
    const bool supported = (src0_type >= 36 && src0_type <= 39) || ggml_block_elems(src0_type) > 0;
    if (!supported || !src1_is_f32 || !dst_is_f32) return 0;
    if (src0_name && (!strcmp(src0_name, "token_embd.weight") || !strcmp(src0_name, "output.weight"))) return 0;
    return 1;
}

size_t ggml_tmac_b200_mul_mat_get_wsize(int ne01, int ne10, int ne11, int bits) {  // ggml-tmac.cpp:250-265
    tmac_b200_kcfg c;
    if (tmac_b200_find_kcfg(ne01 * bits, ne10, bits, &c)) return 0;
    const size_t lss = (size_t)ne10 / c.act_group_size;
    size_t wsize = (size_t)ne10 * ne11 * 4 + lss * ne11 * 2 * sizeof(float);
    return ((wsize - 1) / 64 + 1) * 64;
}

size_t ggml_tmac_b200_get_nbytes(int ne00, int ne01, int bits) {  // ggml-tmac.cpp:277-288
    tmac_b200_kcfg c;
    if (tmac_b200_find_kcfg(ne01 * bits, ne00, bits, &c)) return 0;
    const size_t ss = c.one_scale ? 1 : (size_t)c.M * (c.K / c.group_size) * (c.zero_point ? 2 : 1);
    return (size_t)ne00 * ne01 / 8 * bits + ss * sizeof(float);
}

int ggml_tmac_b200_transform_tensor(void *data, int ne00, int ne01, int bits, struct tmac_tensor_extra_b200 *extra) {
    // ggml-tmac.cpp:290-354, I1..I4 branch (:336-345): the blob is `permuted weights || fp32 scales`.
    tmac_b200_kcfg c;
    if (tmac_b200_find_kcfg(ne01 * bits, ne00, bits, &c)) return -1;
    if (c.M != ne01) return fail("transform_tensor: kcfg is for a different M");
    uint8_t *qweights = (uint8_t *)data;
    float *scales = (float *)(qweights + (size_t)ne00 * ne01 * bits / 8);
    const int64_t h = tmac_b200_upload_weights(&c, qweights, scales, TMAC_B200_F32);
    if (h < 0) return -1;
    if (extra) {
        extra->lut_scales_size = ne00 / c.act_group_size;
        extra->scales_size = c.one_scale ? 1 : c.M * (c.K / c.group_size) * (c.zero_point ? 2 : 1);
        extra->n_tile_num = c.M * c.bits / c.bm;
        extra->qweights = qweights;
        extra->scales = scales;
    }
    return (int)h;
}

// ggml-tmac.cpp:290-498 for every type it supports: I1..I4 blobs are aliased in place (above); Q4_0 / TQ1_0 / TQ2_0
// blocks are decoded element by element like the reference's accessors and encoded into the stream layout.  The
// reference hands ggml a freshly allocated permuted copy in extra->qweights; here that pointer is only an ADDRESS KEY
// (ggml.c adds tile offsets to it and passes it back), so a PROT_NONE reservation of the same size stands in for it.
int ggml_tmac_b200_transform_tensor_typed(void *data, int ggml_type, int ne00, int ne01, struct tmac_tensor_extra_b200 *extra) {
    const int bits = ggml_tmac_get_type_bits(ggml_type);
    if (!bits || !data) return fail("transform_tensor: unsupported ggml type " + std::to_string(ggml_type));
    if (ggml_type >= 36 && ggml_type <= 39) return ggml_tmac_b200_transform_tensor(data, ne00, ne01, bits, extra);
    tmac_b200_kcfg c;
    if (tmac_b200_find_kcfg(ne01 * bits, ne00, bits, &c)) return -1;
    if (c.M != ne01) return fail("transform_tensor: kcfg is for a different M");
    const int E = ggml_block_elems(ggml_type);
    if (c.one_scale || c.zero_point || c.group_size != E)
        return fail("transform_tensor: block type needs a kcfg with group_size = " + std::to_string(E) + ", no zero point, per-group scales");
    if (validate_cfg(c)) return -1;
    std::vector<uint8_t> w((size_t)ne01 * ne00);
    std::vector<float> sc((size_t)ne01 * (ne00 / E));
    if (!decode_ggml_blocks(ggml_type, data, ne01, ne00, w.data(), sc.data())) return fail("transform_tensor: K is not a multiple of the block size");
    const size_t abytes = (size_t)ne00 * ne01 * bits / 8;
    void *key = mmap(nullptr, abytes, PROT_NONE, MAP_PRIVATE | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
    if (key == MAP_FAILED) return fail("transform_tensor: cannot reserve an address range for the tensor");
    // scales in the reference's run-time order [M/bm][K/gs][bm/bits] (ggml-tmac.cpp:464-489)
    const int NG = ne00 / E, rows_per_tile = c.bm / bits;
    float *hs = (float *)std::malloc(sc.size() * sizeof(float));
    if (!hs) { munmap(key, abytes); return fail("out of host memory"); }
    for (int r = 0; r < ne01; ++r)
        for (int gk = 0; gk < NG; ++gk)
            hs[((size_t)(r / rows_per_tile) * NG + gk) * rows_per_tile + r % rows_per_tile] = sc[(size_t)r * NG + gk];
    int64_t h;
    {
        std::unique_lock<std::shared_mutex> lk(g_mu);
        if (ensure_init()) { munmap(key, abytes); std::free(hs); return -1; }
        PlainWeights P;
        plain_from_w(w.data(), ne01, ne00, bits, 0, ne01, &P);
        P.scales = sc;
        h = register_resident(c, P, key, abytes, 0);
        if (h < 0) { munmap(key, abytes); std::free(hs); return -1; }
        Resident &R = g.res[h];
        R.reserved = key; R.reserved_bytes = abytes; R.host_scales = hs;
    }
    if (extra) {
        extra->lut_scales_size = ne00 / c.act_group_size;
        extra->scales_size = ne01 * NG;
        extra->n_tile_num = c.M * c.bits / c.bm;
        extra->qweights = (uint8_t *)key;
        extra->scales = hs;
    }
    return (int)h;
}

// Host-only (no GPU): the decode step of the typed transform, for the CPU suite.  w [ne01][ne00] codes, scales
// [ne01][ne00 / block elems].  Returns the block size or -1.
int tmac_b200_debug_decode_ggml(int ggml_type, const void *data, int ne00, int ne01, uint8_t *w, float *scales) {
    if (!data || !w || !scales) return fail("debug_decode_ggml: null argument");
    if (!decode_ggml_blocks(ggml_type, data, ne01, ne00, w, scales)) return fail("debug_decode_ggml: unsupported type or K");
    return ggml_block_elems(ggml_type);
}

// The reference's default tiling when no tuned kcfg exists (python/t_mac/ops/qgemm.py:98-115: the first candidate of each knob):
// bm = first of {256,128,512,1024,320,640} ({192,384,576,768} for 3 bits) dividing M*bits with bm % bits == 0; kfactor = first
// of {8,16} with (4*kfactor) % act_group_size == 0 and group_size % (4*kfactor) == 0 (any of them on the do_scale_final path).
int tmac_b200_default_kcfg(int M, int K, int bits, int group_size, int act_group_size, int zero_point, int one_scale, tmac_b200_kcfg *out) {
    if (!out || M <= 0 || K <= 0 || bits < 1 || bits > 4) return fail("default_kcfg: bad argument");
    static const int bms3[] = {192, 384, 576, 768}, bmsx[] = {256, 128, 512, 1024, 320, 640};
    const int *bms = bits == 3 ? bms3 : bmsx;
    const int nb = bits == 3 ? 4 : 6;
    int bm = 0;
    for (int i = 0; i < nb && !bm; ++i)
        if ((M * bits) % bms[i] == 0 && bms[i] % bits == 0) bm = bms[i];
    if (!bm) return fail("default_kcfg: no tile size divides M*bits = " + std::to_string(M * bits));
    const int ags = (act_group_size <= 0 || act_group_size > K) ? K : act_group_size;
    const bool scale_final = one_scale && ags == K;
    const int wgs = one_scale ? K : group_size;
    int kf = 0;
    for (int cand : {8, 16})
        if (!kf && (scale_final || ((cand * 4) % ags == 0 && wgs > 0 && wgs % (cand * 4) == 0))) kf = cand;
    if (!kf) {   // act group wider than 64 K positions: the reference has no candidate; the stream layout only needs kfactor | K/4
        for (int cand : {16, 8})
            if (!kf && (K / 4) % cand == 0) kf = cand;
    }
    if (!kf || (K / 4) % kf) return fail("default_kcfg: no kfactor for this grouping");
    std::memset(out, 0, sizeof *out);
    out->M = M; out->K = K; out->bits = bits; out->bm = bm; out->kfactor = kf; out->simd_n_in = 16; out->simd_n_out = 8;
    out->group_size = one_scale ? (group_size > 0 ? group_size : 128) : group_size; out->act_group_size = ags;
    out->zero_point = zero_point ? 1 : 0; out->one_scale = one_scale ? 1 : 0;
    return 0;
}

// ---- GGUF files (tmac_gguf.h) ----------------------------------------------------------------------------------------

int64_t tmac_b200_gguf_open(const char *path) {
    if (!path) return fail("gguf_open: null path");
    GgufFile *f = new GgufFile();
    if (!f->open(path)) { const std::string e = f->error; delete f; return fail("gguf_open: " + e); }
    std::unique_lock<std::shared_mutex> lk(g_mu);
    const int64_t h = g_next_gguf++;
    g_gguf[h] = f;
    return h;
}
int tmac_b200_gguf_close(int64_t gguf) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    auto it = g_gguf.find(gguf);
    if (it == g_gguf.end()) return fail("gguf_close: bad handle");
    // the file is unmapped: weights uploaded from it stay resident, but their host alias keys (ranges inside the mapping)
    // must not survive -- a later mapping can land on the same addresses and would resolve to the old tensor
    const unsigned char *lo = it->second->base, *hi = lo + it->second->size;
    for (auto &kv : g.res)
        if (kv.second.host_a && kv.second.host_a >= lo && kv.second.host_a < hi) { kv.second.host_a = nullptr; kv.second.host_a_bytes = 0; }
    delete it->second;
    g_gguf.erase(it);
    return 0;
}
static GgufFile *gguf_locked(int64_t gguf) {
    auto it = g_gguf.find(gguf);
    return it == g_gguf.end() ? nullptr : it->second;
}
int tmac_b200_gguf_tensor_count(int64_t gguf) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    GgufFile *f = gguf_locked(gguf);
    return f ? (int)f->tensors.size() : fail("gguf: bad handle");
}
int tmac_b200_gguf_tensor_info(int64_t gguf, int index, struct tmac_b200_gguf_tensor *out) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    GgufFile *f = gguf_locked(gguf);
    if (!f || !out) return fail("gguf: bad handle / null argument");
    if (index < 0 || index >= (int)f->tensors.size()) return fail("gguf: tensor index out of range");
    const GgufTensor &T = f->tensors[index];
    std::memset(out, 0, sizeof *out);
    std::strncpy(out->name, T.name.c_str(), sizeof out->name - 1);
    out->ggml_type = T.type; out->n_dims = T.n_dims;
    for (int d = 0; d < 4; ++d) out->ne[d] = T.ne[d];
    out->offset = T.offset; out->nbytes = T.nbytes;
    out->data = f->data(index);
    return 0;
}
int tmac_b200_gguf_find_tensor(int64_t gguf, const char *name) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    GgufFile *f = gguf_locked(gguf);
    if (!f || !name) return fail("gguf: bad handle / null argument");
    const int i = f->find(name);
    return i >= 0 ? i : fail(std::string("gguf: no tensor named '") + name + "'");
}
// Metadata: integers / bools / floats (as double) and strings.  Return 0, or -1 when the key is absent or of another kind.
int tmac_b200_gguf_meta_number(int64_t gguf, const char *key, double *out) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    GgufFile *f = gguf_locked(gguf);
    if (!f || !key || !out) return fail("gguf: bad handle / null argument");
    auto it = f->meta.find(key);
    if (it == f->meta.end() || it->second.type == 8 || it->second.type == 9) return fail(std::string("gguf: no numeric key '") + key + "'");
    *out = it->second.f;
    return 0;
}
int tmac_b200_gguf_meta_string(int64_t gguf, const char *key, char *dst, size_t cap) {
    std::unique_lock<std::shared_mutex> lk(g_mu);
    GgufFile *f = gguf_locked(gguf);
    if (!f || !key || !dst || !cap) return fail("gguf: bad handle / null argument");
    auto it = f->meta.find(key);
    if (it == f->meta.end() || it->second.type != 8) return fail(std::string("gguf: no string key '") + key + "'");
    std::strncpy(dst, it->second.s.c_str(), cap - 1); dst[cap - 1] = 0;
    return (int)it->second.s.size();
}
// Upload one quantised linear of the file (I1..I4, Q4_0, TQ1_0, TQ2_0; 2-D) through the typed transform; the kcfg for its
// shape must be registered (tmac_b200_load_kcfg_file).  The mapped file region serves as the host alias of I-type tensors.
int64_t tmac_b200_gguf_load_tensor(int64_t gguf, int index, struct tmac_tensor_extra_b200 *extra) {
    const uint8_t *data; int type, ne0, ne1; uint64_t nbytes;
    {
        std::unique_lock<std::shared_mutex> lk(g_mu);
        GgufFile *f = gguf_locked(gguf);
        if (!f) return fail("gguf: bad handle");
        if (index < 0 || index >= (int)f->tensors.size()) return fail("gguf: tensor index out of range");
        const GgufTensor &T = f->tensors[index];
        if (T.n_dims != 2) return fail("gguf_load_tensor: '" + T.name + "' is not a matrix");
        data = f->data(index); type = T.type; ne0 = (int)T.ne[0]; ne1 = (int)T.ne[1]; nbytes = T.nbytes;
    }
    const int bits = ggml_tmac_get_type_bits(type);
    if (!bits) return fail("gguf_load_tensor: ggml type " + std::to_string(type) + " is not a T-MAC type");
    uint64_t need;
    if (ggml_block_elems(type)) {
        need = (uint64_t)ne1 * (ne0 / ggml_block_elems(type)) * ggml_block_bytes(type);
        tmac_b200_kcfg c;   // block types fix their grouping themselves: without a tuned kcfg the reference's default tiling will do
        if (tmac_b200_find_kcfg(ne1 * bits, ne0, bits, &c) != 0) {
            const int E = ggml_block_elems(type);
            if (tmac_b200_default_kcfg(ne1, ne0, bits, E, E == 32 ? 32 : 64, 0, 0, &c) != 0 || tmac_b200_register_kcfg(&c) != 0) return -1;
        }
    } else need = ggml_tmac_b200_get_nbytes(ne0, ne1, bits);
    if (need == 0) return -1;                      // no kcfg for the shape (message set by the lookup)
    if (nbytes < need) return fail("gguf_load_tensor: tensor data is shorter than its type and shape require");
    return ggml_tmac_b200_transform_tensor_typed((void *)data, type, ne0, ne1, extra);
}

}  // extern "C"
