// engine.cu -- C-ABI implementation: handle, device workspace, block plan (the scheduler side of
// DBSLMMFIT::est, reference scr/dbslmmfit.cpp:56-244) and the launch sequence of one fit.
//
// Host work per fit: group the blocks into batches (size classes; upload regions when the panel
// streams in with the call), lay the blocks out in device memory (int8 code rows, one row-major
// FP64 matrix per block), build the tile / panel work lists, ship everything in ONE pinned blob,
// launch decode -> gram -> (per fold, per batch on its own stream) cholesky steps -> back
// substitution, and read the betas back.  With fit_args.bed the panel upload is cut along the
// batches and overlaps all of that; with fit_args.quadform_out the solve is replaced by the
// `valid` tool's quadratic form.  No CPU arithmetic on the data path: without a CUDA device every
// entry point fails.
#include <nvtx3/nvToolsExt.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include <cudaTypedefs.h>
#include "../../include/dbslmm_b200.h"
#include "common.cuh"
#include "kernels.h"
#include "hostpool.hpp"

using namespace dbslmm;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 16 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

constexpr int kNumClasses = 4;                 // timing slots reported per size class (dbslmm_b200_timing.class_ms)
constexpr int kBulkMaxPanels = 16;             // blocks up to 16 panels (m <= 1024) are "bulk": one-CTA back substitution

struct StepList {
    int32_t diag_off, n_diag, panel_off, n_panel, group_base, n_groups, nsl;
    int32_t n_first;    // leading panel items that are macro tile 0 of their block (one CTA each when the diagonal tile is fused)
    int32_t defer;      // the diagonal tile of panel k+1 is NOT factored at the end of this step but first thing in step k+1
};

// A batch = the blocks that run one Cholesky step loop together on one stream.  With the reference panel resident
// (load_bed) there is one batch per size class.  When the panel streams in from host memory inside the fit
// (fit_args.bed), batches are also the upload units: big classes first, the bulk class cut into sub-batches, so a
// batch's decode -> Gram -> factorisation starts as soon as ITS rows have crossed PCIe.
constexpr int kMaxBatches = 12;
// Rough device rates for the upload-order rule of the streaming fit (make_batches) and nothing else -- measured on C3
// (DESIGN.md 4): a panel step of a chain-bound block ~45 us, the bulk factorisation ~23 Tflop/s, the Gram ~1.2 Pop/s.
constexpr double kChainStepUs = 45.0;
constexpr double kBulkFlopPerUs = 23.0e6;
constexpr double kGramOpsPerUs = 1.2e9;
struct Batch {
    int cls = 0;                          // size class (timing slot)
    bool big = false;                     // some member has mp > 1024: cluster back substitution
    int32_t tile_rows = 128;              // rows per Cholesky panel item (128: 256-thread CTAs, 64: 128-thread CTAs, three per SM)
    int32_t ord_off = 0, ord_n = 0;       // members = order[ord_off, ord_off + ord_n)
    int64_t grow0 = 0, grow1 = 0;         // SNP rows of the members (contiguous only in the streaming layout)
    int32_t tile0 = 0, tile1 = 0;         // range of the one-plane Gram tile list (128 x 128 tiles)
    int32_t mtile0 = 0, mtile1 = 0;       // range of the four-plane Gram tile list (64-row x 128-column tiles)
    int32_t ptile0 = 0, ptile1 = 0;       // range of the one-plane kernels' tile RECORD list (128 x 128 tiles, or 256 x 256 super tiles for the CTA-pair kernel)
    std::vector<StepList> steps;          // per panel step
    int64_t scratch_off = 0;              // split-K scratch region (doubles)
};

struct Plan {
    int32_t n_blocks = 0;
    int64_t n_snp_rows = 0;       // total SNP rows (sum m)
    int64_t n_code_rows = 0;      // int8 code rows: per block m genotype rows followed by m call-mask rows
    int64_t mat_doubles = 0;      // total doubles of all block matrices
    int64_t tot_s = 0, tot_l = 0;
    int32_t max_mp = 0;
    std::vector<BlockDesc> blocks;
    std::vector<int32_t> order;                       // concatenated batch member lists (big classes first)
    std::vector<int32_t> code_layout;                 // block sizes in code-row order: which code rows are genotype rows, which mask rows
    std::vector<Batch> batches;
    bool streaming = false;                           // layout in batch order (else block-index order)
    bool chain_bound = false;                         // the big classes' dependency chains outlast the bulk's throughput time (make_batches)
    std::vector<int32_t> up_order;                    // streaming: the order in which the batches' rows cross PCIe
    int32_t n_tiles_plain = 0, n_tiles_miss = 0, n_tiles_pair = 0;
    int64_t scratch_doubles = 0;
    int32_t n_groups = 0;                             // split-K groups (one arrival counter each)
    int32_t n_test = 0;                               // selected test individuals (variance side channel), 0 = off
    // blob layout (byte offsets inside the plan blob, identical on host and device)
    size_t o_blocks = 0, o_rowsrc = 0, o_crow = 0, o_mrow = 0, o_z = 0, o_tiles_plain = 0, o_tiles_miss = 0, o_tiles_pair = 0, o_order = 0,
           o_diag = 0, o_panel = 0, o_lmaps = 0, blob_bytes = 0;
    const void* lmaps_base = nullptr;                 // L buffer the per-block tensor maps in the blob were encoded for
    uint64_t fingerprint = 0;                         // of the inputs the plan was built from (FLAG_PLAN_CACHED re-use check)
    double gram_ops = 0, solve_flops = 0, decode_bytes = 0;
    bool valid = false;
};

}  // namespace

struct dbslmm_b200_handle {
    int device = 0;
    int n_sm = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t b_stream[kMaxBatches] = {};    // one Cholesky stream per batch, priority falling with the batch index
    cudaEvent_t ev[8] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[kMaxBatches] = {}, ev_cend[kMaxBatches] = {};
    cudaStream_t up_stream = nullptr;    // streaming fit: class-ordered panel upload
    cudaEvent_t ev_up[kMaxBatches] = {}, ev_gram[kMaxBatches] = {}, ev_blob = nullptr;
    std::string err;
    bool fuse_diag = true;               // panel step k also factors the diagonal tile of panel k+1 (one launch per step)
    bool stream_bed = true;              // fit_args.bed: overlap the panel upload with the fit (else upload, then fit)
    // size classes of the Cholesky step loops, by #panels (upper bounds, ascending; the last class is unbounded).
    // Each class (batch) has its own stream: the step loops interleave and fill each other's thin last steps.
    std::vector<int> cls_bounds = {8, 16, 32};
    int splitk_max = 16, splitk_min_blocks = 2;  // split-K: at most this many slices, each at least this many 64-deep K blocks
    // programmatic dependent launch for chain-bound batches (0 = never; DBSLMM_B200_PDL=0.8 turns it on for batches
    // whose chain rivals the fit's throughput time).  Measured on an 8-GPU shard: the longest chain shrinks by 4 %, but
    // the waiting CTAs hold SM slots the bulk batches need, and the streaming fit gets slower -- off by default.
    double pdl_ratio = 0.0;
    int defer_max_ctas = -1;                     // steps with at most this many CTAs take their diagonal tile first (see StepList); -1: one wave of panel CTAs
    // Panel items of 64 rows (128-thread CTAs, three per SM; DBSLMM_B200_TILE64: 2 = everywhere (default), 1 = only for the
    // batches of bulk blocks (<= 16 panels), 0 = 128-row items, 256-thread CTAs, two per SM).  Measured on C3, one GPU:
    // factorisation 13.7 / 13.35 / 13.0 ms for 0 / 1 / 2 -- a third independent instruction stream per SM and fewer idle
    // warps in partially filled items outweigh the slower 128-thread diagonal-tile code even in the chain-bound classes.
    int tile64_mode = 2;
    // The back substitution writes the betas straight into the pinned result buffer (mapped host memory: 9 MB spread over the
    // whole fit) instead of a device buffer that is copied back when everything is done (0.47 ms at C3, all of it exposed).
    bool zero_copy_beta = true;
    int next_pf = 1;                             // panel kernel (64-row items): the next item's first chunk is issued during the epilogue (DBSLMM_B200_NEXT_PF=0: off)
    int l2_pf = 0;                               // panel kernel: L2 tensor prefetch distance in 16-wide K chunks (0 = off: measured 13.0 ms without, 13.1 with 2 or 4)
    // panel step kernel: TMA/mbarrier pipeline (default) or the cp.async version (DBSLMM_B200_PANEL=legacy)
    int upload_bulk_first = 1;                   // streaming fit: bulk regions sent before the big classes (see make_batches)
    bool upload_auto = true;                     // ... only when the fit is throughput-bound and the first region is small (make_batches); an explicit DBSLMM_B200_UPLOAD_BULK_FIRST switches the rule off
    // streaming fit: the bulk is cut into this many regions (upload units).  The FIRST region goes out before the plan is
    // built and the plan blob queues behind it on the copy engine, so it should take about as long to cross PCIe as the
    // plan takes to build: with 4 regions (138 MB each at C3) the blob arrived 4.1 ms after the call started, with 6
    // (92 MB) it arrives at ~2.7 ms, and the first decode starts that much earlier.
    int n_regions = 6;
    int region_min_blocks = 256;                 // ... when the bulk has at least this many blocks (and 100,000 SNPs), else it is ONE region (DBSLMM_B200_REGION_MIN_BLOCKS)
    double first_region = 0.3;                   // SNP share of the FIRST bulk region relative to an equal share (< 1: a small first region crosses PCIe sooner, so the first decode / Gram / Cholesky start sooner; DBSLMM_B200_FIRST_REGION)
    double preplan_mb = 60.0;                    // ... and at most this much panel data is queued ahead of the plan blob
    // correlation builder for blocks without missing calls: the int8-row kernel fed by the decoder (default), or the fused
    // unpack + Gram from packed 2-bit rows (DBSLMM_B200_GRAM=packed).  Measured on C3 / C5: 1.8 / 10.8 ms against 3.9 / 34.7 ms --
    // expanding the operands in shared memory (8 unpack warps, generic-proxy stores + fence.proxy.async per K step) costs
    // more than the L2 traffic it saves, so the fused kernel stays an experiment.
    bool gram_packed = false;
    int gram_hint = 0;                          // DBSLMM_B200_GRAM_HINT: tuning bits of GramArgs.hint
    bool gram_pair = false;                     // DBSLMM_B200_GRAM=pair: one-plane Gram by CTA pairs (256 x 256 super tiles, half the L2 -> SM operand traffic; 1.8 ms against 1.5 ms at C3: its tile order re-reads the code rows from DRAM, see gram.cu)
    bool panel_tma = true;
    int tpc_max = 4, tpc_waves = 2;              // items per CTA: at most tpc_max, and only while a step keeps >= tpc_waves waves of CTAs
    int tmap_perm = -1;                          // 1: 4-D row-permuting tensor maps, 0: plain 2-D maps (driver refused), -1: not probed yet
    // reference panel
    DevBuf bed, stats;
    PinBuf h_stats;                      // per-SNP statistics, filled asynchronously by load_bed
    cudaEvent_t ev_bed = nullptr;        // completes when the panel, its statistics and their host copy have landed
    bool bed_pending = false;
    bool stats_valid = false;            // `stats` / `h_stats` describe the resident panel (a streaming fit skips them)
    std::vector<int32_t> miss_flags;     // per-block "has missing calls" of the last fit (computed on the device, copied back)
    int64_t n_snp = 0;
    int32_t n_ref = 0, pitch = 0, n_pad = 0;
    // workspace
    DevBuf codes, sigma, lbuf, rowN, rowS, rowR, planblob, beta, status, intQ, intA, intN, scratch, counters, wbuf, vbed, vstats, vwork, dflag, dirty, bflags, packed, rowC, rowmap;
    // validation panel of the scoring step, announced by dbslmm_b200_score_prefetch: uploaded in the shadow of the next fit
    const uint8_t* val_host = nullptr;
    int64_t val_n_snp = 0;
    int32_t val_n = 0;
    bool val_announced = false, val_inflight = false;
    cudaEvent_t ev_val = nullptr;
    // streaming scorer (dbslmm_b200_score_stream): pinned staging ring, device chunk slots, per-call work buffer
    PinBuf s_pin[3];
    DevBuf s_dev[2], s_work;
    // LD scores (dbslmm_b200_ldscore): row statistics, segment code rows + dirty map, decoder scratch, partial slots, reduction
    DevBuf ld_stats, ld_codes, ld_dirty, ld_work, ld_slots, ld_red;
    PinBuf ld_pin[2], ld_roff;           // SNP pairs (dbslmm_b200_ld_pairs): the two pinned pair buffers the sink reads, row offsets
    cudaEvent_t ev_pin_free[3] = {}, ev_copied[2] = {}, ev_slot_free[2] = {};
    std::vector<cudaEvent_t> ev_chunk;   // 4 timing events per chunk (copy begin / end, kernels begin / end), grow-only
    size_t dirty_rows = 0;               // code rows the dirty map covers
    int32_t dirty_n_ref = 0;             // ... for this panel width (another width = another default mask pattern)
    const void* dirty_codes = nullptr;   // ... and this code buffer
    std::vector<int32_t> dirty_layout;   // ... and this code-row layout (Plan::code_layout)
    PinBuf h_blob, h_out;
    Plan plan;

    int32_t last_flags = 0, last_solver = 0, last_nfolds = 0;
    bool last_quad = false;                   // the last fit computed quadform_out: nothing was factored
    PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
};

namespace {

int fail(dbslmm_b200_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    return code;
}
#define CU_TRY(h, expr)                                                                             \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            return fail(h, (_e == cudaErrorMemoryAllocation) ? DBSLMM_B200_ERR_NOMEM : DBSLMM_B200_ERR_CUDA, \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                        \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// memcpy split over up to four host threads (large result vectors only)
inline void par_memcpy(void* dst, const void* src, size_t bytes) {
    const size_t kMin = (size_t)2 << 20;
    const int nthr = (int)std::min<size_t>(4, bytes / kMin);
    if (nthr <= 1) { std::memcpy(dst, src, bytes); return; }
    std::vector<std::thread> th;
    const size_t chunk = (bytes / nthr + 63) & ~(size_t)63;
    for (int t = 1; t < nthr; ++t) {
        const size_t o = chunk * t, n = (t == nthr - 1) ? bytes - o : chunk;
        th.emplace_back([=]() { std::memcpy((char*)dst + o, (const char*)src + o, n); });
    }
    std::memcpy(dst, src, chunk);
    for (std::thread& x : th) x.join();
}

// DBSLMM_B200_TRACE=1: host-side wall-clock marks of one fit on stderr (tuning aid)
// The process-wide pool of host worker threads (hostpool.hpp): plan building, tensor maps, the row-range scan.
HostPool& host_pool() {
    static HostPool pool;
    return pool;
}

// Phase marks of a fit: NVTX markers always (free without a profiler attached; they line the phases up with the kernels in
// an Nsight timeline), wall-clock lines on stderr with DBSLMM_B200_TRACE=1.
struct Trace {
    bool on;
    std::chrono::steady_clock::time_point t0;
    Trace() : on(std::getenv("DBSLMM_B200_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) const {
        nvtxMarkA(what);
        if (on) std::fprintf(stderr, "[dbslmm_b200 trace] %-28s %8.3f ms\n", what,
                             std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
};

// ------------------------------------------------------------------------------------------
// Plan construction (host): the block scheduler's bookkeeping
// ------------------------------------------------------------------------------------------
// Step 1: block sizes, size classes, batches and the block order.  Cheap (O(n_blocks)), so the streaming fit can
// start its class-ordered uploads before the rest of the plan exists.
int make_batches(dbslmm_b200_handle* h, const dbslmm_b200_fit_args* a, Plan& P, bool streaming) {
    const int nb = a->n_blocks;
    P = Plan();
    P.n_blocks = nb;
    P.streaming = streaming;
    P.blocks.resize(nb);
    P.tot_s = a->s_off[nb];
    P.tot_l = a->l_off ? a->l_off[nb] : 0;
    const std::vector<int>& bounds = h->cls_bounds;
    const int nc = (int)bounds.size() + 1;
    std::vector<std::vector<int32_t>> by_cls((size_t)nc);
    double chain_us = 0.0, bulk_us = 0.0;
    for (int b = 0; b < nb; ++b) {
        const int ms = a->s_off[b + 1] - a->s_off[b];
        const int ml = a->l_off ? a->l_off[b + 1] - a->l_off[b] : 0;
        if (ms < 0 || ml < 0) return fail(h, DBSLMM_B200_ERR_ARG, "CSR offsets must be non-decreasing");
        BlockDesc& d = P.blocks[b];
        d.m = ms + ml;
        d.ms = ms;
        d.mp = (d.m + 7) / 8 * 8;
        d.ld = d.mp;
        const int K = (d.mp + 63) / 64;
        int c = 0;
        while (c < nc - 1 && K > bounds[c]) ++c;
        by_cls[c].push_back(b);          // m == 0 blocks land in class 0: no tiles, no steps, they only exist
        const double m = (double)d.m;
        if (K > kBulkMaxPanels) chain_us = std::max(chain_us, kChainStepUs * (double)(K + 1));
        else bulk_us += (m * m * m / 3.0 + 2.0 * m * m) / kBulkFlopPerUs + (double)h->n_pad * m * (m + 1.0) / kGramOpsPerUs;
    }
    // CHAIN-bound fit (typically one rank's shard of a multi-GPU run: a 3,000-SNP block is 47 serial panel steps next to a
    // bulk of a millisecond or two): the big classes' dependency chains are the critical path, the bulk runs in their shadow.
    // (Measured and dropped: padding the bulk batches' shared-memory request so that only two of their CTAs fit on an SM and
    // the third slot stays free for the chains' CTAs -- the bulk slowed down as expected, 1.92 -> 2.09 ms, but a chain step
    // stayed at 61 us against 42 us alone: the chains do not wait for CTA slots, they share the SMs' FP64 pipes.)
    P.chain_bound = chain_us > bulk_us;
    P.order.reserve(nb);
    auto add_batch = [&](std::vector<int32_t>& sub, int cls) {
        if (sub.empty()) return;
        Batch B;
        B.cls = cls;
        B.ord_off = (int32_t)P.order.size();
        std::stable_sort(sub.begin(), sub.end(), [&](int x, int y) { return P.blocks[x].m > P.blocks[y].m; });
        P.order.insert(P.order.end(), sub.begin(), sub.end());
        B.ord_n = (int32_t)sub.size();
        B.big = P.blocks[sub[0]].mp > 64 * kBulkMaxPanels;
        P.batches.push_back(std::move(B));
    };
    if (!streaming) {
        for (int c = nc - 1; c >= 0; --c) add_batch(by_cls[c], c);
        return DBSLMM_B200_OK;
    }
    // Streaming: the two big classes first (few, scattered blocks with the longest dependency chains), then the
    // bulk (classes 1 and 0 together) cut into REGIONS of consecutive blocks with equal SNP counts: a region is one
    // contiguous stretch of the .bed (minus the big blocks inside it), so its upload is a handful of large copies,
    // and its factorisation starts while the next region is still crossing PCIe.  Regions alternate between the two
    // bulk streams so the thin last steps of one overlap the first steps of the next.
    std::vector<int32_t> bulk;
    for (int c = nc - 1; c >= 0; --c) {
        const bool is_bulk = (c < nc - 1) && bounds[c] <= kBulkMaxPanels;
        if (!is_bulk && (int)P.batches.size() < kMaxBatches - h->n_regions) { add_batch(by_cls[c], c); continue; }
        const size_t n0 = bulk.size();
        bulk.insert(bulk.end(), by_cls[c].begin(), by_cls[c].end());
        std::inplace_merge(bulk.begin(), bulk.begin() + n0, bulk.end());
    }
    int64_t tot = 0;
    for (int b : bulk) tot += P.blocks[b].m;
    const int nsub = ((int)bulk.size() >= h->region_min_blocks && tot >= 100000) ? h->n_regions : 1;
    size_t i = 0;
    int64_t acc = 0;
    // region sb ends at SNP count `target`: equal shares, except that the first region may be a fraction of a share
    const double share0 = (nsub > 1) ? h->first_region / (double)nsub : 1.0;
    for (int sb = 0; sb < nsub; ++sb) {
        const int64_t target = (nsub > 1) ? (int64_t)((double)tot * (share0 + (1.0 - share0) * (double)sb / (double)(nsub - 1))) : tot;
        std::vector<int32_t> sub;
        while (i < bulk.size() && (sb == nsub - 1 || acc < target)) { acc += P.blocks[bulk[i]].m; sub.push_back(bulk[i]); ++i; }
        add_batch(sub, (sb & 1) ? 0 : 1);
    }
    // Upload order.  The batches are NUMBERED big classes first (their streams get the highest priorities: longest
    // dependency chains), but the fit as a whole is throughput-bound on the bulk, and the big classes' chains (about half the
    // fit) fit in the bulk's shadow: sending `upload_bulk_first` bulk regions ahead of the big classes gets the GPU busy
    // earlier.  0 = big classes first (the numbering order).
    const int nbt = (int)P.batches.size();
    int n_big = 0;
    while (n_big < nbt && P.batches[n_big].cls > 1) ++n_big;          // bulk regions carry class 0 / 1
    int lead = std::max(0, std::min(h->upload_bulk_first, nbt - n_big));
    if (h->upload_auto && lead > 0 && n_big > 0) {
        // ... unless the fit is chain-bound (above) or the first bulk region is too big to send ahead of the plan blob (few
        // bulk blocks are ONE region): everything queued on the copy engine ahead of the big classes -- and ahead of the plan
        // blob, which follows the pre-plan uploads -- then delays the whole fit (rank 0 of 8 at C3: 5.1-5.7 -> 4.5-4.8 ms per call, profiles/r05u_shard_upload_order.txt).
        double first_mb = 0.0;
        for (int j = 0; j < P.batches[n_big].ord_n; ++j)
            first_mb += (double)P.blocks[P.order[P.batches[n_big].ord_off + j]].m * (double)h->pitch / 1.0e6;
        if (P.chain_bound || first_mb > h->preplan_mb) lead = 0;
    }
    for (int i = 0; i < lead; ++i) P.up_order.push_back(n_big + i);
    for (int i = 0; i < n_big; ++i) P.up_order.push_back(i);
    for (int i = n_big + lead; i < nbt; ++i) P.up_order.push_back(i);
    return DBSLMM_B200_OK;
}

// A list that is built in place inside the pinned plan blob (no temporary vector -- a fresh 5 MB vector per fit costs
// more in page faults than the list costs to fill -- and no copy into the blob afterwards).
// Non-temporal stores for the O(#SNPs) part of the pinned plan blob.  The blob is written by several host threads and read
// once, by the GPU's copy engine: with ordinary stores its lines sit dirty in the caches of whichever cores ran the fill
// threads, and the H2D copy then crawls at 13-17 GB/s instead of 54 (measured: tools/h2d_probe.py, 28 MB written by one
// thread 0.55 ms, by eight threads 2.2-3.0 ms; in the streaming fit the blob arrived 1.6 ms after the first panel region).
#if defined(__x86_64__)
static bool g_nt = std::getenv("DBSLMM_B200_NT") == nullptr || std::atoi(std::getenv("DBSLMM_B200_NT")) != 0;      // DBSLMM_B200_NT=0: ordinary stores
inline void nt_store(uint32_t* p, uint32_t v) { if (g_nt) _mm_stream_si32(reinterpret_cast<int*>(p), (int)v); else *p = v; }
inline void nt_store(int32_t* p, int32_t v) { if (g_nt) _mm_stream_si32(reinterpret_cast<int*>(p), v); else *p = v; }
inline void nt_store(double* p, double v) { if (!g_nt) { *p = v; return; } long long b; std::memcpy(&b, &v, 8); _mm_stream_si64(reinterpret_cast<long long*>(p), b); }
template <class T>
inline void nt_copy(T* dst, const T& v) {          // records of the plan lists: 4 bytes or a multiple of 16 (16-byte aligned)
    if (!g_nt) { *dst = v; return; }
    if constexpr (sizeof(T) % 16 == 0) {
        const __m128i* src = reinterpret_cast<const __m128i*>(&v);
        for (size_t i = 0; i < sizeof(T) / 16; ++i) _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + i, _mm_loadu_si128(src + i));
    } else {
        static_assert(sizeof(T) == 4, "plan list records are 4 bytes or a multiple of 16");
        int b; std::memcpy(&b, &v, 4); _mm_stream_si32(reinterpret_cast<int*>(dst), b);
    }
}
inline void nt_fence() { _mm_sfence(); }
#else
template <class T>
inline void nt_copy(T* dst, const T& v) { *dst = v; }
inline void nt_store(uint32_t* p, uint32_t v) { *p = v; }
inline void nt_store(int32_t* p, int32_t v) { *p = v; }
inline void nt_store(double* p, double v) { *p = v; }
inline void nt_fence() {}
#endif

template <class T>
struct BlobList {
    T* p = nullptr;
    size_t n = 0, cap = 0;
    void push_back(const T& v) { if (n < cap) nt_copy(&p[n], v); ++n; }      // (non-temporal, see nt_store) overflow is detected by the caller (n > cap)
    size_t size() const { return n; }
};

// Step 2: device layout, Gram tiles, Cholesky step lists, the pinned blob.
// Every block gets m genotype code rows followed by m call-mask code rows; which blocks really have missing calls is
// found out on the device (decoder counts -> block_flags_kernel), so the plan never looks at the panel.
int build_plan(dbslmm_b200_handle* h, const dbslmm_b200_fit_args* a, Plan& P, const Trace* tr = nullptr) {
    const int nb = a->n_blocks;
    int n_test = 0;
    if (a->test_bed) for (int i = 0; i < a->test_n_total; ++i) n_test += (a->test_indicator[i] != 0);
    P.n_test = n_test;
    // build_plan may run twice on the same batches (speculative no-missing plan, then the real flags): start the
    // accumulated quantities from zero every time -- the split-K scratch offsets are derived from them
    P.scratch_doubles = 0;
    P.gram_ops = P.solve_flops = 0.0;
    P.max_mp = 0;
    const int64_t n_snp = h->n_snp;
    int64_t goff = 0, croff = 0, moff = 0;
    // layout order: block index (resident panel) or batch order (streaming: a batch's rows are one range)
    std::vector<int32_t> lay(nb);
    if (P.streaming) lay = P.order; else std::iota(lay.begin(), lay.end(), 0);
    P.code_layout.clear();
    for (int b : lay) {
        BlockDesc& d = P.blocks[b];
        P.code_layout.push_back(d.m);
        const int ms = d.ms, ml = d.m - d.ms;
        d.goff = (int32_t)goff;
        d.croff = (int32_t)croff;
        d.moff = moff;
        d.out_s = a->s_off[b];
        d.out_l = a->l_off ? a->l_off[b] : 0;
        d.nrows = d.mp + 8 + n_test * (1 + (ml > 0 ? 1 : 0));       // test-genotype rows of the variance side channel
        (void)ms;
        d.has_missing = 0;            // (unused: the flag lives on the device)
        goff += d.m;
        croff += 2 * (int64_t)d.m;
        if (d.m > 0) moff += align_up((size_t)d.nrows * d.ld, 16);
        P.max_mp = std::max(P.max_mp, d.mp);
        const double m = d.m;
        P.gram_ops += (double)h->n_pad * m * (m + 1.0);   // one plane; 2 ops per MAC, lower triangle (x4 for blocks with missing calls, added after the fit)
        P.solve_flops += m * m * m / 3.0 + 2.0 * m * m;
    }
    if (goff > INT32_MAX || croff > INT32_MAX) return fail(h, DBSLMM_B200_ERR_ARG, "too many SNP rows for one call");
    P.n_snp_rows = goff;
    P.n_code_rows = croff;
    P.mat_doubles = moff;
    // .bed row read + what the packer (2-bit rows, n_pad / 4 bytes) or the decoder (int8 rows) writes; mask rows: see fit
    P.decode_bytes = (double)goff * ((double)h->pitch + (h->gram_packed ? (double)h->n_pad / 4.0 : (double)h->n_pad));

    // ---- the per-SNP part of the blob (block descriptors, .bed row / code row maps, z-scores) has a size that is known
    // now: it is filled by a few host threads WHILE this thread builds the tile and step lists, which follow it in the blob
    size_t o = 0;
    auto place = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    P.o_blocks = place(sizeof(BlockDesc) * (size_t)nb);
    P.o_rowsrc = place(sizeof(uint32_t) * (size_t)goff);
    P.o_crow = P.o_mrow = 0;      // (the code-row / mask-row maps are a function of the layout: written on the device, fill_rowmaps)
    P.o_z = place(sizeof(double) * (size_t)goff);
    size_t n_t1 = 0, n_t2 = 0, n_t3 = 0, n_steps_tiles = 0, n_diag_max = 0;
    for (int b = 0; b < nb; ++b) {
        const BlockDesc& d = P.blocks[b];
        const size_t nt = (size_t)(d.mp + 127) / 128, nt64 = (size_t)(d.mp + 63) / 64;
        n_t1 += nt * (nt + 1) / 2;
        n_t2 += nt64 * (nt64 / 2 + 1);
        const size_t np = h->gram_pair ? (size_t)(d.mp + 255) / 256 : nt;
        n_t3 += np * (np + 1) / 2;
        const int K = (d.mp + 63) / 64;
        n_diag_max += (size_t)K;
        for (int k = 0; k < K; ++k) {
            const int wk = std::min(64, d.mp - 64 * k);
            n_steps_tiles += (size_t)((d.nrows - (64 * k + wk) + 63) / 64);      // 64-row items (the finer of the two shapes)
        }
    }
    // upper bound of the list part: a split-K step has at most max(#tiles, 2 n_sm) items
    const size_t n_panel_max = n_steps_tiles + (size_t)3 * h->n_sm * kMaxBatches * (size_t)(P.max_mp / 64 + 2);
    // ... and so are the places of the lists: the two Gram tile lists and the diagonal items have exact sizes, the panel
    // items (split-K makes their number known only afterwards) go last
    if (!h->gram_packed) n_t1 = 0;            // the 128 x 128 GramTile list feeds only the packed-row kernel; the others read records
    P.o_tiles_plain = place(sizeof(GramTile) * n_t1);
    P.o_tiles_miss = place(sizeof(GramTile) * n_t2);
    P.o_tiles_pair = place(sizeof(TileRec) * n_t3);
    P.o_order = place(sizeof(int32_t) * (size_t)nb);
    P.o_diag = place(sizeof(int32_t) * n_diag_max);
    P.o_lmaps = place(sizeof(CUtensorMap) * (size_t)nb);     // filled by encode_lmaps once the L buffer exists
    P.o_panel = place(0);
    if (h->h_blob.ensure(o + sizeof(int4) * n_panel_max + 512) != cudaSuccess) return fail(h, DBSLMM_B200_ERR_NOMEM, "pinned plan buffer");
    struct { uint8_t* p; uint8_t* data() const { return p; } } blob{(uint8_t*)h->h_blob.p};
    std::memcpy(blob.data() + P.o_blocks, P.blocks.data(), sizeof(BlockDesc) * (size_t)nb);
    uint32_t* rs = reinterpret_cast<uint32_t*>(blob.data() + P.o_rowsrc);
    double* z = reinterpret_cast<double*>(blob.data() + P.o_z);
    // every helper task below references this frame: the guard waits for all of them on every way out
    TaskGroup g_fill, g_tiles, g_lists;
    struct PoolGuard { HostPool& p; TaskGroup& a; TaskGroup& b; TaskGroup& c; ~PoolGuard() { p.wait(a); p.wait(b); p.wait(c); } } pool_guard{host_pool(), g_fill, g_tiles, g_lists};
    std::atomic<int> fill_bad{0};
    // per-SNP rows (source .bed row, SNP-row index, z-score): the only O(#SNPs) part of the plan, filled by a few
    // host threads, each owning a contiguous range of blocks; the .bed row range check rides along
    {
        static const int fill_max = std::getenv("DBSLMM_B200_FILL_THREADS") ? std::max(1, std::atoi(std::getenv("DBSLMM_B200_FILL_THREADS"))) : 12;      // (the pool also runs two tile-list tasks and one step-list task per batch)
        const int nthr = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)fill_max, (int64_t)std::thread::hardware_concurrency(), goff / 65536}));
        auto fill = [&, rs, z](int b0, int b1) {
            int oob = 0;
            for (int b = b0; b < b1; ++b) {
                const BlockDesc& d = P.blocks[b];
                const int32_t* sp = a->s_pos + a->s_off[b];
                const double* sz = a->s_z + a->s_off[b];
                uint32_t* rsb = rs + d.goff;
                double* zb = z + d.goff;
                for (int j = 0; j < d.ms; ++j) {
                    const int32_t p = sp[j];
                    oob |= (p < 0) | (p >= n_snp);
                    nt_store(rsb + j, (uint32_t)p); nt_store(zb + j, sz[j]);
                }
                if (d.m > d.ms) {
                    const int32_t* lp = a->l_pos + a->l_off[b];
                    const double* lz = a->l_z + a->l_off[b];
                    for (int j = d.ms; j < d.m; ++j) {
                        const int32_t p = lp[j - d.ms];
                        oob |= (p < 0) | (p >= n_snp);
                        nt_store(rsb + j, (uint32_t)p); nt_store(zb + j, lz[j - d.ms]);
                    }
                }
            }
            nt_fence();
            if (oob) fill_bad.store(1);
        };
        if (nthr == 1) fill(0, nb);
        else {
            int b0 = 0;
            for (int t = 0; t < nthr; ++t) {
                // cut at equal SNP counts (block-index order; goff is monotone only in the resident layout, so count)
                int b1 = b0;
                int64_t acc = 0;
                const int64_t share = (goff + nthr - 1) / nthr;
                while (b1 < nb && (t == nthr - 1 || acc < share)) acc += P.blocks[b1++].m;
                host_pool().submit(g_fill, [fill, b0, b1]() { fill(b0, b1); });      // (by value: `fill` leaves scope before the tasks run)
                b0 = b1;
            }
        }
    }
    if (tr) tr->mark("  plan: layout");
    // Gram tiles in batch order, big blocks first inside a batch: the lower triangle as 128 x 128 tiles for the one-plane
    // kernel and as 64-row x 128-column tiles for the four-plane kernel (every block is in both lists; the kernels pick
    // their blocks by the device-side flag)
    // (built by a helper thread while this thread builds the Cholesky step lists: the two touch different fields)
    BlobList<GramTile> tiles_plain, tiles_miss;
    BlobList<TileRec> tiles_pair;
    tiles_pair.p = reinterpret_cast<TileRec*>(blob.data() + P.o_tiles_pair); tiles_pair.cap = n_t3;
    const bool want_plain = h->gram_packed;
    const int rec_edge = h->gram_pair ? 256 : 128;
    tiles_plain.p = reinterpret_cast<GramTile*>(blob.data() + P.o_tiles_plain); tiles_plain.cap = n_t1;
    tiles_miss.p = reinterpret_cast<GramTile*>(blob.data() + P.o_tiles_miss); tiles_miss.cap = n_t2;
    // The places of every batch's tiles follow from block sizes alone (serial, arithmetic only); the entries themselves are
    // written by one pool task per batch and list while this thread builds the Cholesky step lists.
    {
        size_t c_plain = 0, c_miss = 0, c_rec = 0;
        for (Batch& B : P.batches) {
            B.tile0 = (int32_t)c_plain;
            B.mtile0 = (int32_t)c_miss;
            B.ptile0 = (int32_t)c_rec;
            B.grow0 = INT64_MAX;
            B.grow1 = 0;
            for (int i = 0; i < B.ord_n; ++i) {
                const BlockDesc& d = P.blocks[P.order[B.ord_off + i]];
                if (d.m == 0) continue;
                B.grow0 = std::min<int64_t>(B.grow0, d.goff);
                B.grow1 = std::max<int64_t>(B.grow1, (int64_t)d.goff + d.m);
                const size_t nt = (size_t)(d.mp + 127) / 128, nt64 = (size_t)(d.mp + 63) / 64, np = (size_t)(d.mp + rec_edge - 1) / rec_edge;
                if (want_plain) c_plain += nt * (nt + 1) / 2;
                for (size_t ti = 0; ti < nt64; ++ti) c_miss += (64 * ti + 63) / 128 + 1;
                c_rec += np * (np + 1) / 2;
            }
            if (B.grow0 == INT64_MAX) B.grow0 = B.grow1 = 0;
            B.tile1 = (int32_t)c_plain;
            B.mtile1 = (int32_t)c_miss;
            B.ptile1 = (int32_t)c_rec;
        }
        tiles_plain.n = c_plain;
        tiles_miss.n = c_miss;
        tiles_pair.n = c_rec;
        P.n_tiles_plain = (int32_t)c_plain;
        P.n_tiles_miss = (int32_t)c_miss;
        P.n_tiles_pair = (int32_t)c_rec;
    }
    if (tiles_plain.n <= tiles_plain.cap && tiles_miss.n <= tiles_miss.cap && tiles_pair.n <= tiles_pair.cap) {
        for (size_t bi = 0; bi < P.batches.size(); ++bi) {
            const Batch* Bp = &P.batches[bi];
            host_pool().submit(g_tiles, [&P, &tiles_miss, Bp]() {
                GramTile* out = tiles_miss.p + Bp->mtile0;
                for (int i = 0; i < Bp->ord_n; ++i) {
                    const int b = P.order[Bp->ord_off + i];
                    const BlockDesc& d = P.blocks[b];
                    if (d.m == 0) continue;
                    const int nt64 = (d.mp + 63) / 64;
                    for (int ti = 0; ti < nt64; ++ti)
                        for (int tj = 0; 128 * tj <= 64 * ti + 63; ++tj) nt_copy(out++, GramTile{b, ti, tj, 0});
                }
                nt_fence();
            });
            host_pool().submit(g_tiles, [&P, &tiles_plain, &tiles_pair, Bp, want_plain, rec_edge]() {
                GramTile* outp = tiles_plain.p + Bp->tile0;
                TileRec* outr = tiles_pair.p + Bp->ptile0;
                for (int i = 0; i < Bp->ord_n; ++i) {
                    const int b = P.order[Bp->ord_off + i];
                    const BlockDesc& d = P.blocks[b];
                    if (d.m == 0) continue;
                    const int nt = (d.mp + 127) / 128;
                    for (int ti = 0; ti < nt && want_plain; ++ti)
                        for (int tj = 0; tj <= ti; ++tj) nt_copy(outp++, GramTile{b, ti, tj, 0});
                    const int np = (d.mp + rec_edge - 1) / rec_edge;
                    for (int ti = 0; ti < np; ++ti)
                        for (int tj = 0; tj <= ti; ++tj) nt_copy(outr++, TileRec{b, ti, tj, d.croff, d.goff, d.m, d.mp, d.ld, d.moff, 0});
                }
                nt_fence();
            });
        }
    }

    // Cholesky step lists per batch
    BlobList<int32_t> diag_items;
    BlobList<int4> panel_items;
    diag_items.p = reinterpret_cast<int32_t*>(blob.data() + P.o_diag); diag_items.cap = n_diag_max;
    panel_items.p = reinterpret_cast<int4*>(blob.data() + P.o_panel); panel_items.cap = n_panel_max;
    // Two passes.  Pass 1 (serial, arithmetic only): per batch and step the split-K factor and the list sizes, hence the
    // place of every step's items; pass 2 (one host thread per batch): the items themselves -- 120 k non-temporal 16-byte
    // stores at C3, 0.65 ms on one thread, and on the critical path of a streaming fit.
    int32_t n_groups = 0;
    size_t n_diag_tot = 0, n_panel_tot = 0;
    for (Batch& B : P.batches) {
        const int32_t* members = P.order.data() + B.ord_off;
        B.tile_rows = (h->panel_tma && (h->tile64_mode >= 2 || (h->tile64_mode == 1 && !B.big))) ? 64 : 128;
        const int TR = B.tile_rows;
        const int kTargetCtas = chol_panel_ctas_per_sm(TR) * h->n_sm;      // one wave of panel CTAs
        int kmax = 0;
        for (int i = 0; i < B.ord_n; ++i) kmax = std::max(kmax, (P.blocks[members[i]].mp + 63) / 64);
        B.steps.resize(kmax);
        int64_t batch_scratch = 0;
        for (int k = 0; k < kmax; ++k) {
            StepList& s = B.steps[k];
            s.diag_off = (int32_t)n_diag_tot;
            s.panel_off = (int32_t)n_panel_tot;
            // macro tiles of this step, then the split-K factor: when a step has few tiles but a long K
            // loop (late panels of big blocks), slice K so the step still fills the GPU
            int ntiles = 0, nactive = 0, ndiag = 0;
            for (int i = 0; i < B.ord_n; ++i) {
                const BlockDesc& d = P.blocks[members[i]];
                if ((d.mp + 63) / 64 <= k) continue;
                const int wk = std::min(64, d.mp - 64 * k);
                const int nt = (d.nrows - (64 * k + wk) + TR - 1) / TR;
                ntiles += nt;
                nactive += (nt > 0);
                ++ndiag;
            }
            int nsl = 1;
            if (ntiles > 0) nsl = std::max(1, std::min({h->splitk_max, k / h->splitk_min_blocks, kTargetCtas / ntiles}));
            s.nsl = nsl;
            s.group_base = n_groups;
            s.n_groups = (nsl > 1) ? ntiles : 0;
            n_groups += s.n_groups;
            s.n_first = nactive * nsl;                 // macro tile 0 of every block, all its slices
            s.n_diag = ndiag;
            s.n_panel = ntiles * nsl;
            n_diag_tot += (size_t)s.n_diag;
            n_panel_tot += (size_t)s.n_panel;
            batch_scratch = std::max<int64_t>(batch_scratch, (int64_t)s.n_groups * nsl * TR * 64);
        }
        // A chain-bound step (the whole next step fits in one wave of CTAs) defers the next diagonal tile to the
        // next launch, where it overlaps the main loops; otherwise macro tile 0 factors it at the end of this step,
        // in the shadow of the step's later waves.
        for (int k = 0; k < kmax; ++k)
            B.steps[k].defer = (k + 1 < kmax && B.steps[k + 1].n_panel + B.steps[k + 1].n_diag <= (h->defer_max_ctas >= 0 ? h->defer_max_ctas : kTargetCtas)) ? 1 : 0;
        B.scratch_off = P.scratch_doubles;
        P.scratch_doubles += batch_scratch;
    }
    diag_items.n = n_diag_tot;
    panel_items.n = n_panel_tot;
    if (tr) tr->mark("  plan: step sizes");
    if (n_diag_tot <= diag_items.cap && n_panel_tot <= panel_items.cap) {
        auto fill_batch = [&](const Batch& B) {
            const int32_t* members = P.order.data() + B.ord_off;
            const int TR = B.tile_rows;
            for (size_t k = 0; k < B.steps.size(); ++k) {
                const StepList& s = B.steps[k];
                int32_t* dg = diag_items.p + s.diag_off;
                int4* pn = panel_items.p + s.panel_off;
                const int nsl = s.nsl;
                int32_t gid_next = s.group_base;
                // macro tile 0 of every block goes first: its CTA also factors the next diagonal tile (fused), so it
                // should start in the first wave of the launch
                for (int pass = 0; pass < 2; ++pass) {
                    for (int i = 0; i < B.ord_n; ++i) {
                        const int b = members[i];
                        const BlockDesc& d = P.blocks[b];
                        if ((d.mp + 63) / 64 <= (int)k) continue;
                        if (pass == 0) nt_copy(dg++, (int32_t)b);
                        const int wk = std::min(64, d.mp - 64 * (int)k);
                        const int nt = (d.nrows - (64 * (int)k + wk) + TR - 1) / TR;
                        for (int t = (pass == 0 ? 0 : 1); t < (pass == 0 ? std::min(nt, 1) : nt); ++t) {
                            const int gid = (nsl > 1) ? gid_next++ : 0;
                            for (int sl = 0; sl < nsl; ++sl) nt_copy(pn++, make_int4(b, t, sl | (nsl << 8), gid));
                        }
                    }
                }
            }
            nt_fence();
        };
        for (size_t bi = 0; bi < P.batches.size(); ++bi) {
            const Batch* Bp = &P.batches[bi];
            host_pool().submit(g_lists, [&fill_batch, Bp]() { fill_batch(*Bp); });
        }
        host_pool().wait(g_lists);             // (this thread works the queue too)
    }
    if (tr) tr->mark("  plan: step lists");

    nt_fence();
    host_pool().wait(g_tiles);
    if (tr) tr->mark("  plan: tile + step lists");
    // ---- the lists were written in place; the panel items close the blob
    if (tiles_plain.size() > tiles_plain.cap || tiles_miss.size() > tiles_miss.cap || tiles_pair.size() > tiles_pair.cap || diag_items.size() > diag_items.cap ||
        panel_items.size() > panel_items.cap)
        return fail(h, DBSLMM_B200_ERR_NOMEM, "pinned plan buffer: list bound exceeded");
    place(sizeof(int4) * panel_items.size());
    P.lmaps_base = nullptr;
    P.n_groups = n_groups;
    P.blob_bytes = o;
    host_pool().wait(g_fill);
    if (fill_bad.load()) return fail(h, DBSLMM_B200_ERR_ARG, "s_pos / l_pos out of range of the loaded .bed");
    if (tr) tr->mark("  plan: per-SNP arrays");
    std::memcpy(blob.data() + P.o_order, P.order.data(), sizeof(int32_t) * (size_t)nb);
    P.valid = true;
    return DBSLMM_B200_OK;
}

// Fingerprint of everything a cached plan depends on: the CSR block lists (not the z-scores, which a cached plan
// refreshes), the variance side channel's row count and the panel's shape.  Four independent multiply-xor lanes over
// 64-bit words: ~0.3 ms for a genome-wide call.
uint64_t hash_words(const void* p, size_t bytes, uint64_t seed) {
    const uint64_t* w = (const uint64_t*)p;
    const size_t n = bytes / 8;
    uint64_t h0 = seed ^ 0x9E3779B97F4A7C15ull, h1 = seed + 0xC2B2AE3D27D4EB4Full, h2 = ~seed, h3 = seed * 0x165667B19E3779F9ull + 1;
    size_t i = 0;
    for (; i + 4 <= n; i += 4) {
        h0 = (h0 ^ w[i]) * 0xFF51AFD7ED558CCDull; h1 = (h1 ^ w[i + 1]) * 0xC4CEB9FE1A85EC53ull;
        h2 = (h2 ^ w[i + 2]) * 0x9FB21C651E98DF25ull; h3 = (h3 ^ w[i + 3]) * 0xD6E8FEB86659FD93ull;
        h0 ^= h0 >> 29; h1 ^= h1 >> 31; h2 ^= h2 >> 30; h3 ^= h3 >> 28;
    }
    uint64_t tail = 0;
    for (size_t b = i * 8; b < bytes; ++b) tail = tail * 257 + ((const uint8_t*)p)[b];
    uint64_t h = h0 ^ (h1 * 3) ^ (h2 * 5) ^ (h3 * 7) ^ tail ^ (uint64_t)bytes;
    h ^= h >> 33; h *= 0xFF51AFD7ED558CCDull; h ^= h >> 33;
    return h;
}
uint64_t plan_fingerprint(const dbslmm_b200_handle* h, const dbslmm_b200_fit_args* a) {
    const int nb = a->n_blocks;
    uint64_t f = hash_words(a->s_off, sizeof(int32_t) * (size_t)(nb + 1), 1);
    f = hash_words(a->s_pos, sizeof(int32_t) * (size_t)a->s_off[nb], f);
    if (a->l_off) {
        f = hash_words(a->l_off, sizeof(int32_t) * (size_t)(nb + 1), f + 2);
        f = hash_words(a->l_pos, sizeof(int32_t) * (size_t)a->l_off[nb], f);
    }
    int64_t n_test = 0;
    if (a->test_bed) for (int i = 0; i < a->test_n_total; ++i) n_test += (a->test_indicator[i] != 0);
    const int64_t shape[4] = {h->n_snp, (int64_t)h->n_ref, n_test, (int64_t)(a->l_off != nullptr)};
    return hash_words(shape, sizeof shape, f);
}

int make_tensor_map(dbslmm_b200_handle* h, CUtensorMap* tm, void* base, int64_t n_rows, int32_t n_pad, int box_rows) {
    if (!h->encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
            return fail(h, DBSLMM_B200_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
        h->encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    }
    cuuint64_t dims[2] = {(cuuint64_t)n_pad, (cuuint64_t)n_rows};
    cuuint64_t strides[1] = {(cuuint64_t)n_pad};
    cuuint32_t box[2] = {128, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = h->encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, DBSLMM_B200_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
    return DBSLMM_B200_OK;
}

// ---- tensor maps of the TMA panel kernel (chol.cu: chol_panel_tma_kernel)
int ensure_encoder(dbslmm_b200_handle* h) {
    if (h->encode) return DBSLMM_B200_OK;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
        return fail(h, DBSLMM_B200_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    h->encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    return DBSLMM_B200_OK;
}
// A row-major FP64 matrix (ld doubles per row, `rows` rows) as [64 rows x 16 columns] boxes, 128-byte swizzle.
// perm: the row index r = 8a + 2b + c is split into the dimensions (b, c, a) with b listed first, so the rows of an
// 8-row group arrive in shared memory in the order 0,2,4,6,1,3,5,7 (conflict-free FP64 fragment loads, see chol.cu).
CUresult encode_f64_boxes(dbslmm_b200_handle* h, CUtensorMap* tm, const void* base, int64_t ld, int64_t rows, bool perm) {
    const cuuint64_t row_bytes = (cuuint64_t)ld * 8;
    if (perm) {
        cuuint64_t dims[4] = {(cuuint64_t)ld, 4, 2, (cuuint64_t)((rows + 7) / 8)};
        cuuint64_t strides[3] = {2 * row_bytes, row_bytes, 8 * row_bytes};
        cuuint32_t box[4] = {16, 4, 2, 8};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        return h->encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
    cuuint64_t strides[1] = {row_bytes};
    cuuint32_t box[2] = {16, 64};
    cuuint32_t estr[2] = {1, 1};
    return h->encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}
// Decide once per handle whether the driver accepts the permuting (non-monotonic stride) 4-D form.
int probe_perm(dbslmm_b200_handle* h, const void* some_device_ptr) {
    if (h->tmap_perm >= 0) return DBSLMM_B200_OK;
    int rc = ensure_encoder(h);
    if (rc != DBSLMM_B200_OK) return rc;
    CUtensorMap tm;
    h->tmap_perm = (encode_f64_boxes(h, &tm, some_device_ptr, 64, 64, true) == CUDA_SUCCESS) ? 1 : 0;
    return DBSLMM_B200_OK;
}
// One tensor map per block over its matrix in the L buffer, written into the pinned plan blob (they travel with it).
// Blocks of a single panel never run a K loop: their slot stays zero.
int encode_lmaps(dbslmm_b200_handle* h, Plan& P) {
    int rc = ensure_encoder(h);
    if (rc != DBSLMM_B200_OK) return rc;
    rc = probe_perm(h, h->lbuf.p);
    if (rc != DBSLMM_B200_OK) return rc;
    CUtensorMap* maps = reinterpret_cast<CUtensorMap*>((uint8_t*)h->h_blob.p + P.o_lmaps);
    const int nb = P.n_blocks;
    const bool perm = h->tmap_perm == 1;
    std::atomic<int> bad{0};
    auto work = [&](int b0, int b1) {
        cudaSetDevice(h->device);          // worker threads: the driver entry point wants a current context
        for (int b = b0; b < b1; ++b) {
            const BlockDesc& d = P.blocks[b];
            if (d.mp <= 64) { std::memset(&maps[b], 0, sizeof(CUtensorMap)); continue; }
            const CUresult r = encode_f64_boxes(h, &maps[b], (const double*)h->lbuf.p + d.moff, d.ld, d.nrows, perm);
            if (r != CUDA_SUCCESS) bad.store((int)r);
        }
    };
    const int nthr = (int)std::max<int64_t>(1, std::min<int64_t>({8, (int64_t)host_pool().size() + 1, (int64_t)nb / 128}));
    if (nthr == 1) work(0, nb);
    else {
        TaskGroup g;
        for (int t = 0; t < nthr; ++t) {
            const int b0 = (int)((int64_t)nb * t / nthr), b1 = (int)((int64_t)nb * (t + 1) / nthr);
            host_pool().submit(g, [&work, b0, b1]() { work(b0, b1); });
        }
        host_pool().wait(g);
    }
    if (bad.load() && nthr > 1) { bad.store(0); work(0, nb); }      // once more on the calling thread
    if (bad.load()) return fail(h, DBSLMM_B200_ERR_CUDA, "cuTensorMapEncodeTiled failed for a block matrix (CUresult " + std::to_string(bad.load()) + ")");
    P.lmaps_base = h->lbuf.p;
    return DBSLMM_B200_OK;
}
}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int dbslmm_b200_abi_version(void) { return DBSLMM_B200_ABI_VERSION; }

int dbslmm_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int dbslmm_b200_create(int device, dbslmm_b200_handle** out) {
    if (!out) return DBSLMM_B200_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return DBSLMM_B200_ERR_CUDA;   // no CPU fallback: the product path needs a GPU
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return DBSLMM_B200_ERR_CUDA;
    if (prop.major != 10) return DBSLMM_B200_ERR_CUDA;   // kernels are sm_100a only
    if (cudaSetDevice(device) != cudaSuccess) return DBSLMM_B200_ERR_CUDA;
    dbslmm_b200_handle* h = new (std::nothrow) dbslmm_b200_handle();
    if (!h) return DBSLMM_B200_ERR_NOMEM;
    h->device = device;
    h->n_sm = prop.multiProcessorCount;
    {
        // host workers, ONE pool per process (all handles of a --gpus N command line share it): leave two hardware threads
        // to the caller; under a one-process-per-GPU launcher (LOCAL_WORLD_SIZE set) a process takes its share of the
        // machine; DBSLMM_B200_HOST_THREADS overrides (0 = no pool: every helper task runs inline)
        int n = (int)std::thread::hardware_concurrency() - 2;
        if (const char* e = std::getenv("LOCAL_WORLD_SIZE")) { const int lws = std::max(1, std::atoi(e)); n = (int)std::thread::hardware_concurrency() / lws - 1; }
        if (const char* e = std::getenv("DBSLMM_B200_HOST_THREADS")) n = std::atoi(e);
        host_pool().start(std::max(0, std::min(n, 14)));
    }
    if (const char* e = std::getenv("DBSLMM_B200_FUSE_DIAG")) h->fuse_diag = (e[0] != '0');   // tuning switches
    if (const char* e = std::getenv("DBSLMM_B200_STREAM_BED")) h->stream_bed = (e[0] != '0');
    if (const char* e = std::getenv("DBSLMM_B200_SPLITK")) {      // "max,min_blocks"
        int a = 0, b = 0;
        if (std::sscanf(e, "%d,%d", &a, &b) == 2 && a >= 1 && a <= 255 && b >= 1) { h->splitk_max = a; h->splitk_min_blocks = b; }
    }
    if (const char* e = std::getenv("DBSLMM_B200_DEFER_CTAS")) h->defer_max_ctas = std::atoi(e);
    if (const char* e = std::getenv("DBSLMM_B200_TILE64")) h->tile64_mode = std::atoi(e);
    if (const char* e = std::getenv("DBSLMM_B200_L2_PF")) h->l2_pf = std::min(255, std::max(0, std::atoi(e)));
    if (const char* e = std::getenv("DBSLMM_B200_NEXT_PF")) h->next_pf = std::atoi(e) != 0;
    if (const char* e = std::getenv("DBSLMM_B200_ZEROCOPY_BETA")) h->zero_copy_beta = (e[0] != '0');
    if (const char* e = std::getenv("DBSLMM_B200_UPLOAD_BULK_FIRST")) { h->upload_bulk_first = std::atoi(e); h->upload_auto = false; }
    if (const char* e = std::getenv("DBSLMM_B200_REGIONS")) h->n_regions = std::max(1, std::min(kMaxBatches - 4, std::atoi(e)));
    if (const char* e = std::getenv("DBSLMM_B200_PREPLAN_MB")) h->preplan_mb = std::atof(e);
    if (const char* e = std::getenv("DBSLMM_B200_REGION_MIN_BLOCKS")) h->region_min_blocks = std::max(1, std::atoi(e));
    if (const char* e = std::getenv("DBSLMM_B200_FIRST_REGION")) h->first_region = std::min(1.0, std::max(0.02, std::atof(e)));
    if (const char* e = std::getenv("DBSLMM_B200_GRAM_HINT")) h->gram_hint = std::atoi(e);
    if (const char* e = std::getenv("DBSLMM_B200_GRAM")) {
        h->gram_packed = (std::strcmp(e, "packed") == 0);
        h->gram_pair = (std::strcmp(e, "pair") == 0);
    }
    if (const char* e = std::getenv("DBSLMM_B200_PANEL")) h->panel_tma = (std::strcmp(e, "legacy") != 0);
    if (const char* e = std::getenv("DBSLMM_B200_TPC")) {         // "max[,waves]"
        int a = 0, b = 0;
        const int n = std::sscanf(e, "%d,%d", &a, &b);
        if (n >= 1 && a >= 1 && a <= 64) h->tpc_max = a;
        if (n >= 2 && b >= 0) h->tpc_waves = b;
    }
    if (const char* e = std::getenv("DBSLMM_B200_TMAP_PERM")) h->tmap_perm = (e[0] != '0') ? -1 : 0;
    if (const char* e = std::getenv("DBSLMM_B200_PDL")) h->pdl_ratio = std::atof(e);
    if (const char* e = std::getenv("DBSLMM_B200_CLASSES")) {     // e.g. "4,8,12,16,32"
        std::vector<int> b;
        for (const char* p = e; *p;) { char* q; long v = std::strtol(p, &q, 10); if (q == p) break; if (v > 0) b.push_back((int)v); p = (*q == ',') ? q + 1 : q; }
        std::sort(b.begin(), b.end());
        if (!b.empty() && (int)b.size() < kMaxBatches) h->cls_bounds = b;
    }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);     // numerically lower = higher priority
    // the main stream (decode, Gram, copies) outranks the Cholesky streams: in a streaming fit the decode/Gram of a
    // later batch must get SMs while earlier batches are being factored
    bool ok = cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
    for (int b = 0; b < kMaxBatches && ok; ++b) {
        // batches come in order of falling dependency-chain length (big classes first): schedule them first
        const int prio = std::max(prio_hi + 1, prio_lo - std::max(0, 4 - b));
        ok = cudaStreamCreateWithPriority(&h->b_stream[b], cudaStreamNonBlocking, prio) == cudaSuccess;
    }
    for (int b = 0; b < kMaxBatches && ok; ++b)
        ok = cudaEventCreate(&h->ev_join[b]) == cudaSuccess && cudaEventCreate(&h->ev_cend[b]) == cudaSuccess &&
             cudaEventCreate(&h->ev_up[b]) == cudaSuccess && cudaEventCreate(&h->ev_gram[b]) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&h->up_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_blob, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 8 && ok; ++i) ok = cudaEventCreate(&h->ev[i]) == cudaSuccess;
    ok = ok && cudaEventCreate(&h->ev_fork) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_bed, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_val, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 3 && ok; ++i) ok = cudaEventCreateWithFlags(&h->ev_pin_free[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i)
        ok = cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&h->ev_slot_free[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && chol_configure() == cudaSuccess;
    if (!ok) { dbslmm_b200_destroy(h); return DBSLMM_B200_ERR_CUDA; }
    *out = h;
    return DBSLMM_B200_OK;
}

void dbslmm_b200_destroy(dbslmm_b200_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    DevBuf* bufs[] = {&h->bed, &h->stats, &h->codes, &h->sigma, &h->lbuf, &h->rowN, &h->rowS, &h->rowR,
                      &h->planblob, &h->beta, &h->status, &h->intQ, &h->intA, &h->intN, &h->scratch, &h->counters, &h->wbuf, &h->vbed, &h->vstats, &h->vwork, &h->dflag, &h->dirty, &h->bflags, &h->packed, &h->rowC, &h->rowmap};
    for (DevBuf* b : bufs) b->release();
    h->h_blob.release();
    h->h_out.release();
    h->h_stats.release();
    for (PinBuf& b : h->s_pin) b.release();
    for (DevBuf& b : h->s_dev) b.release();
    h->s_work.release();
    for (DevBuf* b : {&h->ld_stats, &h->ld_codes, &h->ld_dirty, &h->ld_work, &h->ld_slots, &h->ld_red}) b->release();
    for (PinBuf& b : h->ld_pin) b.release();
    h->ld_roff.release();
    for (cudaEvent_t e : h->ev_pin_free) if (e) cudaEventDestroy(e);
    for (int i = 0; i < 2; ++i) {
        if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
        if (h->ev_slot_free[i]) cudaEventDestroy(h->ev_slot_free[i]);
    }
    for (cudaEvent_t e : h->ev_chunk) cudaEventDestroy(e);
    if (h->ev_bed) cudaEventDestroy(h->ev_bed);
    if (h->ev_val) cudaEventDestroy(h->ev_val);
    for (int i = 0; i < 8; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (int b = 0; b < kMaxBatches; ++b) {
        if (h->ev_join[b]) cudaEventDestroy(h->ev_join[b]);
        if (h->ev_cend[b]) cudaEventDestroy(h->ev_cend[b]);
        if (h->ev_up[b]) cudaEventDestroy(h->ev_up[b]);
        if (h->ev_gram[b]) cudaEventDestroy(h->ev_gram[b]);
    }
    for (int b = 0; b < kMaxBatches; ++b)
        if (h->b_stream[b]) cudaStreamDestroy(h->b_stream[b]);
    if (h->up_stream) cudaStreamDestroy(h->up_stream);
    if (h->ev_blob) cudaEventDestroy(h->ev_blob);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

const char* dbslmm_b200_last_error(const dbslmm_b200_handle* h) { return h ? h->err.c_str() : "null handle"; }

int dbslmm_b200_load_bed(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (!bed || n_snp <= 0 || n_ref <= 1) return fail(h, DBSLMM_B200_ERR_ARG, "load_bed: bad arguments");
    if (n_ref > decode_max_n_ref())
        return fail(h, DBSLMM_B200_ERR_ARG, "load_bed: n_ref = " + std::to_string(n_ref) + " is above the decoder's limit of " +
                                            std::to_string(decode_max_n_ref()) + " individuals (two .bed rows must fit in shared memory)");
    CU_TRY(h, cudaSetDevice(h->device));
    if (h->bed_pending) { CU_TRY(h, cudaEventSynchronize(h->ev_bed)); h->bed_pending = false; }   // buffers may be re-allocated
    const int32_t pitch = (n_ref + 3) / 4;
    const size_t bytes = (size_t)n_snp * pitch;
    CU_TRY(h, h->bed.ensure(bytes + 64));
    CU_TRY(h, h->stats.ensure(sizeof(SnpStat) * (size_t)n_snp));
    CU_TRY(h, cudaMemcpyAsync(h->bed.p, bed, bytes, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaMemsetAsync((uint8_t*)h->bed.p + bytes, 0xFF, 64, h->stream));
    CU_TRY(h, launch_snp_stats((const uint8_t*)h->bed.p, n_snp, n_ref, (SnpStat*)h->stats.p, h->n_sm, h->stream));
    // Asynchronous from here on: the call returns while the panel is still crossing PCIe, so the caller's
    // next step (dbslmm_b200_fit builds its block plan on the host) overlaps the upload.  The per-SNP
    // statistics follow the panel back to pinned host memory; snp_stats() waits for them.
    CU_TRY(h, h->h_stats.ensure(sizeof(SnpStat) * (size_t)n_snp));
    CU_TRY(h, cudaMemcpyAsync(h->h_stats.p, h->stats.p, sizeof(SnpStat) * (size_t)n_snp, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaEventRecord(h->ev_bed, h->stream));
    h->bed_pending = true;
    h->n_snp = n_snp;
    h->n_ref = n_ref;
    h->pitch = pitch;
    h->n_pad = (n_ref + 127) / 128 * 128;
    h->plan.valid = false;
    h->stats_valid = true;
    return DBSLMM_B200_OK;
}

// Per-SNP statistics of the resident panel, computed on demand: a streaming fit (fit_args.bed) uploads the panel
// without them (its decoder derives the counts of the rows it reads itself).
static int ensure_stats(dbslmm_b200_handle* h) {
    if (h->stats_valid) return DBSLMM_B200_OK;
    if (h->bed_pending) { CU_TRY(h, cudaEventSynchronize(h->ev_bed)); h->bed_pending = false; }
    CU_TRY(h, h->stats.ensure(sizeof(SnpStat) * (size_t)h->n_snp));
    CU_TRY(h, h->h_stats.ensure(sizeof(SnpStat) * (size_t)h->n_snp));
    CU_TRY(h, launch_snp_stats((const uint8_t*)h->bed.p, h->n_snp, h->n_ref, (SnpStat*)h->stats.p, h->n_sm, h->stream));
    CU_TRY(h, cudaMemcpyAsync(h->h_stats.p, h->stats.p, sizeof(SnpStat) * (size_t)h->n_snp, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaEventRecord(h->ev_bed, h->stream));
    h->bed_pending = true;
    h->stats_valid = true;
    return DBSLMM_B200_OK;
}

int dbslmm_b200_snp_stats(dbslmm_b200_handle* h, double* maf_out, int32_t* n_nonmiss_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (h->n_snp == 0) return fail(h, DBSLMM_B200_ERR_STATE, "snp_stats before load_bed");
    CU_TRY(h, cudaSetDevice(h->device));
    { int rc = ensure_stats(h); if (rc != DBSLMM_B200_OK) return rc; }
    if (h->bed_pending) { CU_TRY(h, cudaEventSynchronize(h->ev_bed)); h->bed_pending = false; }
    const SnpStat* hs = (const SnpStat*)h->h_stats.p;
    for (int64_t i = 0; i < h->n_snp; ++i) {
        const SnpStat& s = hs[(size_t)i];
        if (maf_out) {
            // readSNPIm (dtpr.cpp:358-362): mean-impute, af = sum(geno) / (2 n) = S / (2 n_i)
            const double af = 0.5 * (double)s.sum / (double)s.n_nonmiss;
            maf_out[i] = std::min(af, 1.0 - af);
        }
        if (n_nonmiss_out) n_nonmiss_out[i] = s.n_nonmiss;
    }
    return DBSLMM_B200_OK;
}

int dbslmm_b200_plan_shards(int32_t n_blocks, const int32_t* m_s, const int32_t* m_l, int32_t n_ref,
                            int32_t n_ranks, int32_t* owner_out, double* rank_cost_out) {
    if (n_blocks < 0 || n_ranks <= 0 || !m_s || !owner_out) return DBSLMM_B200_ERR_ARG;
    const double n_pad = (double)((n_ref + 127) / 128 * 128);
    std::vector<double> cost(n_blocks);
    for (int b = 0; b < n_blocks; ++b) {
        const double m = (double)m_s[b] + (m_l ? (double)m_l[b] : 0.0);
        // seconds-like units: int8 Gram at ~1 Pop/s effective, FP64 factorisation at ~15 TF/s effective,
        // plus a per-block latency floor (panel steps are serial inside a block)
        cost[b] = n_pad * m * (m + 1.0) / 1.0e15 + (m * m * m / 3.0 + 2.0 * m * m) / 1.5e13 + 2.0e-6 * std::ceil(m / 64.0);
    }
    std::vector<int> idx(n_blocks);
    std::iota(idx.begin(), idx.end(), 0);
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return cost[a] > cost[b]; });
    std::vector<double> load(n_ranks, 0.0);
    for (int b : idx) {
        int r = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        owner_out[b] = r;
        load[r] += cost[b];
    }
    if (rank_cost_out) for (int r = 0; r < n_ranks; ++r) rank_cost_out[r] = load[r];
    return DBSLMM_B200_OK;
}

}  // extern "C"

namespace {

// Streaming fit, host side: the class-ordered uploads of the panel rows each batch needs (one copy per run of
// adjacent blocks), then the rows no block uses, so the device copy ends up complete.
struct UploadPlan {
    typedef std::pair<int64_t, int64_t> Range;                  // [first, last] rows
    std::vector<std::vector<Range>> per_batch;
    std::vector<Range> all;
    int next_batch = 0;
};

// Returns 1 if the block -> row map is too scattered to stream (covering ranges would move far more than the
// panel), 0 on success, < 0 on error.
int upload_prepare(dbslmm_b200_handle* h, const dbslmm_b200_fit_args* a, const Plan& P, UploadPlan& U) {
    const int nb = P.n_blocks;
    const int64_t n_snp = h->n_snp;
    std::vector<int32_t> lo((size_t)std::max(nb, 1), INT32_MAX), hi((size_t)std::max(nb, 1), -1);
    {
        // row range of every block: the only O(#SNPs) scan before the first copy can be issued -> a few host threads
        std::atomic<int> bad{0};
        auto scan = [&](int b0, int b1) {
            for (int b = b0; b < b1; ++b) {
                int32_t l = INT32_MAX, u = -1;
                for (int j = a->s_off[b]; j < a->s_off[b + 1]; ++j) { const int32_t p = a->s_pos[j]; l = std::min(l, p); u = std::max(u, p); }
                if (a->l_off) for (int j = a->l_off[b]; j < a->l_off[b + 1]; ++j) { const int32_t p = a->l_pos[j]; l = std::min(l, p); u = std::max(u, p); }
                if (u >= 0 && (l < 0 || u >= n_snp)) bad.store(1);
                lo[b] = l; hi[b] = u;
            }
        };
        const int64_t tot = P.tot_s + P.tot_l;
        const int nthr = (int)std::max<int64_t>(1, std::min<int64_t>({8, (int64_t)host_pool().size() + 1, tot / 131072}));
        if (nthr == 1) scan(0, nb);
        else {
            TaskGroup g;
            for (int t = 0; t < nthr; ++t) {
                const int b0 = (int)((int64_t)nb * t / nthr), b1 = (int)((int64_t)nb * (t + 1) / nthr);
                host_pool().submit(g, [&scan, b0, b1]() { scan(b0, b1); });
            }
            host_pool().wait(g);
        }
        if (bad.load()) return fail(h, DBSLMM_B200_ERR_ARG, "fit: SNP row out of range of the .bed");
    }
    typedef UploadPlan::Range Range;
    U.per_batch.assign(P.batches.size(), std::vector<Range>());
    int64_t rows_total = 0;
    for (size_t bi = 0; bi < P.batches.size(); ++bi) {
        const Batch& B = P.batches[bi];
        std::vector<Range> r;
        for (int i = 0; i < B.ord_n; ++i) {
            const int b = P.order[B.ord_off + i];
            if (hi[b] >= 0) r.push_back(Range(lo[b], hi[b]));
        }
        std::sort(r.begin(), r.end());
        std::vector<Range>& m = U.per_batch[bi];
        for (const Range& x : r) {
            if (!m.empty() && x.first <= m.back().second + 33) m.back().second = std::max(m.back().second, x.second);
            else m.push_back(x);
        }
        for (const Range& x : m) { rows_total += x.second - x.first + 1; U.all.push_back(x); }
    }
    return (rows_total > n_snp + n_snp / 4) ? 1 : 0;            // scattered subsets: a plain full upload is cheaper
}

// Issue the uploads of the batches up_order[next_batch .. upto); upto == #batches also sends the rows outside every block.
int upload_issue(dbslmm_b200_handle* h, const Plan& P, UploadPlan& U, const uint8_t* bed, int upto, bool subset) {
    typedef UploadPlan::Range Range;
    const size_t pitch = (size_t)h->pitch;
    const int64_t n_snp = h->n_snp;
    uint8_t* dev = (uint8_t*)h->bed.p;
    for (; U.next_batch < upto; ++U.next_batch) {
        const int bi = P.up_order[U.next_batch];
        for (const Range& x : U.per_batch[bi])
            CU_TRY(h, cudaMemcpyAsync(dev + (size_t)x.first * pitch, bed + (size_t)x.first * pitch,
                                      (size_t)(x.second - x.first + 1) * pitch, cudaMemcpyHostToDevice, h->up_stream));
        CU_TRY(h, cudaEventRecord(h->ev_up[bi], h->up_stream));
    }
    if (upto < (int)P.batches.size()) return 0;
    // rows outside every block (unmatched SNPs): last, so the resident copy is complete for later calls
    // (FLAG_PANEL_SUBSET: not sent at all -- the handle forgets the panel after the call)
    std::sort(U.all.begin(), U.all.end());
    int64_t next = subset ? n_snp : 0;
    for (const Range& x : U.all) {
        if (subset) break;
        if (x.first > next)
            CU_TRY(h, cudaMemcpyAsync(dev + (size_t)next * pitch, bed + (size_t)next * pitch, (size_t)(x.first - next) * pitch,
                                      cudaMemcpyHostToDevice, h->up_stream));
        next = std::max(next, x.second + 1);
    }
    if (next < n_snp)
        CU_TRY(h, cudaMemcpyAsync(dev + (size_t)next * pitch, bed + (size_t)next * pitch, (size_t)(n_snp - next) * pitch,
                                  cudaMemcpyHostToDevice, h->up_stream));
    CU_TRY(h, cudaMemsetAsync(dev + (size_t)n_snp * pitch, 0xFF, 64, h->up_stream));
    CU_TRY(h, cudaEventRecord(h->ev_bed, h->up_stream));
    h->bed_pending = true;
    return 0;
}

// Upload of an announced validation panel (+ its per-SNP statistics) on the upload stream: called by a fit right after
// it has issued its own panel copies (so the big copy queues BEHIND them and overlaps the fit's kernels), or by score
// itself when no fit came in between.
int issue_val_upload(dbslmm_b200_handle* h) {
    if (!h->val_announced) return DBSLMM_B200_OK;
    const int32_t pitch = (h->val_n + 3) / 4;
    const size_t bytes = (size_t)h->val_n_snp * pitch;
    CU_TRY(h, cudaMemcpyAsync(h->vbed.p, h->val_host, bytes, cudaMemcpyHostToDevice, h->up_stream));
    CU_TRY(h, cudaMemsetAsync((uint8_t*)h->vbed.p + bytes, 0xFF, 64, h->up_stream));
    CU_TRY(h, launch_snp_stats((const uint8_t*)h->vbed.p, h->val_n_snp, h->val_n, (SnpStat*)h->vstats.p, h->n_sm, h->up_stream));
    CU_TRY(h, cudaEventRecord(h->ev_val, h->up_stream));
    h->val_announced = false;
    h->val_inflight = true;
    return DBSLMM_B200_OK;
}

// One fit.  streaming = the panel is uploaded inside this call from a->bed, batch by batch (see Batch); otherwise the
// panel loaded by load_bed is used.  Returns n_bad >= 0 or an error < 0.

int fit_impl(dbslmm_b200_handle* h, const dbslmm_b200_fit_args* a, bool streaming) {
    const bool want_var = a->test_bed != nullptr;
    cudaStream_t st = h->stream;
    const bool pcg = (a->solver == DBSLMM_B200_SOLVER_PCG);
    const bool full = pcg || (a->flags & DBSLMM_B200_FLAG_FULL_SIGMA);
    const bool keep_int = (a->flags & DBSLMM_B200_FLAG_KEEP_INT_GRAM) != 0;
    const bool quad = a->quadform_out != nullptr;          // `valid`: z' Sigma z per block instead of the solve
    const bool subset = streaming && (a->flags & DBSLMM_B200_FLAG_PANEL_SUBSET) != 0;

    Trace tr;
    UploadPlan U;
    // ---- plan
    Plan& P = h->plan;
    // FLAG_PLAN_CACHED re-uses the device plan only if the block lists, the test-row count and the panel shape are the
    // ones it was built from (fingerprint); otherwise the plan is silently rebuilt
    const bool want_reuse = !streaming && (a->flags & DBSLMM_B200_FLAG_PLAN_CACHED) && P.valid && !P.streaming &&
                            P.n_blocks == a->n_blocks && P.tot_s == a->s_off[a->n_blocks] &&
                            P.tot_l == (a->l_off ? a->l_off[a->n_blocks] : 0);
    const uint64_t fp = (want_reuse || !streaming) ? plan_fingerprint(h, a) : 0;
    const bool reuse = want_reuse && P.fingerprint == fp;
    if (!reuse) {
        // The plan is built while the panel may still be crossing PCIe and never looks at it: every block is laid out
        // with both code planes, and which blocks have missing calls is decided on the device.
        int rc = make_batches(h, a, P, streaming);
        if (rc != DBSLMM_B200_OK) { P.valid = false; return rc; }
        if (streaming) {
            tr.mark("batches");
            rc = upload_prepare(h, a, P, U);
            if (rc < 0) { P.valid = false; return rc; }
            // the biggest classes go out before the plan is built (the H2D queue is in issue order: the plan blob must
            // not wait behind the whole panel, and the DMA engine should not idle while the host builds the plan)
            if (rc == 0) {
                // how many batches go out before the plan exists: the first one, and more while they stay under preplan_mb
                int n_pre = 0;
                double mb = 0.0;
                for (size_t ui = 0; ui < P.up_order.size(); ++ui) {
                    double rows = 0.0;
                    for (const UploadPlan::Range& x : U.per_batch[P.up_order[ui]]) rows += (double)(x.second - x.first + 1);
                    mb += rows * (double)h->pitch / 1.0e6;
                    if (n_pre > 0 && mb > h->preplan_mb) break;
                    ++n_pre;
                }
                rc = upload_issue(h, P, U, a->bed, std::min(n_pre, (int)P.batches.size()), subset);
                if (rc < 0) { P.valid = false; return rc; }
            }
            tr.mark("first uploads issued");
            if (rc == 1) {
                // not streamable: plain full upload, then the resident path
                P.valid = false;
                rc = dbslmm_b200_load_bed(h, a->bed, a->bed_n_snp, a->bed_n_ref);
                if (rc != DBSLMM_B200_OK) return rc;
                return fit_impl(h, a, false);
            }
        }
        rc = build_plan(h, a, P, &tr);
        if (rc != DBSLMM_B200_OK) { P.valid = false; return rc; }
        P.fingerprint = fp;
        tr.mark("plan built");
    }
    if (!streaming && h->bed_pending) { CU_TRY(h, cudaEventSynchronize(h->ev_bed)); h->bed_pending = false; }   // load_bed's copy runs on the same stream, but its source buffer may go away
    const int nb = P.n_blocks;
    const int nbatch = (int)P.batches.size();
    const size_t nfold = quad ? 1 : (size_t)a->n_folds;

    // ---- workspace
    CU_TRY(h, h->planblob.ensure(P.blob_bytes + 256));
    CU_TRY(h, h->codes.ensure((size_t)std::max<int64_t>(P.n_code_rows, 1) * h->n_pad));
    {
        // dirty[c] = code row c holds a mask that is NOT the default pattern (decode.cu).  Rows the map has never covered,
        // and all rows when the panel width or the code-row layout changes, start dirty: the first fit then writes their
        // mask rows once.  (Under another layout a mask row may have been a genotype row, which the map does not track:
        // resident and streaming fits lay the blocks out in different orders.)
        const size_t need = (size_t)std::max<int64_t>(P.n_code_rows, 1);
        if (h->dirty_n_ref != h->n_ref || need > h->dirty_rows || h->dirty_codes != h->codes.p || h->dirty_layout != P.code_layout) {
            CU_TRY(h, h->dirty.ensure(need));
            const size_t cover = h->dirty.cap;
            CU_TRY(h, cudaMemsetAsync(h->dirty.p, 1, cover, st));
            h->dirty_rows = cover;
            h->dirty_n_ref = h->n_ref;
            h->dirty_codes = h->codes.p;         // a re-allocated code buffer has lost every mask row
            h->dirty_layout = P.code_layout;
        }
    }
    CU_TRY(h, h->bflags.ensure(sizeof(int32_t) * (size_t)(std::max(nb, 1) + kMaxBatches + 1)));
    const bool packed_gram = h->gram_packed;
    if (packed_gram) CU_TRY(h, h->packed.ensure((size_t)std::max<int64_t>(P.n_snp_rows, 1) * (size_t)(h->n_pad / 4) + 4096));
    CU_TRY(h, h->sigma.ensure(sizeof(double) * (size_t)std::max<int64_t>(P.mat_doubles, 1)));
    if (!pcg && !quad) CU_TRY(h, h->lbuf.ensure(sizeof(double) * (size_t)std::max<int64_t>(P.mat_doubles, 1)));
    CU_TRY(h, h->rowN.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(P.n_snp_rows, 1)));
    CU_TRY(h, h->rowS.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(P.n_snp_rows, 1)));
    CU_TRY(h, h->rowR.ensure(sizeof(double) * (size_t)std::max<int64_t>(P.n_snp_rows, 1)));
    CU_TRY(h, h->rowC.ensure(sizeof(double2) * (size_t)std::max<int64_t>(P.n_snp_rows, 1)));
    CU_TRY(h, h->rowmap.ensure(2 * sizeof(int32_t) * (size_t)std::max<int64_t>(P.n_snp_rows, 1)));
    const size_t n_out = (size_t)(P.tot_s + P.tot_l);
    const size_t n_res = quad ? (size_t)nb : n_out * nfold;          // doubles coming back: betas of all folds, or one z'Sigma z per block
    CU_TRY(h, h->beta.ensure(sizeof(double) * std::max<size_t>(n_res, 1)));
    CU_TRY(h, h->status.ensure(sizeof(int32_t) * (size_t)std::max(2 * nb, 1)));
    if (!pcg && !quad) {
        CU_TRY(h, h->scratch.ensure(sizeof(double) * (size_t)std::max<int64_t>(P.scratch_doubles, 1)));
        CU_TRY(h, h->wbuf.ensure(2 * sizeof(double) * 64 * 64 * (size_t)std::max(nb, 1)));   // two parities, see launch_chol_diag
        CU_TRY(h, h->counters.ensure(sizeof(int32_t) * (size_t)std::max(P.n_groups, 1)));
        CU_TRY(h, h->dflag.ensure(sizeof(int32_t) * (size_t)std::max(nb, 1)));
    }
    if (keep_int) {
        CU_TRY(h, h->intQ.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(P.mat_doubles, 1)));
        CU_TRY(h, h->intA.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(P.mat_doubles, 1)));
        CU_TRY(h, h->intN.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(P.mat_doubles, 1)));
    }
    const size_t out_bytes = sizeof(double) * n_res + sizeof(int32_t) * (size_t)(3 * nb);     // results, status, iterations, missing-call flags
    CU_TRY(h, h->h_out.ensure(out_bytes + 128));
    const bool tma_panel = h->panel_tma && !pcg && !quad;
    bool lmaps_dirty = false;                   // the maps in the pinned blob were (re)encoded: a cached device plan needs them again
    if (tma_panel && nb > 0) {
        if (P.lmaps_base != h->lbuf.p) {
            int rc = encode_lmaps(h, P);
            if (rc != DBSLMM_B200_OK) return rc;
            lmaps_dirty = true;
            tr.mark("tensor maps encoded");
        }
    }

    uint8_t* dblob = (uint8_t*)h->planblob.p;   // (re-pointed below if the plan has to be rebuilt)
    const BlockDesc* d_blocks = (const BlockDesc*)(dblob + P.o_blocks);
    const uint32_t* d_rowsrc = (const uint32_t*)(dblob + P.o_rowsrc);
    const int32_t* d_crow = (const int32_t*)h->rowmap.p;                       // [n_snp_rows] code row, then [n_snp_rows] mask row
    const int32_t* d_mrow = d_crow + std::max<int64_t>(P.n_snp_rows, 1);
    int32_t* d_bflags = (int32_t*)h->bflags.p;               // [nb] per-block flag, then one "any" word per batch
    int32_t* d_any = d_bflags + std::max(nb, 1);
    const double* d_z = (const double*)(dblob + P.o_z);
    const GramTile* d_tiles_plain = (const GramTile*)(dblob + P.o_tiles_plain);
    const GramTile* d_tiles_miss = (const GramTile*)(dblob + P.o_tiles_miss);
    const TileRec* d_recs = (const TileRec*)(dblob + P.o_tiles_pair);
    const int32_t* d_order = (const int32_t*)(dblob + P.o_order);
    const int32_t* d_diag = (const int32_t*)(dblob + P.o_diag);
    const int4* d_panel = (const int4*)(dblob + P.o_panel);
    const bool zc_beta = h->zero_copy_beta && !pcg;         // (the PCG kernel reads its own betas back: device buffer)
    double* d_beta = zc_beta ? (double*)h->h_out.p : (double*)h->beta.p;
    int32_t* d_status = (int32_t*)h->status.p;
    int32_t* d_iters = d_status + nb;

    int n_launch = 0, n_chol_launch = 0;
    if (reuse && P.n_snp_rows > 0) {
        // same CSR layout, new z-scores: refill the pinned z array (host work, before the first event)
        double* z = reinterpret_cast<double*>((uint8_t*)h->h_blob.p + P.o_z);
        for (int b = 0; b < nb; ++b) {
            const BlockDesc& d = P.blocks[b];
            if (d.ms > 0) std::memcpy(z + d.goff, a->s_z + a->s_off[b], sizeof(double) * (size_t)d.ms);
            if (d.m > d.ms) std::memcpy(z + d.goff + d.ms, a->l_z + a->l_off[b], sizeof(double) * (size_t)(d.m - d.ms));
        }
    }
    cudaEvent_t tr_blob = nullptr, tr_blob0 = nullptr, tr_dec[kMaxBatches] = {}, tr_start[kMaxBatches] = {};      // DBSLMM_B200_TRACE only
    int tr_chain = 0;
    CU_TRY(h, cudaEventRecord(h->ev[0], st));
    // ---- upload
    if (!reuse) {
        if (!streaming) {
            if (P.blob_bytes) CU_TRY(h, cudaMemcpyAsync(dblob, h->h_blob.p, P.blob_bytes, cudaMemcpyHostToDevice, st));
        } else {
            // The plan blob travels on the UPLOAD stream, between the first batches and the rest of the panel: copies
            // of one stream run in issue order, whereas a copy on another stream may sit behind the whole panel.
            if (tr.on) { cudaEventCreate(&tr_blob0); cudaEventRecord(tr_blob0, h->up_stream); }
            if (P.blob_bytes) CU_TRY(h, cudaMemcpyAsync(dblob, h->h_blob.p, P.blob_bytes, cudaMemcpyHostToDevice, h->up_stream));
            CU_TRY(h, cudaEventRecord(h->ev_blob, h->up_stream));
            CU_TRY(h, cudaStreamWaitEvent(st, h->ev_blob, 0));
            if (tr.on) { cudaEventCreate(&tr_blob); cudaEventRecord(tr_blob, h->up_stream); }
            int rc = upload_issue(h, P, U, a->bed, nbatch, subset);
            if (rc < 0) return rc;
            tr.mark("all uploads issued");
        }
    } else if (P.n_snp_rows > 0) {
        if (lmaps_dirty)
            CU_TRY(h, cudaMemcpyAsync(dblob + P.o_lmaps, (uint8_t*)h->h_blob.p + P.o_lmaps, sizeof(CUtensorMap) * (size_t)nb,
                                      cudaMemcpyHostToDevice, st));
        CU_TRY(h, cudaMemcpyAsync(dblob + P.o_z, (uint8_t*)h->h_blob.p + P.o_z, sizeof(double) * (size_t)P.n_snp_rows,
                                  cudaMemcpyHostToDevice, st));
    }
    if (!reuse && nb > 0 && P.n_snp_rows > 0) {
        // code-row / mask-row of every SNP row from the block descriptors (the stream already waits for the blob)
        CU_TRY(h, launch_fill_rowmaps(d_blocks, nb, (int32_t*)h->rowmap.p, (int32_t*)h->rowmap.p + P.n_snp_rows, st));
        ++n_launch;
    }
    { int rc = issue_val_upload(h); if (rc != DBSLMM_B200_OK) return rc; }     // an announced validation panel follows the fit's own copies
    CU_TRY(h, cudaMemsetAsync(d_status, 0, sizeof(int32_t) * (size_t)std::max(2 * nb, 1), st));
    CU_TRY(h, cudaMemsetAsync(d_any, 0, sizeof(int32_t) * (size_t)(kMaxBatches + 1), st));
    CU_TRY(h, cudaEventRecord(h->ev[1], st));

    if (!pcg && !quad && P.n_groups > 0) CU_TRY(h, cudaMemsetAsync(h->counters.p, 0, sizeof(int32_t) * (size_t)P.n_groups, st));
    if (!pcg && !quad) CU_TRY(h, cudaMemsetAsync(h->dflag.p, 0, sizeof(int32_t) * (size_t)std::max(nb, 1), st));
    // ---- decode + gram
    GramArgs g;
    CUtensorMap tmap, tmap64, pmap;
    if (P.n_code_rows > 0) {
        int rc = make_tensor_map(h, &tmap, h->codes.p, P.n_code_rows, h->n_pad, 128);
        if (rc != DBSLMM_B200_OK) return rc;
        rc = make_tensor_map(h, &tmap64, h->codes.p, P.n_code_rows, h->n_pad, 64);      // I side of the four-plane kernel
        if (rc != DBSLMM_B200_OK) return rc;
        if (packed_gram) {
            // packed 2-bit rows: [n_snp_rows][n_pad / 4 bytes], operand tile = 128 rows x 32 bytes (128 samples), no swizzle
            cuuint64_t dims[2] = {(cuuint64_t)(h->n_pad / 4), (cuuint64_t)P.n_snp_rows};
            cuuint64_t strides[1] = {(cuuint64_t)(h->n_pad / 4)};
            cuuint32_t box[2] = {32, 128};
            cuuint32_t estr[2] = {1, 1};
            if (h->encode(&pmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, h->packed.p, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                return fail(h, DBSLMM_B200_ERR_CUDA, "cuTensorMapEncodeTiled failed for the packed rows");
        }
        g.blocks = d_blocks;
        g.nk = h->n_pad / 128;
        g.n_ref = h->n_ref;
        g.one_minus_tau = 1.0 - a->tau;
        g.rowN = (const int32_t*)h->rowN.p;
        g.rowS = (const int32_t*)h->rowS.p;
        g.rowR = (const double*)h->rowR.p;
        g.rowC = (const double2*)h->rowC.p;
        g.sigma = (double*)h->sigma.p;
        g.intQ = keep_int ? (int32_t*)h->intQ.p : nullptr;
        g.intA = keep_int ? (int32_t*)h->intA.p : nullptr;
        g.intN = keep_int ? (int32_t*)h->intN.p : nullptr;
        g.full = full ? 1 : 0;
        g.light = 0;
        g.flags = d_bflags;
        g.hint = h->gram_hint;
    }
    // One chain per batch of blocks: decode its SNP rows (both code planes where needed) -> per-block missing-call flags
    // -> one-plane Gram over the blocks without missing calls -> four-plane Gram over the others (returns at once if
    // there are none) -> z rows.  A resident fit runs ONE chain over everything.
    auto chain = [&](int64_t g0, int64_t g1, const int32_t* list, int32_t n_list, int32_t t0, int32_t t1, int32_t mt0, int32_t mt1,
                     int32_t pt0, int32_t pt1, int32_t* any, bool light) -> int {
        if (g1 <= g0) return DBSLMM_B200_OK;
        if (tr.on && streaming && tr_chain < kMaxBatches) { cudaEventCreate(&tr_start[tr_chain]); cudaEventRecord(tr_start[tr_chain], st); }
        if (packed_gram)        // 2-bit rows in plan order + per-SNP statistics; int8 rows only if a block turns out to need them
            CU_TRY(h, launch_pack_rows((const uint8_t*)h->bed.p, h->n_ref, h->n_pad, d_rowsrc, g0, g1 - g0, a->tau, (uint32_t*)h->packed.p,
                                       (int32_t*)h->rowN.p, (int32_t*)h->rowS.p, (double*)h->rowR.p, (double2*)h->rowC.p, h->n_sm, st));
        else
            CU_TRY(h, launch_decode_rows((const uint8_t*)h->bed.p, h->n_ref, h->n_pad, d_rowsrc, d_crow, d_mrow, g0, g1 - g0, a->tau,
                                         (int8_t*)h->codes.p, (uint8_t*)h->dirty.p, (int32_t*)h->rowN.p, (int32_t*)h->rowS.p,
                                         (double*)h->rowR.p, (double2*)h->rowC.p, nullptr, h->n_sm, st));
        if (tr.on && streaming && tr_chain < kMaxBatches) { cudaEventCreate(&tr_dec[tr_chain]); cudaEventRecord(tr_dec[tr_chain], st); ++tr_chain; }
        CU_TRY(h, launch_block_flags(d_blocks, list, n_list, (const int32_t*)h->rowN.p, h->n_ref, d_bflags, any, st));
        n_launch += 2;
        g.any = any;
        g.light = light ? 1 : 0;         // 3-stage ring: a Gram CTA fits on an SM next to one Cholesky panel CTA
        if (t1 > t0 || pt1 > pt0) {
            g.tiles = d_tiles_plain + t0;
            g.n_tiles = t1 - t0;
            if (packed_gram) CU_TRY(h, launch_gram_packed(pmap, g, st));
            else {
                g.tiles = nullptr;
                g.recs = d_recs + pt0;
                g.n_tiles = pt1 - pt0;
                if (h->gram_pair) CU_TRY(h, launch_gram_pair(tmap, tmap64, g, st));
                else CU_TRY(h, launch_gram(tmap, g, st));
            }
            ++n_launch;
        }
        if (packed_gram) {      // returns at once unless some block of this chain has missing calls
            CU_TRY(h, launch_decode_rows((const uint8_t*)h->bed.p, h->n_ref, h->n_pad, d_rowsrc, d_crow, d_mrow, g0, g1 - g0, a->tau,
                                         (int8_t*)h->codes.p, (uint8_t*)h->dirty.p, (int32_t*)h->rowN.p, (int32_t*)h->rowS.p,
                                         (double*)h->rowR.p, (double2*)h->rowC.p, any, h->n_sm, st));
            ++n_launch;
        }
        if (mt1 > mt0) {
            g.tiles = d_tiles_miss + mt0;
            g.n_tiles = mt1 - mt0;
            CU_TRY(h, launch_gram_missing(tmap, tmap64, g, st));
            ++n_launch;
        }
        CU_TRY(h, launch_fill_z(d_blocks, list, n_list, d_z, (double*)h->sigma.p, st));
        ++n_launch;
        return DBSLMM_B200_OK;
    };
    if (!streaming) {
        // ONE chain over everything.  decode_ms = the packer / decoder; the rest of the chain counts as Gram time
        if (P.n_snp_rows > 0) {
            if (packed_gram)
                CU_TRY(h, launch_pack_rows((const uint8_t*)h->bed.p, h->n_ref, h->n_pad, d_rowsrc, 0, P.n_snp_rows, a->tau, (uint32_t*)h->packed.p,
                                           (int32_t*)h->rowN.p, (int32_t*)h->rowS.p, (double*)h->rowR.p, (double2*)h->rowC.p, h->n_sm, st));
            else
                CU_TRY(h, launch_decode_rows((const uint8_t*)h->bed.p, h->n_ref, h->n_pad, d_rowsrc, d_crow, d_mrow, 0, P.n_snp_rows, a->tau,
                                             (int8_t*)h->codes.p, (uint8_t*)h->dirty.p, (int32_t*)h->rowN.p, (int32_t*)h->rowS.p,
                                             (double*)h->rowR.p, (double2*)h->rowC.p, nullptr, h->n_sm, st));
            ++n_launch;
        }
        CU_TRY(h, cudaEventRecord(h->ev[2], st));          // packer / decoder done
        if (P.n_snp_rows > 0) {
            CU_TRY(h, launch_block_flags(d_blocks, nullptr, nb, (const int32_t*)h->rowN.p, h->n_ref, d_bflags, d_any, st));
            ++n_launch;
            g.any = d_any;
            g.tiles = d_tiles_plain;
            g.n_tiles = P.n_tiles_plain;
            if (packed_gram) {
                CU_TRY(h, launch_gram_packed(pmap, g, st));
                CU_TRY(h, launch_decode_rows((const uint8_t*)h->bed.p, h->n_ref, h->n_pad, d_rowsrc, d_crow, d_mrow, 0, P.n_snp_rows, a->tau,
                                             (int8_t*)h->codes.p, (uint8_t*)h->dirty.p, (int32_t*)h->rowN.p, (int32_t*)h->rowS.p,
                                             (double*)h->rowR.p, (double2*)h->rowC.p, d_any, h->n_sm, st));
                ++n_launch;
            } else {
                g.tiles = nullptr;
                g.recs = d_recs;
                g.n_tiles = P.n_tiles_pair;
                if (h->gram_pair) CU_TRY(h, launch_gram_pair(tmap, tmap64, g, st));
                else CU_TRY(h, launch_gram(tmap, g, st));
            }
            g.tiles = d_tiles_miss;
            g.n_tiles = P.n_tiles_miss;
            CU_TRY(h, launch_gram_missing(tmap, tmap64, g, st));
            CU_TRY(h, launch_fill_z(d_blocks, nullptr, nb, d_z, (double*)h->sigma.p, st));
            n_launch += 3;
        }
    } else {
        // one chain per batch, each gated on the upload of that batch's rows; the batch's Cholesky (on its class
        // stream, below) is gated on ev_gram, so big classes factor while the bulk is still in flight
        CU_TRY(h, cudaEventRecord(h->ev[2], st));
        for (int ui = 0; ui < nbatch; ++ui) {
            const int bi = P.up_order[ui];                 // decode / Gram in the order the rows arrive
            const Batch& B = P.batches[bi];
            CU_TRY(h, cudaStreamWaitEvent(st, h->ev_up[bi], 0));
            int rc = chain(B.grow0, B.grow1, d_order + B.ord_off, B.ord_n, B.tile0, B.tile1, B.mtile0, B.mtile1, B.ptile0, B.ptile1, d_any + 1 + bi, true);
            if (rc != DBSLMM_B200_OK) return rc;
            CU_TRY(h, cudaEventRecord(h->ev_gram[bi], st));
        }
    }
    double* d_var = nullptr;
    if (want_var && P.n_test > 0 && P.n_snp_rows > 0) {
        // ---- variance side channel: test panel, selection list and per-SNP test rows to the device, then the
        // standardised test genotypes become extra rows of every block matrix
        const int32_t tpitch = (a->test_n_total + 3) / 4;
        const size_t tbytes = (size_t)a->test_n_snp * tpitch;
        std::vector<int32_t> sel, tpos((size_t)P.n_snp_rows);
        for (int i = 0; i < a->test_n_total; ++i) if (a->test_indicator[i] != 0) sel.push_back(i);
        for (int b = 0; b < nb; ++b) {
            const BlockDesc& d = P.blocks[b];
            for (int j = 0; j < d.m; ++j) {
                const int32_t tp = (j < d.ms) ? a->s_tpos[a->s_off[b] + j] : a->l_tpos[a->l_off[b] + (j - d.ms)];
                if (tp < 0 || tp >= a->test_n_snp) return fail(h, DBSLMM_B200_ERR_ARG, "fit: test .bed row out of range");
                tpos[(size_t)d.goff + j] = tp;
            }
        }
        size_t o = 0;
        auto place = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
        const size_t o_sel = place(sizeof(int32_t) * sel.size()), o_tpos = place(sizeof(int32_t) * tpos.size()),
                     o_mu = place(sizeof(double) * tpos.size()), o_isd = place(sizeof(double) * tpos.size()),
                     o_var = place(sizeof(double) * (size_t)a->n_folds * nb * P.n_test);
        CU_TRY(h, h->vbed.ensure(tbytes + 64));
        CU_TRY(h, h->vwork.ensure(o));
        uint8_t* vw = (uint8_t*)h->vwork.p;
        CU_TRY(h, cudaMemcpyAsync(h->vbed.p, a->test_bed, tbytes, cudaMemcpyHostToDevice, st));
        CU_TRY(h, cudaMemcpyAsync(vw + o_sel, sel.data(), sizeof(int32_t) * sel.size(), cudaMemcpyHostToDevice, st));
        CU_TRY(h, cudaMemcpyAsync(vw + o_tpos, tpos.data(), sizeof(int32_t) * tpos.size(), cudaMemcpyHostToDevice, st));
        CU_TRY(h, cudaStreamSynchronize(st));      // sel / tpos are stack-lifetime host vectors
        CU_TRY(h, launch_test_rows(d_blocks, nb, (const uint8_t*)h->vbed.p, a->test_n_total, (const int32_t*)(vw + o_sel),
                                   P.n_test, (const int32_t*)(vw + o_tpos), P.n_snp_rows, (double*)(vw + o_mu),
                                   (double*)(vw + o_isd), (double*)h->sigma.p, st));
        n_launch += 2;
        d_var = (double*)(vw + o_var);
    }
    CU_TRY(h, cudaEventRecord(h->ev[3], st));
    tr.mark("decode/gram launched");

    // ---- solve, once per heritability fold (Sigma is shared: only the ridge changes)
    float chol_ms_total = 0.f;
    const double inv_sqrt_n = quad ? 0.0 : 1.0 / std::sqrt((double)a->n_obs);
    if (quad && nb > 0) {
        // scr/validate.cpp:255-258: deno_b = z1' Sigma_b z1.  The per-block results take the place of the betas.
        CU_TRY(h, launch_quadform(d_blocks, nb, (const double*)h->sigma.p, d_z, d_beta, st));
        ++n_launch;
    }
    for (int f = 0; f < a->n_folds && !quad; ++f) {
        const double ridge = 1.0 / (a->sigma_s[f] * (double)a->n_obs);    // dbslmmfit.cpp:712 / :759
        double* bs = d_beta + (size_t)f * n_out;
        double* bl = bs + P.tot_s;
        if (!pcg) {
            if (f > 0 && P.n_groups > 0) CU_TRY(h, cudaMemsetAsync(h->counters.p, 0, sizeof(int32_t) * (size_t)P.n_groups, st));
            if (f > 0) CU_TRY(h, cudaMemsetAsync(h->dflag.p, 0, sizeof(int32_t) * (size_t)std::max(nb, 1), st));
            CU_TRY(h, cudaEventRecord(h->ev_fork, st));
            const int64_t wstride = (int64_t)64 * 64 * std::max(nb, 1);
            for (int bi = 0; bi < nbatch; ++bi) {
                const Batch& B = P.batches[bi];
                static const bool one_stream = std::getenv("DBSLMM_B200_ONE_STREAM") != nullptr;       // debugging aid
                cudaStream_t cs = h->b_stream[one_stream ? 0 : bi];
                // A batch whose dependency chain (steps x ~50 us) rivals the whole fit's throughput time is latency-bound:
                // its steps are launched programmatically dependent, so the next step's CTAs are resident (and waiting)
                // before the current step ends instead of queueing for SM slots behind lower-priority tiles afterwards.
                const bool pdl_batch = h->pdl_ratio > 0.0 &&
                                       (double)B.steps.size() * 50.0 > h->pdl_ratio * (P.solve_flops / 17.0e6);
                // a streaming fit's first fold starts each batch as soon as ITS Gram is done
                CU_TRY(h, cudaStreamWaitEvent(cs, (streaming && f == 0) ? h->ev_gram[bi] : h->ev_fork, 0));
                for (size_t k = 0; k < B.steps.size(); ++k) {
                    const StepList& s = B.steps[k];
                    // Who factors the diagonal tile of panel k: its own launch (k == 0, or no fusion at all), macro tile 0
                    // of step k-1 (fused at the end), or extra CTAs at the head of THIS launch (step k-1 deferred it).
                    const bool deferred_here = h->fuse_diag && k > 0 && B.steps[k - 1].defer;
                    if (k == 0 || !h->fuse_diag) {
                        CU_TRY(h, launch_chol_diag(d_blocks, d_diag + s.diag_off, s.n_diag, (int32_t)k,
                                                   (const double*)h->sigma.p, (double*)h->lbuf.p, (double*)h->wbuf.p, wstride,
                                                   ridge, d_status, cs));
                        ++n_launch;
                        ++n_chol_launch;
                    }
                    const bool fuse_end = h->fuse_diag && !s.defer;
                    if (tma_panel) {
                        // CTAs: one per item for split-K / flag-synchronised steps and for the macro tiles that factor
                        // the next diagonal tile; otherwise up to tpc_max consecutive items (same block, same W) per CTA
                        // as long as the step keeps several waves of CTAs
                        int n_single = s.n_panel, tpc = 1;
                        if (s.nsl == 1 && !deferred_here) {
                            n_single = fuse_end ? s.n_first : 0;
                            const int rest = s.n_panel - n_single;
                            tpc = std::max(1, std::min(h->tpc_max, rest / std::max(1, h->tpc_waves * chol_panel_ctas_per_sm(B.tile_rows) * h->n_sm)));   // tpc_waves = 0: always tpc_max
                        }
                        CU_TRY(h, launch_chol_panel_tma(B.tile_rows, d_blocks, d_panel + s.panel_off, s.n_panel, n_single, tpc,
                                                        d_diag + s.diag_off, deferred_here ? s.n_diag : 0, (int32_t)k,
                                                        (const CUtensorMap*)(dblob + P.o_lmaps), h->tmap_perm == 1 ? 1 : 0, h->l2_pf | (h->next_pf << 8),
                                                        (const double*)h->sigma.p, (double*)h->lbuf.p, (double*)h->wbuf.p,
                                                        wstride, fuse_end, ridge, (double*)h->scratch.p + B.scratch_off,
                                                        (int32_t*)h->counters.p, s.group_base, d_status, (int32_t*)h->dflag.p,
                                                        pdl_batch && k > 0, cs));
                    } else {
                        CU_TRY(h, launch_chol_panel(d_blocks, d_panel + s.panel_off, s.n_panel, d_diag + s.diag_off,
                                                    deferred_here ? s.n_diag : 0, (int32_t)k, (const double*)h->sigma.p,
                                                    (double*)h->lbuf.p, (double*)h->wbuf.p, wstride, fuse_end, ridge,
                                                    (double*)h->scratch.p + B.scratch_off, (int32_t*)h->counters.p, s.group_base,
                                                    d_status, (int32_t*)h->dflag.p, pdl_batch && k > 0, cs));
                    }
                    ++n_launch;
                    ++n_chol_launch;
                }
                // the batch's back substitution follows on its own stream: the big blocks' substitutions overlap
                // the factorisation of the bulk classes, which finish last
                CU_TRY(h, cudaEventRecord(h->ev_cend[bi], cs));
                CU_TRY(h, launch_backsolve(d_blocks, d_order + B.ord_off, B.ord_n, B.big,
                                           (const double*)h->lbuf.p, inv_sqrt_n, bs, bl, P.max_mp, cs));
                ++n_launch;
                CU_TRY(h, cudaEventRecord(h->ev_join[bi], cs));
                CU_TRY(h, cudaStreamWaitEvent(st, h->ev_join[bi], 0));
            }
            if (d_var) {
                CU_TRY(h, launch_variance(d_blocks, nb, P.n_test, (const double*)h->sigma.p, (const double*)h->lbuf.p,
                                          a->sigma_s[f], (double)a->n_obs, d_var + (size_t)f * nb * P.n_test, st));
                ++n_launch;
            }
            if (a->timing) {
                // factorisation time of this fold = latest class end (events are read after a sync)
                CU_TRY(h, cudaEventRecord(h->ev[7], st));
                CU_TRY(h, cudaEventSynchronize(h->ev[7]));
                float worst = 0.f;
                for (int bi = 0; bi < nbatch && !(streaming && f == 0); ++bi) {
                    float ms = 0.f;
                    cudaEventElapsedTime(&ms, h->ev_fork, h->ev_cend[bi]);
                    worst = std::max(worst, ms);
                }
                chol_ms_total += worst;
            }
        } else {
            // reference-faithful Jacobi-PCG (pcg.cu): per-block scratch vectors live in `scratch`
            std::vector<int64_t> woff((size_t)std::max(nb, 1), 0);
            int64_t wtot = 0;
            int32_t max_ms = 8;
            for (int b = 0; b < nb; ++b) {
                const int64_t ms = P.blocks[b].ms, ml = P.blocks[b].m - P.blocks[b].ms;
                woff[b] = wtot;
                wtot += 7 * ms + ms * ml + ml * ml + 7 * ml + 8;
                max_ms = std::max<int32_t>(max_ms, (int32_t)std::max(ms, ml));
            }
            const size_t off_bytes = align_up(sizeof(int64_t) * (size_t)std::max(nb, 1), 256);
            CU_TRY(h, h->scratch.ensure(off_bytes + sizeof(double) * (size_t)std::max<int64_t>(wtot, 1)));
            CU_TRY(h, cudaMemcpyAsync(h->scratch.p, woff.data(), sizeof(int64_t) * (size_t)std::max(nb, 1), cudaMemcpyHostToDevice, st));
            CU_TRY(h, cudaStreamSynchronize(st));          // woff is a stack-lifetime host vector
            PcgArgs pa;
            pa.blocks = d_blocks;
            pa.order = d_order;
            pa.n_blocks = nb;
            pa.sigma = (const double*)h->sigma.p;
            pa.work = (double*)((uint8_t*)h->scratch.p + off_bytes);
            pa.work_off = (const int64_t*)h->scratch.p;
            pa.ridge = ridge;
            pa.sigma_s = a->sigma_s[f];
            pa.n_obs = (double)a->n_obs;
            pa.beta_s = bs;
            pa.beta_l = bl;
            pa.status = d_status;
            pa.iters = d_iters;
            CU_TRY(h, launch_pcg(pa, max_ms, st));
            ++n_launch;
        }
    }
    CU_TRY(h, cudaEventRecord(h->ev[4], st));

    // ---- download
    uint8_t* hout = (uint8_t*)h->h_out.p;
    if (n_res && !zc_beta) CU_TRY(h, cudaMemcpyAsync(hout, d_beta, sizeof(double) * n_res, cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaMemcpyAsync(hout + sizeof(double) * n_res, d_status, sizeof(int32_t) * (size_t)(2 * nb),
                              cudaMemcpyDeviceToHost, st));
    if (d_var) CU_TRY(h, cudaMemcpyAsync(a->variance_out, d_var, sizeof(double) * (size_t)a->n_folds * nb * P.n_test,
                                         cudaMemcpyDeviceToHost, st));
    if (nb > 0)     // which blocks had missing calls (decided on the device): for the work accounting and the inspection hooks
        CU_TRY(h, cudaMemcpyAsync(hout + sizeof(double) * n_res + sizeof(int32_t) * (size_t)(2 * nb), d_bflags, sizeof(int32_t) * (size_t)nb,
                                  cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaEventRecord(h->ev[5], st));
    tr.mark("all launched");
    if (tr.on && streaming) {
        for (int bi = 0; bi < nbatch; ++bi) {
            cudaEventSynchronize(h->ev_up[bi]);
            char buf[64];
            std::snprintf(buf, sizeof buf, "upload of batch %d (cls %d) done", bi, P.batches[bi].cls);
            tr.mark(buf);
        }
    }
    CU_TRY(h, cudaStreamSynchronize(st));
    tr.mark("device done");
    if (tr.on && streaming && !pcg) {
        if (tr_blob && tr_blob0) {
            float b = 0.f, b0 = 0.f;
            cudaEventElapsedTime(&b, h->ev[0], tr_blob);
            cudaEventElapsedTime(&b0, h->ev[0], tr_blob0);
            std::fprintf(stderr, "[dbslmm_b200 trace] plan blob (%.1f MB): copy starts %.2f, on the device at %.2f (device ms after fit start)\n", (double)P.blob_bytes / 1e6, b0, b);
            cudaEventDestroy(tr_blob); cudaEventDestroy(tr_blob0);
        }
        for (int c = 0; c < tr_chain; ++c) {
            float s0 = 0.f, d0 = 0.f;
            cudaEventElapsedTime(&s0, h->ev[0], tr_start[c]);
            cudaEventElapsedTime(&d0, h->ev[0], tr_dec[c]);
            std::fprintf(stderr, "[dbslmm_b200 trace] chain %d (batch %d): starts %.2f  decoded %.2f\n", c, P.up_order[c], s0, d0);
            cudaEventDestroy(tr_start[c]); cudaEventDestroy(tr_dec[c]);
        }
        for (int bi = 0; bi < nbatch; ++bi) {
            float u = 0.f, g2 = 0.f, c = 0.f, j = 0.f;
            cudaEventElapsedTime(&u, h->ev[0], h->ev_up[bi]);
            cudaEventElapsedTime(&g2, h->ev[0], h->ev_gram[bi]);
            cudaEventElapsedTime(&c, h->ev[0], h->ev_cend[bi]);
            cudaEventElapsedTime(&j, h->ev[0], h->ev_join[bi]);
            std::fprintf(stderr, "[dbslmm_b200 trace] batch %d cls %d blocks %d rows %lld: uploaded %.2f  gram done %.2f  chol done %.2f  backsolve done %.2f (device ms after fit start)\n",
                         bi, P.batches[bi].cls, P.batches[bi].ord_n, (long long)(P.batches[bi].grow1 - P.batches[bi].grow0), u, g2, c, j);
        }
    }
    {
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(h, DBSLMM_B200_ERR_CUDA, std::string("fit: ") + cudaGetErrorString(e));
    }
    if (streaming) {
        // the caller's panel buffer must not be needed after the call returns: the batch uploads are done (their batches
        // consumed them), this only waits for the rows no block uses
        CU_TRY(h, cudaEventSynchronize(h->ev_bed));
        h->bed_pending = false;
    }
    const double* hb = (const double*)hout;
    if (quad && nb > 0) std::memcpy(a->quadform_out, hb, sizeof(double) * (size_t)nb);
    for (int f = 0; f < a->n_folds && !quad; ++f) {
        // pinned staging -> caller's arrays; a genome-wide beta vector is ~9 MB, so the copy is split over a few threads
        par_memcpy(a->beta_s_out + (size_t)f * P.tot_s, hb + (size_t)f * n_out, sizeof(double) * (size_t)P.tot_s);
        if (P.tot_l) std::memcpy(a->beta_l_out + (size_t)f * P.tot_l, hb + (size_t)f * n_out + P.tot_s, sizeof(double) * (size_t)P.tot_l);
    }
    const int32_t* hs = (const int32_t*)(hout + sizeof(double) * n_res);
    int n_bad = 0;
    for (int b = 0; b < nb; ++b) {
        if (a->block_status_out) a->block_status_out[b] = hs[b];
        n_bad += (hs[b] != 0);
    }
    // which blocks took the four-plane path
    h->miss_flags.assign(hs + 2 * nb, hs + 3 * nb);
    double gram_ops = 0.0, mask_bytes = 0.0;
    for (int b = 0; b < nb; ++b) {
        const double m = P.blocks[b].m;
        gram_ops += (h->miss_flags[b] ? 4.0 : 1.0) * (double)h->n_pad * m * (m + 1.0);
        if (h->miss_flags[b]) mask_bytes += m * (double)h->n_pad;            // (upper bound: mask rows of SNPs with missing calls)
    }
    h->last_flags = a->flags | (full ? DBSLMM_B200_FLAG_FULL_SIGMA : 0);
    h->last_solver = a->solver;
    h->last_quad = quad;
    h->last_nfolds = a->n_folds;
    if (a->timing) {
        dbslmm_b200_timing* t = a->timing;
        cudaEventElapsedTime(&t->h2d_ms, h->ev[0], h->ev[1]);
        cudaEventElapsedTime(&t->decode_ms, h->ev[1], h->ev[2]);
        cudaEventElapsedTime(&t->gram_ms, h->ev[2], h->ev[3]);
        cudaEventElapsedTime(&t->solve_ms, h->ev[3], h->ev[4]);
        cudaEventElapsedTime(&t->d2h_ms, h->ev[4], h->ev[5]);
        cudaEventElapsedTime(&t->total_ms, h->ev[0], h->ev[5]);
        t->chol_ms = chol_ms_total;
        for (int c = 0; c < kNumClasses; ++c) t->class_ms[c] = 0.f;
        for (int bi = 0; bi < nbatch && !pcg && !quad && !(streaming && a->n_folds == 1); ++bi) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, h->ev_fork, h->ev_cend[bi]);
            const int slot = std::min(P.batches[bi].cls, kNumClasses - 1);
            t->class_ms[slot] = std::max(t->class_ms[slot], ms);
        }
        t->n_launches = n_launch;
        t->n_chol_launches = n_chol_launch;
        t->gram_ops = gram_ops;
        t->streamed = streaming ? 1 : 0;
        t->n_blocks_missing = 0;
        for (int b = 0; b < nb; ++b) t->n_blocks_missing += (h->miss_flags[b] != 0);
        t->solve_flops = quad ? 0.0 : P.solve_flops * (double)a->n_folds;
        t->decode_bytes = P.decode_bytes + mask_bytes;
    }
    return n_bad;
}

}  // namespace

extern "C" {

int dbslmm_b200_fit(dbslmm_b200_handle* h, const dbslmm_b200_fit_args* a) {
    struct Range { Range() { nvtxRangePushA("dbslmm_b200_fit"); } ~Range() { nvtxRangePop(); } } nvtx_range;
    if (!h || !a) return DBSLMM_B200_ERR_ARG;
    if (!a->bed && h->n_snp == 0) return fail(h, DBSLMM_B200_ERR_STATE, "fit before load_bed (and no fit_args.bed)");
    if (a->bed && (a->bed_n_snp <= 0 || a->bed_n_ref <= 1)) return fail(h, DBSLMM_B200_ERR_ARG, "fit: bad bed_n_snp / bed_n_ref");
    if (a->bed && a->bed_n_ref > decode_max_n_ref())
        return fail(h, DBSLMM_B200_ERR_ARG, "fit: bed_n_ref = " + std::to_string(a->bed_n_ref) + " is above the decoder's limit of " +
                                            std::to_string(decode_max_n_ref()) + " individuals");
    const bool quad = a->quadform_out != nullptr;
    if (a->n_blocks < 0 || !a->s_off || (!quad && (a->n_folds < 1 || !a->sigma_s || a->n_obs <= 0 || !a->beta_s_out)))
        return fail(h, DBSLMM_B200_ERR_ARG, "fit: bad arguments");
    if (quad && (a->l_off || a->test_bed || a->solver != DBSLMM_B200_SOLVER_CHOLESKY))
        return fail(h, DBSLMM_B200_ERR_ARG, "fit: quadform_out takes small-effect lists only, no variance side channel, default solver");
    if (a->n_blocks > 0 && a->s_off[a->n_blocks] > 0 && (!a->s_pos || !a->s_z))
        return fail(h, DBSLMM_B200_ERR_ARG, "fit: s_pos/s_z missing");
    if (a->l_off && a->l_off[a->n_blocks] > 0 && (!a->l_pos || !a->l_z || !a->beta_l_out))
        return fail(h, DBSLMM_B200_ERR_ARG, "fit: l_pos/l_z/beta_l_out missing");
    if (!(a->tau > 0.0 && a->tau <= 1.0)) return fail(h, DBSLMM_B200_ERR_ARG, "fit: tau must be in (0,1]");
    if (a->solver != DBSLMM_B200_SOLVER_CHOLESKY && a->solver != DBSLMM_B200_SOLVER_PCG)
        return fail(h, DBSLMM_B200_ERR_ARG, "fit: unknown solver");
    for (int f = 0; f < a->n_folds && !quad; ++f)
        if (!(a->sigma_s[f] > 0.0)) return fail(h, DBSLMM_B200_ERR_ARG, "fit: sigma_s must be > 0");
    const bool want_var = a->test_bed != nullptr;
    if (want_var) {
        if (a->solver != DBSLMM_B200_SOLVER_CHOLESKY) return fail(h, DBSLMM_B200_ERR_ARG, "fit: the variance side channel needs the Cholesky solver");
        if (a->test_n_snp <= 0 || a->test_n_total <= 1 || !a->test_indicator || !a->variance_out || (a->s_off[a->n_blocks] > 0 && !a->s_tpos) ||
            (a->l_off && a->l_off[a->n_blocks] > 0 && !a->l_tpos))
            return fail(h, DBSLMM_B200_ERR_ARG, "fit: incomplete test-data arguments for the variance side channel");
        if (a->flags & DBSLMM_B200_FLAG_PLAN_CACHED) return fail(h, DBSLMM_B200_ERR_ARG, "fit: PLAN_CACHED cannot be combined with the variance side channel");
    }
    CU_TRY(h, cudaSetDevice(h->device));
    if (!a->bed) return fit_impl(h, a, false);

    // ---- the panel comes with the call (what DBSLMMFIT::est does with its bed_str argument)
    if (h->bed_pending) { CU_TRY(h, cudaEventSynchronize(h->ev_bed)); h->bed_pending = false; }
    const bool can_stream = !want_var && !quad && a->solver == DBSLMM_B200_SOLVER_CHOLESKY && !(a->flags & DBSLMM_B200_FLAG_PLAN_CACHED) &&
                            a->n_blocks > 0 && h->stream_bed;
    if (!can_stream) {
        int rc = dbslmm_b200_load_bed(h, a->bed, a->bed_n_snp, a->bed_n_ref);
        if (rc != DBSLMM_B200_OK) return rc;
        return fit_impl(h, a, false);
    }
    const int32_t pitch = (a->bed_n_ref + 3) / 4;
    CU_TRY(h, h->bed.ensure((size_t)a->bed_n_snp * pitch + 64));
    h->n_snp = a->bed_n_snp;
    h->n_ref = a->bed_n_ref;
    h->pitch = pitch;
    h->n_pad = (a->bed_n_ref + 127) / 128 * 128;
    h->stats_valid = false;
    h->plan.valid = false;
    int rc = fit_impl(h, a, true);
    if (rc < 0) {
        // A streaming fit that failed part-way may have copies from the caller's buffer and kernels in flight, and the
        // panel on the device is incomplete: drain everything (the header promises `bed` is not needed after the call
        // returns) and forget the panel, so a later fit without fit_args.bed fails with ERR_STATE instead of decoding it.
        const std::string msg = h->err;
        cudaDeviceSynchronize();
        cudaGetLastError();
        h->n_snp = 0; h->n_ref = 0; h->pitch = 0; h->n_pad = 0;
        h->bed_pending = false;
        h->stats_valid = false;
        h->plan.valid = false;
        h->err = msg;
        return rc;
    }
    if (a->flags & DBSLMM_B200_FLAG_PANEL_SUBSET) {
        // only the rows of this call's blocks were uploaded: the device copy is no panel a later call could use
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        h->n_snp = 0; h->n_ref = 0; h->pitch = 0; h->n_pad = 0;
        h->stats_valid = false;
        h->plan.valid = false;
    }
    return rc;
}

// One fit over several GPUs: the block scheduler (dbslmm_b200_plan_shards) assigns every block to one handle, every handle
// fits its blocks from the SAME host panel (FLAG_PANEL_SUBSET: it uploads only the rows its blocks use) on its own host
// thread, and the results are written straight into the caller's block-major arrays.  No collective: LD blocks are
// independent (scr/dbslmmfit.cpp:193-213).
int dbslmm_b200_fit_multi(dbslmm_b200_handle* const* hs, int32_t n_handles, const dbslmm_b200_fit_args* a) {
    if (!hs || n_handles < 1 || !a || !hs[0]) return DBSLMM_B200_ERR_ARG;
    dbslmm_b200_handle* h0 = hs[0];
    if (n_handles == 1) return dbslmm_b200_fit(h0, a);
    if (!a->bed) return fail(h0, DBSLMM_B200_ERR_ARG, "fit_multi: the panel must come with the call (fit_args.bed)");
    if (a->test_bed || a->quadform_out || (a->flags & DBSLMM_B200_FLAG_PLAN_CACHED))
        return fail(h0, DBSLMM_B200_ERR_ARG, "fit_multi: variance side channel, quadform and PLAN_CACHED are single-GPU features");
    if (a->n_blocks < 0 || !a->s_off || a->n_folds < 1) return fail(h0, DBSLMM_B200_ERR_ARG, "fit_multi: bad arguments");
    const int nb = a->n_blocks;
    const bool with_large = a->l_off != nullptr;
    std::vector<int32_t> m_s((size_t)std::max(nb, 1)), m_l((size_t)std::max(nb, 1), 0), owner((size_t)std::max(nb, 1), 0);
    for (int b = 0; b < nb; ++b) {
        m_s[b] = a->s_off[b + 1] - a->s_off[b];
        if (with_large) m_l[b] = a->l_off[b + 1] - a->l_off[b];
    }
    int rc = dbslmm_b200_plan_shards(nb, m_s.data(), m_l.data(), a->bed_n_ref, n_handles, owner.data(), nullptr);
    if (rc != DBSLMM_B200_OK) return fail(h0, rc, "fit_multi: plan_shards failed");
    struct Shard {
        std::vector<int32_t> blocks, s_off, s_pos, l_off, l_pos, status;
        std::vector<double> s_z, l_z, beta_s, beta_l;
        dbslmm_b200_timing timing{};
        int rc = 0;
    };
    std::vector<Shard> sh((size_t)n_handles);
    const int nf = a->n_folds;
    for (int g = 0; g < n_handles; ++g) {
        Shard& S = sh[g];
        S.s_off.push_back(0);
        if (with_large) S.l_off.push_back(0);
        for (int b = 0; b < nb; ++b) {
            if (owner[b] != g) continue;
            S.blocks.push_back(b);
            S.s_pos.insert(S.s_pos.end(), a->s_pos + a->s_off[b], a->s_pos + a->s_off[b + 1]);
            S.s_z.insert(S.s_z.end(), a->s_z + a->s_off[b], a->s_z + a->s_off[b + 1]);
            S.s_off.push_back((int32_t)S.s_pos.size());
            if (with_large) {
                S.l_pos.insert(S.l_pos.end(), a->l_pos + a->l_off[b], a->l_pos + a->l_off[b + 1]);
                S.l_z.insert(S.l_z.end(), a->l_z + a->l_off[b], a->l_z + a->l_off[b + 1]);
                S.l_off.push_back((int32_t)S.l_pos.size());
            }
        }
        S.beta_s.assign(S.s_pos.size() * (size_t)nf + 1, 0.0);
        S.beta_l.assign(S.l_pos.size() * (size_t)nf + 1, 0.0);
        S.status.assign(S.blocks.size() + 1, 0);
    }
    auto run = [&](int g) {
        Shard& S = sh[g];
        if (S.blocks.empty()) return;
        dbslmm_b200_fit_args x = *a;
        x.n_blocks = (int32_t)S.blocks.size();
        x.s_off = S.s_off.data(); x.s_pos = S.s_pos.data(); x.s_z = S.s_z.data();
        x.l_off = with_large ? S.l_off.data() : nullptr;
        x.l_pos = with_large ? S.l_pos.data() : nullptr;
        x.l_z = with_large ? S.l_z.data() : nullptr;
        x.beta_s_out = S.beta_s.data();
        x.beta_l_out = with_large ? S.beta_l.data() : nullptr;
        x.block_status_out = S.status.data();
        x.timing = &S.timing;
        x.flags = a->flags | DBSLMM_B200_FLAG_PANEL_SUBSET;
        S.rc = dbslmm_b200_fit(hs[g], &x);
    };
    {
        std::vector<std::thread> th;
        for (int g = 1; g < n_handles; ++g) th.emplace_back(run, g);
        run(0);
        for (std::thread& t : th) t.join();
    }
    int n_bad = 0;
    for (int g = 0; g < n_handles; ++g) {
        if (sh[g].rc < 0) return fail(h0, sh[g].rc, "fit_multi: GPU " + std::to_string(g) + ": " + dbslmm_b200_last_error(hs[g]));
        n_bad += sh[g].rc;
    }
    // gather to the caller's block-major arrays
    const size_t tot_s = (size_t)a->s_off[nb], tot_l = with_large ? (size_t)a->l_off[nb] : 0;
    for (int g = 0; g < n_handles; ++g) {
        const Shard& S = sh[g];
        const size_t ns = S.s_pos.size(), nl = S.l_pos.size();
        for (size_t i = 0; i < S.blocks.size(); ++i) {
            const int b = S.blocks[i];
            if (a->block_status_out) a->block_status_out[b] = S.status[i];
            for (int f = 0; f < nf; ++f) {
                std::memcpy(a->beta_s_out + (size_t)f * tot_s + a->s_off[b], S.beta_s.data() + (size_t)f * ns + S.s_off[i], sizeof(double) * (size_t)m_s[b]);
                if (with_large && m_l[b] > 0)
                    std::memcpy(a->beta_l_out + (size_t)f * tot_l + a->l_off[b], S.beta_l.data() + (size_t)f * nl + S.l_off[i], sizeof(double) * (size_t)m_l[b]);
            }
        }
    }
    if (a->timing) {
        // the slowest GPU's phase times; work counters summed over the GPUs
        int slow = 0;
        double gram_ops = 0.0, solve_flops = 0.0, decode_bytes = 0.0;
        int n_launches = 0, n_chol = 0, n_miss = 0;
        for (int g = 0; g < n_handles; ++g) {
            const dbslmm_b200_timing& u = sh[g].timing;
            if (u.total_ms > sh[slow].timing.total_ms) slow = g;
            gram_ops += u.gram_ops; solve_flops += u.solve_flops; decode_bytes += u.decode_bytes;
            n_launches += u.n_launches; n_chol += u.n_chol_launches; n_miss += u.n_blocks_missing;
        }
        dbslmm_b200_timing t = sh[slow].timing;
        t.gram_ops = gram_ops; t.solve_flops = solve_flops; t.decode_bytes = decode_bytes;
        t.n_launches = n_launches; t.n_chol_launches = n_chol; t.n_blocks_missing = n_miss;
        *a->timing = t;
    }
    return n_bad;
}

int dbslmm_b200_host_alloc(dbslmm_b200_handle* h, uint64_t bytes, void** out) {
    if (!h || !out) return DBSLMM_B200_ERR_ARG;
    *out = nullptr;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaHostAlloc(out, (size_t)std::max<uint64_t>(bytes, 1), cudaHostAllocPortable));
    return DBSLMM_B200_OK;
}
void dbslmm_b200_host_free(dbslmm_b200_handle* h, void* p) {
    if (!h || !p) return;
    cudaSetDevice(h->device);
    cudaFreeHost(p);
}

int dbslmm_b200_score_prefetch(dbslmm_b200_handle* h, const uint8_t* bed_val, int64_t n_snp_val, int32_t n_val) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (!bed_val || n_snp_val <= 0 || n_val <= 0) return fail(h, DBSLMM_B200_ERR_ARG, "score_prefetch: bad arguments");
    CU_TRY(h, cudaSetDevice(h->device));
    if (h->val_inflight) { CU_TRY(h, cudaEventSynchronize(h->ev_val)); h->val_inflight = false; }
    const size_t bytes = (size_t)n_snp_val * ((n_val + 3) / 4);
    CU_TRY(h, h->vbed.ensure(bytes + 64));
    CU_TRY(h, h->vstats.ensure(sizeof(SnpStat) * (size_t)n_snp_val));
    h->val_host = bed_val;
    h->val_n_snp = n_snp_val;
    h->val_n = n_val;
    h->val_announced = true;
    return DBSLMM_B200_OK;
}

int dbslmm_b200_score(dbslmm_b200_handle* h, const uint8_t* bed_val, int64_t n_snp_val, int32_t n_val,
                      const int32_t* pos, const uint8_t* flip, int64_t n_scored, const double* beta,
                      int32_t n_folds, double* scores_out, float* kernel_ms_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    // bed_val == NULL: the panel announced by score_prefetch (or left resident by the previous score call)
    const bool prefetched = bed_val == nullptr;
    if (prefetched) {
        if (!h->val_announced && !h->val_inflight && h->val_n_snp == 0) return fail(h, DBSLMM_B200_ERR_STATE, "score: no validation panel (bed_val == NULL without score_prefetch)");
        n_snp_val = h->val_n_snp;
        n_val = h->val_n;
    }
    if (n_snp_val <= 0 || n_val <= 0 || n_scored < 0 || n_folds < 1 || !scores_out || (n_scored > 0 && (!pos || !beta)))
        return fail(h, DBSLMM_B200_ERR_ARG, "score: bad arguments");
    if (n_scored > INT32_MAX) return fail(h, DBSLMM_B200_ERR_ARG, "score: too many SNPs");
    for (int64_t j = 0; j < n_scored; ++j)
        if (pos[j] < 0 || pos[j] >= n_snp_val) return fail(h, DBSLMM_B200_ERR_ARG, "score: pos out of range of the validation .bed");
    CU_TRY(h, cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int32_t pitch = (n_val + 3) / 4;
    const size_t bytes = (size_t)n_snp_val * pitch;
    const int n_chunks = prs_slices(h->n_sm, n_val, n_scored);
    const int nf_pass = std::min(n_folds, 3);            // folds per pass of the scoring kernel (score.cu: kMaxFolds)
    // work buffer: pos | flip | beta | partial | scores
    size_t o = 0;
    auto place = [&](size_t b) { size_t r = o; o = align_up(o + b, 256); return r; };
    const size_t o_pos = place(sizeof(int32_t) * (size_t)n_scored), o_flip = place((size_t)n_scored),
                 o_beta = place(sizeof(double) * (size_t)n_scored * n_folds),
                 o_part = place(sizeof(double) * (size_t)n_chunks * nf_pass * n_val),
                 o_sc = place(sizeof(double) * (size_t)n_folds * n_val);
    if (!prefetched) {
        if (h->val_inflight) { CU_TRY(h, cudaEventSynchronize(h->ev_val)); h->val_inflight = false; }
        h->val_announced = false;
        CU_TRY(h, h->vbed.ensure(bytes + 64));
        CU_TRY(h, h->vstats.ensure(sizeof(SnpStat) * (size_t)n_snp_val));
    }
    CU_TRY(h, h->vwork.ensure(o));
    uint8_t* w = (uint8_t*)h->vwork.p;
    if (!prefetched) {
        CU_TRY(h, cudaMemcpyAsync(h->vbed.p, bed_val, bytes, cudaMemcpyHostToDevice, st));
        CU_TRY(h, cudaMemsetAsync((uint8_t*)h->vbed.p + bytes, 0xFF, 64, st));
        h->val_n_snp = n_snp_val;
        h->val_n = n_val;
    } else {
        if (h->val_announced) { int rc = issue_val_upload(h); if (rc != DBSLMM_B200_OK) return rc; }   // no fit came in between
        if (h->val_inflight) CU_TRY(h, cudaStreamWaitEvent(st, h->ev_val, 0));
    }
    if (n_scored) {
        CU_TRY(h, cudaMemcpyAsync(w + o_pos, pos, sizeof(int32_t) * (size_t)n_scored, cudaMemcpyHostToDevice, st));
        if (flip) CU_TRY(h, cudaMemcpyAsync(w + o_flip, flip, (size_t)n_scored, cudaMemcpyHostToDevice, st));
        CU_TRY(h, cudaMemcpyAsync(w + o_beta, beta, sizeof(double) * (size_t)n_scored * n_folds, cudaMemcpyHostToDevice, st));
    }
    if (!prefetched) CU_TRY(h, launch_snp_stats((const uint8_t*)h->vbed.p, n_snp_val, n_val, (SnpStat*)h->vstats.p, h->n_sm, st));
    CU_TRY(h, cudaMemsetAsync(w + o_sc, 0, sizeof(double) * (size_t)n_folds * n_val, st));
    CU_TRY(h, cudaEventRecord(h->ev[0], st));
    for (int f0 = 0; f0 < n_folds; f0 += 3) {
        const int nf = std::min(3, n_folds - f0);
        CU_TRY(h, launch_prs((const uint8_t*)h->vbed.p, n_val, (const SnpStat*)h->vstats.p, (const int32_t*)(w + o_pos),
                             flip ? (const uint8_t*)(w + o_flip) : nullptr, (const double*)(w + o_beta) + (size_t)f0 * n_scored,
                             n_scored, (int32_t)n_scored, nf, n_chunks, (double*)(w + o_part),
                             (double*)(w + o_sc) + (size_t)f0 * n_val, st));
    }
    CU_TRY(h, cudaEventRecord(h->ev[1], st));
    CU_TRY(h, cudaMemcpyAsync(scores_out, w + o_sc, sizeof(double) * (size_t)n_folds * n_val, cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaStreamSynchronize(st));
    h->val_inflight = false;                 // (the stream waited for its event)
    if (kernel_ms_out) cudaEventElapsedTime(kernel_ms_out, h->ev[0], h->ev[1]);
    return DBSLMM_B200_OK;
}

// Streaming scorer.  A chunk is rows_cap scored rows (the last one fewer) gathered in scored order by host workers into a
// pinned staging slot laid out as  genotype rows (pitch bytes each) | beta slice [n_folds][rows] | flip slice [rows],  so
// one cudaMemcpyAsync on the copy stream carries all of it.  Three staging slots and two device slots: the gather of chunk
// k + 2, the copy of chunk k + 1 and the kernels of chunk k (statistics, counts, one scoring pass per 3 folds) overlap.
static constexpr uint64_t kStreamChunkDefault = 64ull << 20;
struct ChunkLayout {
    int64_t j0 = 0;
    int32_t rows = 0;
    size_t o_beta = 0, o_flip = 0, bytes = 0;
};
static ChunkLayout chunk_layout(int64_t j0, int32_t rows, int64_t pitch, int32_t n_folds) {
    ChunkLayout c;
    c.j0 = j0;
    c.rows = rows;
    c.o_beta = align_up((size_t)rows * pitch + 4, 256);          // + 4: the statistics kernel reads whole words past the last row
    c.o_flip = c.o_beta + sizeof(double) * (size_t)n_folds * rows;
    c.bytes = align_up(c.o_flip + (size_t)rows, 256);
    return c;
}

}  // extern "C"

// The host gather ring of the streaming calls (dbslmm_b200_score_stream, dbslmm_b200_ldscore).  Chunk k is gathered by the
// host worker pool into pinned staging slot k % 3 and crosses PCIe in ONE cudaMemcpyAsync on the copy stream into device
// slot k % 2; its kernels run on the main stream.  The gather of chunk k + 2, the copy of chunk k + 1 and the kernels of
// chunk k overlap.  gather(k, dst, group) fills staging slot dst (pieces may go to the pool under `group`); launch(k, dev)
// enqueues the kernels of chunk k, whose bytes are at `dev`, on h->stream.  Events ev_chunk[4 (ev0 + k) + 0..3] record the
// begin and end of the chunk's copy and kernels.  Returns with the work enqueued; the caller synchronises h->stream.
template <class BytesOf, class Gather, class Launch>
static int stream_chunks(dbslmm_b200_handle* h, int64_t n_chunks, size_t max_bytes, int64_t ev0, BytesOf bytes_of, Gather gather,
                         Launch launch) {
    cudaStream_t st = h->stream, cp = h->up_stream;
    const int n_pin = (int)std::min<int64_t>(3, std::max<int64_t>(n_chunks, 1)), n_dev = std::min(2, n_pin);
    for (int i = 0; i < n_pin; ++i) CU_TRY(h, h->s_pin[i].ensure(max_bytes));
    for (int i = 0; i < n_dev; ++i) CU_TRY(h, h->s_dev[i].ensure(max_bytes));
    while (h->ev_chunk.size() < (size_t)(4 * (ev0 + n_chunks))) {
        cudaEvent_t e;
        CU_TRY(h, cudaEventCreate(&e));
        h->ev_chunk.push_back(e);
    }
    HostPool& pool = host_pool();
    TaskGroup groups[3];
    struct Drain { HostPool& p; TaskGroup* g; ~Drain() { for (int i = 0; i < 3; ++i) p.wait(g[i]); } } drain{pool, groups};
    for (int64_t k = 0; k < std::min<int64_t>(2, n_chunks); ++k) gather(k, (uint8_t*)h->s_pin[k % 3].p, groups[k % 3]);
    for (int64_t k = 0; k < n_chunks; ++k) {
        const int p = (int)(k % 3), d = (int)(k % 2);
        cudaEvent_t* ev = h->ev_chunk.data() + 4 * (ev0 + k);
        pool.wait(groups[p]);
        uint8_t* dev = (uint8_t*)h->s_dev[d].p;
        if (k >= 2) CU_TRY(h, cudaStreamWaitEvent(cp, h->ev_slot_free[d], 0));          // the kernels of chunk k - 2 are done with it
        CU_TRY(h, cudaEventRecord(ev[0], cp));
        CU_TRY(h, cudaMemcpyAsync(dev, h->s_pin[p].p, bytes_of(k), cudaMemcpyHostToDevice, cp));
        CU_TRY(h, cudaEventRecord(ev[1], cp));
        CU_TRY(h, cudaEventRecord(h->ev_pin_free[p], cp));
        CU_TRY(h, cudaEventRecord(h->ev_copied[d], cp));
        CU_TRY(h, cudaStreamWaitEvent(st, h->ev_copied[d], 0));
        CU_TRY(h, cudaEventRecord(ev[2], st));
        const int rc = launch(k, (const uint8_t*)dev);
        if (rc != DBSLMM_B200_OK) return rc;
        CU_TRY(h, cudaEventRecord(ev[3], st));
        CU_TRY(h, cudaEventRecord(h->ev_slot_free[d], st));
        if (k + 2 < n_chunks) {
            if (k + 2 >= 3) CU_TRY(h, cudaEventSynchronize(h->ev_pin_free[(k + 2) % 3]));    // the copy of chunk k - 1 has left it
            gather(k + 2, (uint8_t*)h->s_pin[(k + 2) % 3].p, groups[(k + 2) % 3]);
        }
    }
    return DBSLMM_B200_OK;
}

// Summed kernel time of the chunks [ev0, ev0 + n) of stream_chunks, once h->stream has been synchronised.  With
// DBSLMM_B200_TRACE, one line per chunk: its copy and kernel intervals relative to the call's first copy (do the kernels
// hide behind the next copy?).
template <class RowsOf, class BytesOf>
static int chunk_kernel_ms(dbslmm_b200_handle* h, const char* label, int64_t ev0, int64_t n, RowsOf rows_of, BytesOf bytes_of, float* out) {
    const Trace tr;
    float kms = 0.0f;
    for (int64_t k = 0; k < n; ++k) {
        const cudaEvent_t* ev = h->ev_chunk.data() + 4 * (ev0 + k);
        float t = 0.0f;
        CU_TRY(h, cudaEventElapsedTime(&t, ev[2], ev[3]));
        kms += t;
        if (tr.on) {
            float c0 = 0, c1 = 0, k0 = 0, k1 = 0;
            cudaEventElapsedTime(&c0, h->ev_chunk[0], ev[0]); cudaEventElapsedTime(&c1, h->ev_chunk[0], ev[1]);
            cudaEventElapsedTime(&k0, h->ev_chunk[0], ev[2]); cudaEventElapsedTime(&k1, h->ev_chunk[0], ev[3]);
            std::fprintf(stderr, "[dbslmm_b200 trace] %s chunk %lld rows %lld bytes %zu copy %.4f %.4f kernels %.4f %.4f ms\n", label,
                         (long long)k, (long long)rows_of(k), (size_t)bytes_of(k), c0, c1, k0, k1);
        }
    }
    *out = kms;
    return DBSLMM_B200_OK;
}

// .bed rows src(0..nr) -> dst (pitch bytes each), in pieces of >= 2 MB for the pool's workers
template <class Src>
static void gather_bed_rows(HostPool& pool, const uint8_t* bed, int64_t pitch, uint8_t* dst, int64_t nr, TaskGroup& g, Src src) {
    const int64_t per = std::max<int64_t>(1, ((int64_t)2 << 20) / pitch);
    for (int64_t r0 = 0; r0 < nr; r0 += per) {
        const int64_t r1 = std::min<int64_t>(nr, r0 + per);
        pool.submit(g, [=]() { for (int64_t r = r0; r < r1; ++r) std::memcpy(dst + r * pitch, bed + (int64_t)src(r) * pitch, (size_t)pitch); });
    }
}

// Pass 1 of the LD calls: per-row statistics of .bed rows rows[0..n_rows) -> hs, streamed as chunks [0, *n_chunks) of
// stream_chunks; *ms = their kernel time.
static int ld_stats_pass(dbslmm_b200_handle* h, const uint8_t* bed, int32_t n_ref, const int32_t* rows, int64_t n_rows,
                         const char* label, std::vector<SnpStat>& hs, int64_t* n_chunks, float* ms) {
    cudaStream_t st = h->stream;
    const int64_t pitch = (n_ref + 3) / 4;
    HostPool& pool = host_pool();
    const int64_t rows1 = std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(n_rows, 1), (int64_t)(kStreamChunkDefault / (uint64_t)pitch)));
    const int64_t n1 = (n_rows + rows1 - 1) / rows1;
    CU_TRY(h, h->ld_stats.ensure(sizeof(SnpStat) * (size_t)std::max<int64_t>(n_rows, 1)));
    SnpStat* d_stats = (SnpStat*)h->ld_stats.p;
    auto rows_of1 = [&](int64_t k) { return std::min<int64_t>(rows1, n_rows - k * rows1); };
    auto bytes_of1 = [&](int64_t k) { return align_up((size_t)std::max<int64_t>(rows_of1(k), 0) * pitch + 4, 256); };   // + 4: whole-word reads
    int rc = stream_chunks(h, n1, bytes_of1(0), 0, bytes_of1,
                           [&](int64_t k, uint8_t* dst, TaskGroup& g) {
                               const int64_t j0 = k * rows1;
                               gather_bed_rows(pool, bed, pitch, dst, rows_of1(k), g, [=](int64_t r) { return rows[j0 + r]; });
                           },
                           [&](int64_t k, const uint8_t* dev) -> int {
                               CU_TRY(h, launch_chunk_stats(dev, (int32_t)rows_of1(k), n_ref, d_stats + k * rows1, nullptr, h->n_sm, st));
                               return DBSLMM_B200_OK;
                           });
    if (rc != DBSLMM_B200_OK) return rc;
    hs.assign((size_t)n_rows, SnpStat{});
    if (n_rows > 0) CU_TRY(h, cudaMemcpyAsync(hs.data(), d_stats, sizeof(SnpStat) * (size_t)n_rows, cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaStreamSynchronize(st));
    *n_chunks = n1;
    return chunk_kernel_ms(h, label, 0, n1, rows_of1, bytes_of1, ms);
}

extern "C" {

int dbslmm_b200_score_stream(dbslmm_b200_handle* h, const uint8_t* bed_val, int64_t n_snp_val, int32_t n_val,
                             const int32_t* pos, const uint8_t* flip, int64_t n_scored, const double* beta, int32_t n_folds,
                             uint64_t chunk_bytes, double* scores_out, int32_t* cnt_out, int32_t* cnt2_out, int32_t* n_empty_out,
                             float* kernel_ms_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (!bed_val || n_snp_val <= 0 || n_val <= 0 || n_scored < 0 || n_folds < 1 || !scores_out || (n_scored > 0 && (!pos || !beta)))
        return fail(h, DBSLMM_B200_ERR_ARG, "score_stream: bad arguments");
    if (n_val > kScoreMaxNVal)
        return fail(h, DBSLMM_B200_ERR_ARG, "score_stream: n_val = " + std::to_string(n_val) + " is above the limit of " +
                                            std::to_string(kScoreMaxNVal) + " individuals (int32 row sums)");
    if (n_scored > INT32_MAX / 2) return fail(h, DBSLMM_B200_ERR_ARG, "score_stream: too many SNPs (CNT = 2 x calls must fit in int32)");
    for (int64_t j = 0; j < n_scored; ++j)
        if (pos[j] < 0 || pos[j] >= n_snp_val) return fail(h, DBSLMM_B200_ERR_ARG, "score_stream: pos out of range of the .bed");
    CU_TRY(h, cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int64_t pitch = (n_val + 3) / 4;
    const bool counts = cnt_out || cnt2_out;
    const uint64_t budget = chunk_bytes ? chunk_bytes : kStreamChunkDefault;
    // rows per chunk: a function of chunk_bytes and n_val only, so fold f of an F-fold call sums exactly like a 1-fold call
    const int64_t rows_cap = std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(n_scored, 1), (int64_t)(budget / (uint64_t)(pitch + 1))));
    const int64_t n_chunks = (n_scored + rows_cap - 1) / rows_cap;
    const ChunkLayout full = chunk_layout(0, (int32_t)rows_cap, pitch, n_folds);
    const int32_t nf_pass = std::min(n_folds, 3);             // folds per scoring pass (score.cu: kMaxFolds)
    // work buffer: chunk statistics | partial sums of one pass | scores | cnt | cnt2 | empty-row count
    size_t o = 0;
    auto place = [&](size_t b) { size_t r = o; o = align_up(o + b, 256); return r; };
    const size_t o_stats = place(sizeof(SnpStat) * (size_t)rows_cap),
                 o_part = place(sizeof(double) * (size_t)prs_slices(h->n_sm, n_val, rows_cap) * nf_pass * n_val),
                 o_sc = place(sizeof(double) * (size_t)n_folds * n_val),
                 o_cnt = place(sizeof(int32_t) * (size_t)n_val), o_cnt2 = place(sizeof(int32_t) * (size_t)n_val),
                 o_empty = place(sizeof(int32_t));
    CU_TRY(h, h->s_work.ensure(o));
    uint8_t* w = (uint8_t*)h->s_work.p;
    double* scores = (double*)(w + o_sc);
    int32_t* cnt = (int32_t*)(w + o_cnt);
    int32_t* cnt2 = (int32_t*)(w + o_cnt2);
    int32_t* n_empty = (int32_t*)(w + o_empty);
    CU_TRY(h, cudaMemsetAsync(scores, 0, sizeof(double) * (size_t)n_folds * n_val, st));
    CU_TRY(h, cudaMemsetAsync(cnt, 0, o - o_cnt, st));

    // host gather of chunk k, cut into pieces of >= 2 MB for the pool's workers
    HostPool& pool = host_pool();
    auto layout_of = [&](int64_t k) { const int64_t j0 = k * rows_cap; return chunk_layout(j0, (int32_t)std::min(rows_cap, n_scored - j0), pitch, n_folds); };
    auto gather = [&](int64_t k, uint8_t* dst, TaskGroup& g) {
        const ChunkLayout c = layout_of(k);
        const int64_t per = std::max<int64_t>(1, ((int64_t)2 << 20) / pitch);
        for (int64_t r0 = 0; r0 < c.rows; r0 += per) {
            const int64_t r1 = std::min<int64_t>(c.rows, r0 + per);
            pool.submit(g, [=]() {
                for (int64_t r = r0; r < r1; ++r) std::memcpy(dst + r * pitch, bed_val + (int64_t)pos[c.j0 + r] * pitch, (size_t)pitch);
            });
        }
        for (int f = 0; f < n_folds; ++f)
            std::memcpy(dst + c.o_beta + sizeof(double) * (size_t)f * c.rows, beta + (size_t)f * n_scored + c.j0, sizeof(double) * (size_t)c.rows);
        if (flip) std::memcpy(dst + c.o_flip, flip + c.j0, (size_t)c.rows);
    };
    auto launch = [&](int64_t k, const uint8_t* dev) -> int {
        const ChunkLayout c = layout_of(k);
        SnpStat* stats = (SnpStat*)(w + o_stats);
        const uint8_t* cflip = flip ? dev + c.o_flip : nullptr;
        const int32_t n_slices = prs_slices(h->n_sm, n_val, c.rows);
        CU_TRY(h, launch_chunk_stats(dev, c.rows, n_val, stats, n_empty, h->n_sm, st));
        if (counts) CU_TRY(h, launch_score_counts(dev, n_val, cflip, c.rows, n_slices, cnt, cnt2, st));
        for (int f0 = 0; f0 < n_folds; f0 += 3)
            CU_TRY(h, launch_prs_chunk(dev, n_val, stats, cflip, (const double*)(dev + c.o_beta) + (size_t)f0 * c.rows, c.rows, c.rows,
                                       std::min(3, n_folds - f0), n_slices, (double*)(w + o_part), scores + (size_t)f0 * n_val, st));
        return DBSLMM_B200_OK;
    };
    int rc = stream_chunks(h, n_chunks, full.bytes, 0, [&](int64_t k) { return layout_of(k).bytes; }, gather, launch);
    if (rc != DBSLMM_B200_OK) return rc;
    CU_TRY(h, cudaMemcpyAsync(scores_out, scores, sizeof(double) * (size_t)n_folds * n_val, cudaMemcpyDeviceToHost, st));
    if (cnt_out) CU_TRY(h, cudaMemcpyAsync(cnt_out, cnt, sizeof(int32_t) * (size_t)n_val, cudaMemcpyDeviceToHost, st));
    if (cnt2_out) CU_TRY(h, cudaMemcpyAsync(cnt2_out, cnt2, sizeof(int32_t) * (size_t)n_val, cudaMemcpyDeviceToHost, st));
    if (n_empty_out) CU_TRY(h, cudaMemcpyAsync(n_empty_out, n_empty, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaStreamSynchronize(st));
    float kms = 0.0f;
    rc = chunk_kernel_ms(h, "score_stream", 0, n_chunks, [&](int64_t k) { return (int64_t)layout_of(k).rows; },
                         [&](int64_t k) { return layout_of(k).bytes; }, &kms);
    if (rc != DBSLMM_B200_OK) return rc;
    if (kernel_ms_out) *kernel_ms_out = kms;
    return DBSLMM_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// LD Scores (ldsc --l2), see ldscore.cu.  Pass 1 streams the requested rows through launch_chunk_stats, and the host keeps
// ldsc's SNPs, builds the windows over the kept SNPs of every chromosome, the band of 128 x 128 tiles and the slot layout.
// Pass 2 streams segments of consecutive row tiles together with the halo of rows their windows reach (decode -> group
// flags -> band kernels, one chunk per segment); ld_reduce_kernel then adds each SNP's slots.
// With annotations (dbslmm_b200_ldscore_annot) the same host path lists the FULL band instead -- tiles (T, P) for every
// tile P that T's windows reach, on both sides -- so a row tile depends only on its own segment (which then starts at its
// left halo, 128 tlo[T0]).  Each segment's chunk also carries its annotation rows; its slots (row, tile, half,
// annotation) live only while the segment is processed: ld_annot_reduce_kernel adds them right after its band kernels.
// ---------------------------------------------------------------------------------------------
namespace {
struct LdSeg {
    int64_t T0 = 0, T1 = 0;           // row tiles [T0, T1)
    int64_t R0 = 0, R1 = 0;           // padded rows on the device: [128 T0, 128 (last tile column reached + 1))
    int64_t K0 = 0, K1 = 0;           // kept SNPs among them
    int64_t n_tiles = 0;
    int64_t n_slots = 0;              // annotated: partial sums of the segment
    size_t o_src = 0, o_crow = 0, o_mrow = 0, o_rows = 0, o_tiles = 0, bytes = 0;
    size_t o_annot = 0, o_sbase = 0, o_nslot = 0;    // annotated: annotation rows [R1 - R0][C], slot base and count per row tile
    size_t o_rid = 0;                 // pairs: the caller's row index of each padded row
};
}  // namespace

int dbslmm_b200_ld_windows(const double* coord, int64_t m, double max_dist, int32_t* lo_out, int32_t* hi_out) {
    if (m < 0 || m > INT32_MAX || (m > 0 && (!lo_out || !hi_out)) || !(max_dist >= 0)) return DBSLMM_B200_ERR_ARG;
    auto x = [&](int64_t k) { return coord ? coord[k] : (double)k; };
    int64_t lo = 0, hi = 0;
    for (int64_t k = 0; k < m; ++k) {
        while (std::fabs(x(k) - x(lo)) > max_dist) ++lo;                 // ldsc's getBlockLefts
        hi = std::max(hi, k);
        while (hi + 1 < m && std::fabs(x(hi + 1) - x(k)) <= max_dist) ++hi;
        lo_out[k] = (int32_t)lo;
        hi_out[k] = (int32_t)hi;
    }
    return DBSLMM_B200_OK;
}

// n_annot = 0: dbslmm_b200_ldscore (annot NULL, l2_out [n_rows]); n_annot >= 1: dbslmm_b200_ldscore_annot.
static int ldscore_impl(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref, const int32_t* rows,
                        int64_t n_rows, const int32_t* chr_off, int32_t n_chr, int32_t wind_kind, const double* coord,
                        double max_dist, double maf_min, int64_t segment_rows, const double* annot, int32_t n_annot,
                        uint8_t* kept_out, double* maf_out, double* l2_out, int32_t* guard_out, float* kernel_ms_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    const char* who = n_annot > 0 ? "ldscore_annot: " : "ldscore: ";
    auto bad = [&](const std::string& m) { return fail(h, DBSLMM_B200_ERR_ARG, who + m); };
    const bool an = n_annot > 0;
    const int64_t C = an ? n_annot : 1;             // values per row of l2_out
    if (!bed || n_snp <= 0 || n_ref <= 0 || n_rows < 0 || n_chr < 0 || !chr_off || (n_rows > 0 && !rows))
        return bad("bad arguments");
    if (n_ref > decode_max_n_ref())
        return bad("n_ref = " + std::to_string(n_ref) + " is above the limit of " + std::to_string(decode_max_n_ref()) +
                   " individuals (the decoder stages whole .bed rows in shared memory)");
    if (n_rows > INT32_MAX) return bad("n_rows = " + std::to_string(n_rows) + " is above INT32_MAX");
    if (wind_kind != DBSLMM_B200_LD_WIND_COORD && wind_kind != DBSLMM_B200_LD_WIND_SNPS) return bad("unknown window kind " + std::to_string(wind_kind));
    if (wind_kind == DBSLMM_B200_LD_WIND_COORD && n_rows > 0 && !coord) return bad("a coordinate window needs coord");
    if (wind_kind == DBSLMM_B200_LD_WIND_SNPS && coord) return bad("a window in SNPs takes coord = NULL");
    if (!std::isfinite(max_dist) || max_dist < 0 ||
        (wind_kind == DBSLMM_B200_LD_WIND_SNPS && (max_dist != std::floor(max_dist) || max_dist > (double)INT32_MAX)))
        return bad("max_dist must be finite and >= 0 (a whole number for a window in SNPs)");
    if (!std::isfinite(maf_min) || maf_min < 0 || maf_min >= 0.5) return bad("maf_min must lie in [0, 0.5)");
    if (segment_rows < 0 || segment_rows % 128 != 0) return bad("segment_rows must be 0 or a positive multiple of 128");
    if (chr_off[0] != 0 || chr_off[n_chr] != n_rows) return bad("bad chromosome offsets: chr_off[0] must be 0 and chr_off[n_chr] = n_rows");
    for (int32_t c = 0; c < n_chr; ++c)
        if (chr_off[c + 1] < chr_off[c]) return bad("bad chromosome offsets: chr_off[" + std::to_string(c + 1) + "] < chr_off[" + std::to_string(c) + "]");
    for (int64_t i = 0; i < n_rows; ++i)
        if (rows[i] < 0 || rows[i] >= n_snp) return bad("rows[" + std::to_string(i) + "] = " + std::to_string(rows[i]) + " is out of range of the .bed");
    if (wind_kind == DBSLMM_B200_LD_WIND_COORD)
        for (int32_t c = 0; c < n_chr; ++c)
            for (int64_t i = chr_off[c]; i < chr_off[c + 1]; ++i) {
                if (!std::isfinite(coord[i])) return bad("coord[" + std::to_string(i) + "] is not finite");
                if (i > chr_off[c] && coord[i] < coord[i - 1])
                    return bad("the coordinates of chromosome " + std::to_string(c) + " are not sorted: coord[" + std::to_string(i) + "] < coord[" +
                               std::to_string(i - 1) + "]");
            }
    if (an) {
        for (int64_t x = 0; x < n_rows * C; ++x)
            if (!std::isfinite(annot[x]))
                return bad("annot[" + std::to_string(x / C) + "][" + std::to_string(x % C) + "] is not finite");
    }
    CU_TRY(h, cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int64_t pitch = (n_ref + 3) / 4;
    const int32_t n_pad = (n_ref + 127) / 128 * 128;
    HostPool& pool = host_pool();
    auto gather_rows = [&](uint8_t* dst, const int64_t nr, TaskGroup& g, auto src) { gather_bed_rows(pool, bed, pitch, dst, nr, g, src); };

    // ---- pass 1: per-row statistics of every requested row
    std::vector<SnpStat> hs;
    float ms1 = 0.0f;
    int64_t n1 = 0;
    int rc = ld_stats_pass(h, bed, n_ref, rows, n_rows, "ldscore pass1", hs, &n1, &ms1);
    if (rc != DBSLMM_B200_OK) return rc;

    // ---- kept SNPs (ldsc's __filter_snps_maf__): min(f, 1 - f) > maf_min and missing + het < n
    std::vector<uint8_t> keep((size_t)n_rows);
    for (int64_t i = 0; i < n_rows; ++i) {
        const SnpStat& s = hs[i];
        const double f = s.n_nonmiss > 0 ? (double)s.sum / (2.0 * (double)s.n_nonmiss) : 0.0;
        const double maf = std::min(f, 1.0 - f);
        const int64_t hom2 = ((int64_t)s.sumsq - s.sum) / 2, het = (int64_t)s.sum - 2 * hom2, miss = (int64_t)n_ref - s.n_nonmiss;
        keep[i] = (maf > maf_min && miss + het < n_ref) ? 1 : 0;
        if (maf_out) maf_out[i] = maf;
        if (kept_out) kept_out[i] = keep[i];
    }
    // ---- windows (ldsc's getBlockLefts over the kept SNPs of each chromosome, both ends), tiles and slots.  Chromosome c
    // takes the padded rows [128 T_c, 128 (T_c + ceil(m_c / 128))); its kept SNP k sits at padded row 128 T_c + k.
    std::vector<int64_t> kept, kpad, klo, khi;          // per kept SNP: row index, padded row, window (padded rows, inclusive)
    std::vector<int64_t> tlo, thi, tbase;               // per row tile: tile columns reached, first slot
    std::vector<int32_t> tnslot;
    int64_t slots_total = 0;
    for (int32_t c = 0; c < n_chr; ++c) {
        const int64_t T_c = (int64_t)tlo.size(), k0 = (int64_t)kept.size();
        for (int64_t i = chr_off[c]; i < chr_off[c + 1]; ++i) if (keep[i]) kept.push_back(i);
        const int64_t m = (int64_t)kept.size() - k0;
        std::vector<double> x;
        if (wind_kind == DBSLMM_B200_LD_WIND_COORD)
            for (int64_t k = 0; k < m; ++k) x.push_back(coord[kept[k0 + k]]);
        std::vector<int32_t> lo((size_t)m), hi((size_t)m);
        dbslmm_b200_ld_windows(x.empty() ? nullptr : x.data(), m, max_dist, lo.data(), hi.data());
        for (int64_t k = 0; k < m; ++k) {
            kpad.push_back(128 * T_c + k);
            klo.push_back(128 * T_c + lo[k]);
            khi.push_back(128 * T_c + hi[k]);
        }
        if (guard_out) guard_out[c] = (m > 0 && klo.back() == 128 * T_c) ? 1 : 0;
        for (int64_t t = 0; t < (m + 127) / 128; ++t) {
            tlo.push_back(klo[k0 + 128 * t] / 128);
            thi.push_back(khi[k0 + std::min(m, 128 * t + 128) - 1] / 128);
            tnslot.push_back((int32_t)(thi.back() - tlo.back() + 1));
            tbase.push_back(slots_total);
            slots_total += 128 * (int64_t)tnslot.back();
        }
    }
    const int64_t n_trows = (int64_t)tlo.size(), n_prows = 128 * n_trows, n_kept = (int64_t)kept.size();
    if (l2_out)
        for (int64_t i = 0; i < n_rows * C; ++i) l2_out[i] = std::nan("");
    if (n_kept == 0 || !l2_out) {                       // (l2_out NULL: the statistics pass only)
        if (kernel_ms_out) *kernel_ms_out = ms1;
        return DBSLMM_B200_OK;
    }

    // ---- segments: consecutive row tiles; nonzero segment_rows fixes their size, else 64 MB of .bed rows (and annotation
    // rows) while the code rows of the widest segment (with its halo), and with annotations its partial sums, take at most
    // half of the free device memory
    int64_t max_nslot = 0;
    for (int64_t T = 0; T < n_trows; ++T) max_nslot = std::max<int64_t>(max_nslot, tnslot[T]);
    if (an && 2 * max_nslot * C > INT32_MAX)
        return bad("a window reaches " + std::to_string(max_nslot) + " tiles of 128 SNPs: too wide for " + std::to_string(C) + " annotations");
    auto plan = [&](int64_t seg_tiles, std::vector<LdSeg>& segs) {
        segs.clear();
        int64_t cap = 0;
        for (int64_t T0 = 0; T0 < n_trows; T0 += seg_tiles) {
            LdSeg S;
            S.T0 = T0;
            S.T1 = std::min(n_trows, T0 + seg_tiles);
            S.R0 = 128 * (an ? tlo[S.T0] : S.T0);
            S.R1 = 128 * (thi[S.T1 - 1] + 1);
            S.K0 = std::lower_bound(kpad.begin(), kpad.end(), S.R0) - kpad.begin();
            S.K1 = std::lower_bound(kpad.begin(), kpad.end(), S.R1) - kpad.begin();
            for (int64_t T = S.T0; T < S.T1; ++T) {
                S.n_tiles += thi[T] - (an ? tlo[T] : T) + 1;
                S.n_slots += an ? 2 * 128 * C * tnslot[T] : 0;
            }
            const int64_t nr = S.K1 - S.K0, np = S.R1 - S.R0, nt = S.T1 - S.T0;
            S.o_src = align_up((size_t)nr * pitch + 16, 256);        // + 16: the decoder's row copies are 16-byte aligned
            S.o_crow = align_up(S.o_src + sizeof(uint32_t) * nr, 256);
            S.o_mrow = align_up(S.o_crow + sizeof(int32_t) * nr, 256);
            S.o_rows = align_up(S.o_mrow + sizeof(int32_t) * nr, 256);
            S.o_tiles = align_up(S.o_rows + sizeof(LdRow) * np, 256);
            S.bytes = align_up(S.o_tiles + sizeof(LdTile) * S.n_tiles, 256);
            if (an) {
                S.o_annot = S.bytes;
                S.o_sbase = align_up(S.o_annot + sizeof(double) * (size_t)(np * C), 256);
                S.o_nslot = align_up(S.o_sbase + sizeof(int64_t) * nt, 256);
                S.bytes = align_up(S.o_nslot + sizeof(int32_t) * nt, 256);
            }
            cap = std::max(cap, np);
            segs.push_back(S);
        }
        return cap;
    };
    auto seg_slots = [&](const std::vector<LdSeg>& segs) {
        int64_t m = 0;
        for (const LdSeg& S : segs) m = std::max(m, S.n_slots);
        return m;
    };
    std::vector<LdSeg> segs;
    const uint64_t row_bytes = (uint64_t)(128 * pitch) + (an ? (uint64_t)(128 * 8 * C) : 0);
    int64_t seg_tiles = segment_rows > 0 ? segment_rows / 128 : std::max<int64_t>(1, (int64_t)(kStreamChunkDefault / row_bytes));
    int64_t cap = plan(seg_tiles, segs);
    size_t free_b = 0, total_b = 0;
    CU_TRY(h, cudaMemGetInfo(&free_b, &total_b));
    auto need = [&](int64_t cp) { return (double)cp * (2.0 * n_pad + 2.0 + 48.0); };
    if (segment_rows == 0)
        while (seg_tiles > 1 && need(cap) + 8.0 * (double)seg_slots(segs) > 0.5 * (double)free_b) cap = plan(seg_tiles = (seg_tiles + 1) / 2, segs);
    const int64_t n_slots = an ? seg_slots(segs) : slots_total;
    const double out_bytes = an ? 8.0 * (double)(n_prows * C) : 0.0;
    if (need(cap) + 8.0 * (double)n_slots + out_bytes > 0.9 * (double)free_b)
        return fail(h, DBSLMM_B200_ERR_NOMEM, who + std::string("a segment of ") + std::to_string(cap) + " rows (with the halo its windows reach) and " +
                                             std::to_string(n_slots) + " partial sums do not fit in device memory");
    size_t max_bytes = 0;
    for (const LdSeg& S : segs) max_bytes = std::max(max_bytes, S.bytes);

    // ---- device buffers of pass 2: code rows [genotype rows 0..cap) [mask rows cap..2 cap), the decoder's dirty map (all
    // ones: every mask row is written the first time its position is used), its per-row outputs, group flags, slots
    CU_TRY(h, h->ld_codes.ensure((size_t)2 * cap * n_pad));
    CU_TRY(h, h->ld_dirty.ensure((size_t)2 * cap));
    CU_TRY(h, cudaMemsetAsync(h->ld_dirty.p, 1, (size_t)2 * cap, st));
    size_t o = 0;
    auto place = [&](size_t b) { size_t r = o; o = align_up(o + b, 256); return r; };
    const size_t o_rowN = place(sizeof(int32_t) * cap), o_rowS = place(sizeof(int32_t) * cap), o_rowR = place(sizeof(double) * cap),
                 o_rowC = place(sizeof(double2) * cap), o_gfl = place(sizeof(int32_t) * (cap / 128 + 1));
    CU_TRY(h, h->ld_work.ensure(o));
    uint8_t* wk = (uint8_t*)h->ld_work.p;
    int32_t* rowN = (int32_t*)(wk + o_rowN);
    int32_t* gflags = (int32_t*)(wk + o_gfl);
    CU_TRY(h, h->ld_slots.ensure(sizeof(double) * (size_t)n_slots));
    double* slots = (double*)h->ld_slots.p;
    if (!an) CU_TRY(h, cudaMemsetAsync(slots, 0, sizeof(double) * (size_t)slots_total, st));     // (annotated: every slot is written)
    double* l2a = nullptr;                                  // annotated: [n_prows][C]
    if (an) {
        CU_TRY(h, h->ld_red.ensure(sizeof(double) * (size_t)(n_prows * C)));
        l2a = (double*)h->ld_red.p;
    }
    CUtensorMap tmap;
    rc = make_tensor_map(h, &tmap, h->ld_codes.p, 2 * cap, n_pad, 128);
    if (rc != DBSLMM_B200_OK) return rc;

    auto gather2 = [&](int64_t k, uint8_t* dst, TaskGroup& g) {
        const LdSeg& S = segs[k];
        const int64_t nr = S.K1 - S.K0, np = S.R1 - S.R0;
        const int64_t* kr = kept.data() + S.K0;
        gather_rows(dst, nr, g, [=](int64_t r) { return rows[kr[r]]; });
        uint32_t* src = (uint32_t*)(dst + S.o_src);
        int32_t* crow = (int32_t*)(dst + S.o_crow);
        int32_t* mrow = (int32_t*)(dst + S.o_mrow);
        LdRow* lr = (LdRow*)(dst + S.o_rows);
        LdTile* tl = (LdTile*)(dst + S.o_tiles);
        for (int64_t p = 0; p < np; ++p) lr[p] = LdRow{0.0, std::nan(""), 0, 1, 0, -1};
        for (int64_t g2 = 0; g2 < nr; ++g2) {
            const int64_t kk = S.K0 + g2, p = kpad[kk] - S.R0;
            const SnpStat& s = hs[kept[kk]];
            const double d = (double)((int64_t)s.n_nonmiss * s.sumsq - (int64_t)s.sum * s.sum);
            src[g2] = (uint32_t)g2;
            crow[g2] = (int32_t)p;
            mrow[g2] = (int32_t)(p + cap);
            lr[p] = LdRow{(double)s.sum, 1.0 / std::sqrt((double)s.n_nonmiss * d), s.n_nonmiss, (int32_t)(klo[kk] - S.R0),
                          (int32_t)(khi[kk] - S.R0), (int32_t)g2};
        }
        int64_t n = 0;
        if (!an) {
            for (int64_t T = S.T0; T < S.T1; ++T)
                for (int64_t c = T; c <= thi[T]; ++c)
                    tl[n++] = LdTile{(int32_t)(T - S.T0), (int32_t)(c - S.T0), tnslot[T], tnslot[c], tbase[T] + (c - tlo[T]), tbase[c] + (T - tlo[c])};
            return;
        }
        // full band: scored tile T on the TMEM lanes (tj), partner tile P (ti); tiles are numbered from the segment's first row
        double* ann = (double*)(dst + S.o_annot);
        int64_t* sbase = (int64_t*)(dst + S.o_sbase);
        int32_t* nslot = (int32_t*)(dst + S.o_nslot);
        std::fill(ann, ann + np * C, 0.0);
        for (int64_t kk = S.K0; kk < S.K1; ++kk) std::memcpy(ann + (kpad[kk] - S.R0) * C, annot + kept[kk] * C, sizeof(double) * (size_t)C);
        const int64_t D0 = S.R0 / 128;
        int64_t sb = 0;
        for (int64_t T = S.T0; T < S.T1; ++T) {
            sbase[T - S.T0] = sb;
            nslot[T - S.T0] = tnslot[T];
            for (int64_t P = tlo[T]; P <= thi[T]; ++P)
                tl[n++] = LdTile{(int32_t)(P - D0), (int32_t)(T - D0), (int32_t)(2 * tnslot[T] * C), 0, sb + (P - tlo[T]) * 2 * C, 0};
            sb += 2 * 128 * C * tnslot[T];
        }
    };
    auto launch2 = [&](int64_t k, const uint8_t* dev) -> int {
        const LdSeg& S = segs[k];
        const int64_t nr = S.K1 - S.K0, ngrp = (S.R1 - S.R0) / 128;
        CU_TRY(h, launch_decode_rows(dev, n_ref, n_pad, (const uint32_t*)(dev + S.o_src), (const int32_t*)(dev + S.o_crow),
                                     (const int32_t*)(dev + S.o_mrow), 0, nr, 1.0, (int8_t*)h->ld_codes.p, (uint8_t*)h->ld_dirty.p,
                                     rowN, (int32_t*)(wk + o_rowS), (double*)(wk + o_rowR), (double2*)(wk + o_rowC), nullptr, h->n_sm, st));
        CU_TRY(h, cudaMemsetAsync(gflags, 0, sizeof(int32_t) * (size_t)(ngrp + 1), st));
        const LdRow* lr = (const LdRow*)(dev + S.o_rows);
        CU_TRY(h, launch_ld_group_flags(lr, (int32_t)ngrp, rowN, n_ref, gflags, gflags + ngrp, st));
        LdArgs a;
        a.tiles = (const LdTile*)(dev + S.o_tiles);
        a.n_tiles = (int32_t)S.n_tiles;
        a.nk = n_pad / 128;
        a.n_ref = n_ref;
        a.mask_off = (int32_t)cap;
        a.rows = lr;
        a.gflags = gflags;
        a.any = gflags + ngrp;
        a.slots = slots;
        if (!an) {
            CU_TRY(h, launch_ld_band(tmap, a, h->n_sm, st));
            return DBSLMM_B200_OK;
        }
        a.annot = (const double*)(dev + S.o_annot);
        a.n_annot = n_annot;
        a.alpha = 1.0 / (n_ref > 2 ? (double)(n_ref - 2) : (double)n_ref);
        CU_TRY(h, launch_ld_band_annot(tmap, a, h->n_sm, st));
        CU_TRY(h, launch_ld_annot_reduce(slots, (const int64_t*)(dev + S.o_sbase), (const int32_t*)(dev + S.o_nslot), lr,
                                         128 * S.T0 - S.R0, 128 * (S.T1 - S.T0), n_annot, l2a + 128 * S.T0 * C, st));
        return DBSLMM_B200_OK;
    };
    const int64_t n2 = (int64_t)segs.size();
    auto bytes_of2 = [&](int64_t k) { return segs[k].bytes; };
    rc = stream_chunks(h, n2, max_bytes, n1, bytes_of2, gather2, launch2);
    if (rc != DBSLMM_B200_OK) return rc;
    if (an) {                                           // the sums are in: back to the caller's rows
        std::vector<double> l2p((size_t)(n_prows * C));
        CU_TRY(h, cudaMemcpyAsync(l2p.data(), l2a, sizeof(double) * l2p.size(), cudaMemcpyDeviceToHost, st));
        CU_TRY(h, cudaStreamSynchronize(st));
        for (int64_t kk = 0; kk < n_kept; ++kk) std::memcpy(l2_out + kept[kk] * C, l2p.data() + kpad[kk] * C, sizeof(double) * (size_t)C);
        float ms2 = 0.0f;
        rc = chunk_kernel_ms(h, "ldscore_annot pass2", n1, n2, [&](int64_t k) { return segs[k].R1 - segs[k].R0; }, bytes_of2, &ms2);
        if (rc != DBSLMM_B200_OK) return rc;
        if (kernel_ms_out) *kernel_ms_out = ms1 + ms2;
        return DBSLMM_B200_OK;
    }

    // ---- every SNP's slots in ascending tile-column order, the unbiased-r^2 affine map, back to the caller's rows
    std::vector<int32_t> wcount((size_t)n_prows, 0);
    for (int64_t kk = 0; kk < n_kept; ++kk) wcount[kpad[kk]] = (int32_t)(khi[kk] - klo[kk] + 1);
    o = 0;
    const size_t o_tb = place(sizeof(int64_t) * n_trows), o_tn = place(sizeof(int32_t) * n_trows), o_wc = place(sizeof(int32_t) * n_prows),
                 o_l2 = place(sizeof(double) * n_prows);
    CU_TRY(h, h->ld_red.ensure(o));
    uint8_t* rd = (uint8_t*)h->ld_red.p;
    CU_TRY(h, cudaMemcpyAsync(rd + o_tb, tbase.data(), sizeof(int64_t) * n_trows, cudaMemcpyHostToDevice, st));
    CU_TRY(h, cudaMemcpyAsync(rd + o_tn, tnslot.data(), sizeof(int32_t) * n_trows, cudaMemcpyHostToDevice, st));
    CU_TRY(h, cudaMemcpyAsync(rd + o_wc, wcount.data(), sizeof(int32_t) * n_prows, cudaMemcpyHostToDevice, st));
    const double denom = n_ref > 2 ? (double)(n_ref - 2) : (double)n_ref;
    CU_TRY(h, cudaEventRecord(h->ev[0], st));
    CU_TRY(h, launch_ld_reduce(slots, (const int64_t*)(rd + o_tb), (const int32_t*)(rd + o_tn), (const int32_t*)(rd + o_wc), n_prows,
                               1.0 / denom, (double*)(rd + o_l2), st));
    CU_TRY(h, cudaEventRecord(h->ev[1], st));
    std::vector<double> l2p((size_t)n_prows);
    CU_TRY(h, cudaMemcpyAsync(l2p.data(), rd + o_l2, sizeof(double) * n_prows, cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaStreamSynchronize(st));
    for (int64_t kk = 0; kk < n_kept; ++kk) l2_out[kept[kk]] = l2p[kpad[kk]];
    float ms2 = 0.0f, msr = 0.0f;
    rc = chunk_kernel_ms(h, "ldscore pass2", n1, n2, [&](int64_t k) { return segs[k].R1 - segs[k].R0; }, bytes_of2, &ms2);
    if (rc != DBSLMM_B200_OK) return rc;
    CU_TRY(h, cudaEventElapsedTime(&msr, h->ev[0], h->ev[1]));
    if (kernel_ms_out) *kernel_ms_out = ms1 + ms2 + msr;
    return DBSLMM_B200_OK;
}

int dbslmm_b200_ldscore(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref, const int32_t* rows,
                        int64_t n_rows, const int32_t* chr_off, int32_t n_chr, int32_t wind_kind, const double* coord,
                        double max_dist, double maf_min, int64_t segment_rows, uint8_t* kept_out, double* maf_out,
                        double* l2_out, int32_t* guard_out, float* kernel_ms_out) {
    return ldscore_impl(h, bed, n_snp, n_ref, rows, n_rows, chr_off, n_chr, wind_kind, coord, max_dist, maf_min, segment_rows,
                        nullptr, 0, kept_out, maf_out, l2_out, guard_out, kernel_ms_out);
}

int dbslmm_b200_ldscore_annot(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref, const int32_t* rows,
                              int64_t n_rows, const int32_t* chr_off, int32_t n_chr, int32_t wind_kind, const double* coord,
                              double max_dist, double maf_min, int64_t segment_rows, const double* annot, int32_t n_annot,
                              uint8_t* kept_out, double* maf_out, double* l2_out, int32_t* guard_out, float* kernel_ms_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (n_annot < 1 || n_annot > DBSLMM_B200_LD_MAX_ANNOT)
        return fail(h, DBSLMM_B200_ERR_ARG, "ldscore_annot: n_annot = " + std::to_string(n_annot) + " must lie in [1, " +
                                            std::to_string(DBSLMM_B200_LD_MAX_ANNOT) + "]");
    if (!annot) return fail(h, DBSLMM_B200_ERR_ARG, "ldscore_annot: annot is NULL");
    return ldscore_impl(h, bed, n_snp, n_ref, rows, n_rows, chr_off, n_chr, wind_kind, coord, max_dist, maf_min, segment_rows,
                        annot, n_annot, kept_out, maf_out, l2_out, guard_out, kernel_ms_out);
}

// ---------------------------------------------------------------------------------------------
// SNP pairs (plink --r2), see ldscore.cu.  Pass 1 is ldscore's statistics pass; every row of a chromosome (usable or not)
// then takes a padded row from a 128-row boundary, so positions in rows and padded rows differ by a constant within a
// chromosome.  A row tile T lists the tiles (T, P), T <= P <= the tile of its last row's window end.  Segments of
// consecutive row tiles with their right halo are streamed as in ldscore; for each, the count pass and the offsets scan
// run, the host reads the per-row offsets and cuts the segment into ranges of row tiles whose pairs fit the pair buffer,
// and each range is emitted, copied to pinned buffer (range number % 2) and handed to the sink while the next range runs.
// ---------------------------------------------------------------------------------------------
static constexpr int64_t kLdPairBuf = (int64_t)1 << 23;      // pairs of the device buffer (12 bytes each)

int dbslmm_b200_ld_pairs(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref, const int32_t* rows,
                         int64_t n_rows, const int32_t* chr_off, int32_t n_chr, const double* coord, int32_t max_snps,
                         double max_dist, double r2_min, int64_t segment_rows, dbslmm_b200_ld_sink sink, void* user,
                         uint8_t* usable_out, int64_t* n_pairs_out, int64_t* n_miss_pairs_out, float* kernel_ms_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    auto bad = [&](const std::string& m) { return fail(h, DBSLMM_B200_ERR_ARG, "ld_pairs: " + m); };
    if (!bed || n_snp <= 0 || n_ref <= 0 || n_rows < 0 || n_chr < 0 || !chr_off || (n_rows > 0 && (!rows || !coord)))
        return bad("bad arguments");
    if (!sink) return bad("sink is NULL");
    if (n_ref > decode_max_n_ref())
        return bad("n_ref = " + std::to_string(n_ref) + " is above the limit of " + std::to_string(decode_max_n_ref()) +
                   " individuals (the decoder stages whole .bed rows in shared memory)");
    if (n_rows > INT32_MAX) return bad("n_rows = " + std::to_string(n_rows) + " is above INT32_MAX");
    if (max_snps < 1) return bad("max_snps must be >= 1");
    if (!(max_dist >= 0)) return bad("max_dist must be >= 0");
    if (std::isnan(r2_min)) return bad("r2_min is NaN");
    if (segment_rows < 0 || segment_rows % 128 != 0) return bad("segment_rows must be 0 or a positive multiple of 128");
    if (chr_off[0] != 0 || chr_off[n_chr] != n_rows) return bad("bad chromosome offsets: chr_off[0] must be 0 and chr_off[n_chr] = n_rows");
    for (int32_t c = 0; c < n_chr; ++c)
        if (chr_off[c + 1] < chr_off[c]) return bad("bad chromosome offsets: chr_off[" + std::to_string(c + 1) + "] < chr_off[" + std::to_string(c) + "]");
    for (int64_t i = 0; i < n_rows; ++i)
        if (rows[i] < 0 || rows[i] >= n_snp) return bad("rows[" + std::to_string(i) + "] = " + std::to_string(rows[i]) + " is out of range of the .bed");
    for (int32_t c = 0; c < n_chr; ++c)
        for (int64_t i = chr_off[c]; i < chr_off[c + 1]; ++i) {
            if (!std::isfinite(coord[i])) return bad("coord[" + std::to_string(i) + "] is not finite");
            if (i > chr_off[c] && coord[i] < coord[i - 1])
                return bad("the coordinates of chromosome " + std::to_string(c) + " are not sorted: coord[" + std::to_string(i) + "] < coord[" +
                           std::to_string(i - 1) + "]");
        }
    CU_TRY(h, cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int64_t pitch = (n_ref + 3) / 4;
    const int32_t n_pad = (n_ref + 127) / 128 * 128;
    HostPool& pool = host_pool();

    // ---- pass 1: statistics; usable rows have a called genotype and nonzero variance
    std::vector<SnpStat> hs;
    float ms = 0.0f;
    int64_t n1 = 0;
    int rc = ld_stats_pass(h, bed, n_ref, rows, n_rows, "ld_pairs pass1", hs, &n1, &ms);
    if (rc != DBSLMM_B200_OK) return rc;
    std::vector<uint8_t> usable((size_t)n_rows);
    for (int64_t i = 0; i < n_rows; ++i) {
        const SnpStat& x = hs[i];
        usable[i] = (x.n_nonmiss > 0 && (int64_t)x.n_nonmiss * x.sumsq - (int64_t)x.sum * x.sum > 0) ? 1 : 0;
        if (usable_out) usable_out[i] = usable[i];
    }

    // ---- padded rows, windows (hi: the last partner's position), tiles; ub: the most pairs a row tile can have
    std::vector<int64_t> prow((size_t)n_rows), hi((size_t)n_rows), trow0, thi, ub;
    for (int32_t c = 0; c < n_chr; ++c) {
        const int64_t i0 = chr_off[c], m = chr_off[c + 1] - i0, T_c = (int64_t)thi.size();
        int64_t j = 0;
        for (int64_t k = 0; k < m; ++k) {
            j = std::max(j, k);
            while (j + 1 < m && j + 1 - k <= (int64_t)max_snps - 1 && coord[i0 + j + 1] - coord[i0 + k] <= max_dist) ++j;
            prow[i0 + k] = 128 * T_c + k;
            hi[i0 + k] = i0 + j;
        }
        for (int64_t t = 0; t < (m + 127) / 128; ++t) {
            const int64_t a0 = i0 + 128 * t, a1 = std::min(i0 + m, a0 + 128);
            trow0.push_back(a0);
            thi.push_back(prow[hi[a1 - 1]] / 128);
            int64_t u = 0;
            for (int64_t a = a0; a < a1; ++a) u += usable[a] ? hi[a] - a : 0;
            ub.push_back(u);
        }
    }
    const int64_t n_trows = (int64_t)thi.size();
    trow0.push_back(n_rows);
    std::vector<int64_t> upad;                          // padded rows of the usable rows (the decoded ones)
    std::vector<int32_t> urow;
    for (int64_t i = 0; i < n_rows; ++i) if (usable[i]) { upad.push_back(prow[i]); urow.push_back((int32_t)i); }
    int64_t ub_max = 1, ub_sum = 0;
    for (int64_t u : ub) { ub_max = std::max(ub_max, u); ub_sum += u; }
    const int64_t pcap = std::max(ub_max, std::min(kLdPairBuf, ub_sum));
    int64_t n_pairs = 0, n_miss = 0;
    if (upad.empty()) {                                 // no row can form a pair: the sink still sees every row
        std::vector<int64_t> off((size_t)n_rows + 1, 0);
        if (n_rows > 0 && sink(user, 0, n_rows, off.data(), nullptr, nullptr) != 0)
            return fail(h, DBSLMM_B200_ERR_SINK, "ld_pairs: the sink returned nonzero");
        if (n_pairs_out) *n_pairs_out = 0;
        if (n_miss_pairs_out) *n_miss_pairs_out = 0;
        if (kernel_ms_out) *kernel_ms_out = ms;
        return DBSLMM_B200_OK;
    }

    // ---- segments (as ldscore's): 64 MB of .bed rows, halved while the code rows with their halo and the count slots take
    // more than half of the free device memory; a nonzero segment_rows fixes them
    auto plan = [&](int64_t seg_tiles, std::vector<LdSeg>& segs) {
        segs.clear();
        int64_t cap = 0;
        for (int64_t T0 = 0; T0 < n_trows; T0 += seg_tiles) {
            LdSeg S;
            S.T0 = T0;
            S.T1 = std::min(n_trows, T0 + seg_tiles);
            S.R0 = 128 * S.T0;
            S.R1 = 128 * (thi[S.T1 - 1] + 1);
            S.K0 = std::lower_bound(upad.begin(), upad.end(), S.R0) - upad.begin();
            S.K1 = std::lower_bound(upad.begin(), upad.end(), S.R1) - upad.begin();
            for (int64_t T = S.T0; T < S.T1; ++T) {
                S.n_tiles += thi[T] - T + 1;
                S.n_slots += 2 * 128 * (thi[T] - T + 1);
            }
            const int64_t nr = S.K1 - S.K0, np = S.R1 - S.R0, nt = S.T1 - S.T0;
            S.o_src = align_up((size_t)nr * pitch + 16, 256);
            S.o_crow = align_up(S.o_src + sizeof(uint32_t) * nr, 256);
            S.o_mrow = align_up(S.o_crow + sizeof(int32_t) * nr, 256);
            S.o_rows = align_up(S.o_mrow + sizeof(int32_t) * nr, 256);
            S.o_tiles = align_up(S.o_rows + sizeof(LdRow) * np, 256);
            S.o_rid = align_up(S.o_tiles + sizeof(LdTile) * S.n_tiles, 256);
            S.o_sbase = align_up(S.o_rid + sizeof(int32_t) * np, 256);
            S.o_nslot = align_up(S.o_sbase + sizeof(int64_t) * nt, 256);
            S.bytes = align_up(S.o_nslot + sizeof(int32_t) * nt, 256);
            cap = std::max(cap, np);
            segs.push_back(S);
        }
        return cap;
    };
    auto seg_slots = [&](const std::vector<LdSeg>& segs) {
        int64_t m = 0;
        for (const LdSeg& S : segs) m = std::max(m, S.n_slots);
        return m;
    };
    std::vector<LdSeg> segs;
    int64_t seg_tiles = segment_rows > 0 ? segment_rows / 128 : std::max<int64_t>(1, (int64_t)(kStreamChunkDefault / (uint64_t)(128 * pitch)));
    int64_t cap = plan(seg_tiles, segs);
    size_t free_b = 0, total_b = 0;
    CU_TRY(h, cudaMemGetInfo(&free_b, &total_b));
    auto need = [&](int64_t cp) { return (double)cp * (2.0 * n_pad + 2.0 + 48.0); };
    if (segment_rows == 0)
        while (seg_tiles > 1 && need(cap) + 12.0 * (double)seg_slots(segs) > 0.5 * (double)free_b) cap = plan(seg_tiles = (seg_tiles + 1) / 2, segs);
    const int64_t n_slots = seg_slots(segs), max_srows = 128 * std::min(seg_tiles, n_trows);
    if (need(cap) + 12.0 * (double)n_slots + 12.0 * (double)pcap > 0.9 * (double)free_b)
        return fail(h, DBSLMM_B200_ERR_NOMEM, "ld_pairs: a segment of " + std::to_string(cap) + " rows (with the halo its windows reach), " +
                                              std::to_string(n_slots) + " count slots and a buffer of " + std::to_string(pcap) +
                                              " pairs do not fit in device memory");
    size_t max_bytes = 0;
    for (const LdSeg& S : segs) max_bytes = std::max(max_bytes, S.bytes);

    // ---- device buffers: code rows and dirty map (as ldscore), decoder outputs, group flags, error flag and missing-call
    // count; count slots | slot offsets | row offsets; the pair buffer b | r; the two pinned pair buffers
    CU_TRY(h, h->ld_codes.ensure((size_t)2 * cap * n_pad));
    CU_TRY(h, h->ld_dirty.ensure((size_t)2 * cap));
    CU_TRY(h, cudaMemsetAsync(h->ld_dirty.p, 1, (size_t)2 * cap, st));
    size_t o = 0;
    auto place = [&](size_t b) { size_t r = o; o = align_up(o + b, 256); return r; };
    const size_t o_rowN = place(sizeof(int32_t) * cap), o_rowS = place(sizeof(int32_t) * cap), o_rowR = place(sizeof(double) * cap),
                 o_rowC = place(sizeof(double2) * cap), o_gfl = place(sizeof(int32_t) * (cap / 128 + 1)),
                 o_err = place(sizeof(int32_t)), o_nmiss = place(sizeof(unsigned long long));
    CU_TRY(h, h->ld_work.ensure(o));
    uint8_t* wk = (uint8_t*)h->ld_work.p;
    int32_t* rowN = (int32_t*)(wk + o_rowN);
    int32_t* gflags = (int32_t*)(wk + o_gfl);
    int32_t* d_err = (int32_t*)(wk + o_err);
    unsigned long long* d_nmiss = (unsigned long long*)(wk + o_nmiss);
    CU_TRY(h, cudaMemsetAsync(wk + o_err, 0, o - o_err, st));
    o = 0;
    const size_t o_cnt = place(sizeof(int32_t) * n_slots), o_off = place(sizeof(int64_t) * n_slots),
                 o_roff = place(sizeof(int64_t) * (max_srows + 1));
    CU_TRY(h, h->ld_slots.ensure(o));
    uint8_t* sl = (uint8_t*)h->ld_slots.p;
    int32_t* d_cnt = (int32_t*)(sl + o_cnt);
    int64_t* d_off = (int64_t*)(sl + o_off);
    int64_t* d_roff = (int64_t*)(sl + o_roff);
    const size_t o_pr = align_up(sizeof(int32_t) * (size_t)pcap, 256);
    CU_TRY(h, h->ld_red.ensure(o_pr + sizeof(double) * (size_t)pcap));
    int32_t* d_pb = (int32_t*)h->ld_red.p;
    double* d_pr = (double*)((uint8_t*)h->ld_red.p + o_pr);
    const size_t o_flag = align_up(o_pr + sizeof(double) * (size_t)pcap, 256);     // the error flag as of the range's emit
    for (PinBuf& b : h->ld_pin) CU_TRY(h, b.ensure(o_flag + sizeof(int32_t)));
    CUtensorMap tmap;
    rc = make_tensor_map(h, &tmap, h->ld_codes.p, 2 * cap, n_pad, 128);
    if (rc != DBSLMM_B200_OK) return rc;
    struct Events {
        cudaEvent_t e[8] = {};
        ~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
    } ev;                                               // count pass begin / end; per pinned buffer: emit begin / end, copied
    for (cudaEvent_t& x : ev.e) CU_TRY(h, cudaEventCreate(&x));

    // ---- the range handed to the sink next: pinned buffer x (-1: no pairs, nothing on the device), rows a0 .. a1
    struct Range { int x = -1; int64_t a0 = 0, a1 = 0, n = 0; std::vector<int64_t> off; bool on = false; } pend;
    int64_t n_ranges = 0;
    auto flush = [&]() -> int {
        if (!pend.on) return DBSLMM_B200_OK;
        pend.on = false;
        const int32_t* pb = nullptr;
        const double* pr = nullptr;
        if (pend.x >= 0) {
            CU_TRY(h, cudaEventSynchronize(ev.e[2 + 3 * pend.x + 2]));
            float t = 0.0f;
            CU_TRY(h, cudaEventElapsedTime(&t, ev.e[2 + 3 * pend.x], ev.e[2 + 3 * pend.x + 1]));
            ms += t;
            const uint8_t* pin = (const uint8_t*)h->ld_pin[pend.x].p;
            if (*(const int32_t*)(pin + o_flag))       // checked before the sink sees the range
                return fail(h, DBSLMM_B200_ERR_CUDA, "ld_pairs: the emit pass wrote other pairs than the count pass counted (rows " +
                                                     std::to_string(pend.a0) + ".." + std::to_string(pend.a1 - 1) + ")");
            pb = (const int32_t*)pin;
            pr = (const double*)(pin + o_pr);
        }
        n_pairs += pend.n;
        if (sink(user, pend.a0, pend.a1, pend.off.data(), pb, pr) != 0)
            return fail(h, DBSLMM_B200_ERR_SINK, "ld_pairs: the sink returned nonzero for rows " + std::to_string(pend.a0) + ".." +
                                                 std::to_string(pend.a1 - 1));
        return DBSLMM_B200_OK;
    };

    auto gather2 = [&](int64_t k, uint8_t* dst, TaskGroup& g) {
        const LdSeg& S = segs[k];
        const int64_t nr = S.K1 - S.K0, np = S.R1 - S.R0;
        const int32_t* ur = urow.data() + S.K0;
        gather_bed_rows(pool, bed, pitch, dst, nr, g, [=](int64_t r) { return rows[ur[r]]; });
        uint32_t* src = (uint32_t*)(dst + S.o_src);
        int32_t* crow = (int32_t*)(dst + S.o_crow);
        int32_t* mrow = (int32_t*)(dst + S.o_mrow);
        LdRow* lr = (LdRow*)(dst + S.o_rows);
        LdTile* tl = (LdTile*)(dst + S.o_tiles);
        int32_t* rid = (int32_t*)(dst + S.o_rid);
        int64_t* sbase = (int64_t*)(dst + S.o_sbase);
        int32_t* nslot = (int32_t*)(dst + S.o_nslot);
        for (int64_t p = 0; p < np; ++p) { lr[p] = LdRow{0.0, std::nan(""), 0, 1, -1, -1}; rid[p] = -1; }
        for (int64_t T = S.T0; T <= thi[S.T1 - 1] && T < n_trows; ++T)
            for (int64_t i = trow0[T]; i < trow0[T + 1]; ++i) rid[prow[i] - S.R0] = (int32_t)i;
        for (int64_t g2 = 0; g2 < nr; ++g2) {
            const int64_t i = urow[S.K0 + g2], p = prow[i] - S.R0;
            const SnpStat& x = hs[i];
            const double d = (double)((int64_t)x.n_nonmiss * x.sumsq - (int64_t)x.sum * x.sum);
            src[g2] = (uint32_t)g2;
            crow[g2] = (int32_t)p;
            mrow[g2] = (int32_t)(p + cap);
            lr[p] = LdRow{(double)x.sum, 1.0 / std::sqrt((double)x.n_nonmiss * d), x.n_nonmiss, 0, (int32_t)(prow[hi[i]] - S.R0), (int32_t)g2};
        }
        int64_t n = 0, sb = 0;
        for (int64_t T = S.T0; T < S.T1; ++T) {
            const int32_t ns = (int32_t)(thi[T] - T + 1);
            sbase[T - S.T0] = sb;
            nslot[T - S.T0] = ns;
            for (int64_t P = T; P <= thi[T]; ++P)
                tl[n++] = LdTile{(int32_t)(P - S.T0), (int32_t)(T - S.T0), 2 * ns, 0, sb + 2 * (P - T), 0};
            sb += 2 * 128 * (int64_t)ns;
        }
    };
    CU_TRY(h, h->ld_roff.ensure(sizeof(int64_t) * (size_t)(max_srows + 1)));
    const int64_t* hroff = (const int64_t*)h->ld_roff.p;
    auto launch2 = [&](int64_t k, const uint8_t* dev) -> int {
        const LdSeg& S = segs[k];
        const int64_t nr = S.K1 - S.K0, ngrp = (S.R1 - S.R0) / 128, nsr = 128 * (S.T1 - S.T0);
        CU_TRY(h, cudaEventRecord(ev.e[0], st));
        CU_TRY(h, launch_decode_rows(dev, n_ref, n_pad, (const uint32_t*)(dev + S.o_src), (const int32_t*)(dev + S.o_crow),
                                     (const int32_t*)(dev + S.o_mrow), 0, nr, 1.0, (int8_t*)h->ld_codes.p, (uint8_t*)h->ld_dirty.p,
                                     rowN, (int32_t*)(wk + o_rowS), (double*)(wk + o_rowR), (double2*)(wk + o_rowC), nullptr, h->n_sm, st));
        CU_TRY(h, cudaMemsetAsync(gflags, 0, sizeof(int32_t) * (size_t)(ngrp + 1), st));
        const LdRow* lr = (const LdRow*)(dev + S.o_rows);
        CU_TRY(h, launch_ld_group_flags(lr, (int32_t)ngrp, rowN, n_ref, gflags, gflags + ngrp, st));
        LdArgs a{};
        a.tiles = (const LdTile*)(dev + S.o_tiles);
        a.n_tiles = (int32_t)S.n_tiles;
        a.nk = n_pad / 128;
        a.n_ref = n_ref;
        a.mask_off = (int32_t)cap;
        a.rows = lr;
        a.gflags = gflags;
        a.any = gflags + ngrp;
        LdPairArgs p{};
        p.r2_min = r2_min;
        p.cnt = d_cnt;
        CU_TRY(h, launch_ld_pairs(tmap, a, p, false, h->n_sm, st));
        CU_TRY(h, launch_ld_pair_scan(d_cnt, (const int64_t*)(dev + S.o_sbase), (const int32_t*)(dev + S.o_nslot), nsr, d_off, d_roff, st));
        CU_TRY(h, cudaEventRecord(ev.e[1], st));
        CU_TRY(h, cudaMemcpyAsync(h->ld_roff.p, d_roff, sizeof(int64_t) * (size_t)(nsr + 1), cudaMemcpyDeviceToHost, st));
        int r = flush();                                // the previous range's sink runs while this segment is counted
        if (r != DBSLMM_B200_OK) return r;
        CU_TRY(h, cudaStreamSynchronize(st));
        float t = 0.0f;
        CU_TRY(h, cudaEventElapsedTime(&t, ev.e[0], ev.e[1]));
        ms += t;
        // ranges of row tiles [Ta, Tb) whose pairs fit the buffer (one tile always does: pcap >= its bound)
        std::vector<int64_t> tfirst((size_t)(S.T1 - S.T0) + 1, 0);
        for (int64_t T = S.T0; T < S.T1; ++T) tfirst[T - S.T0 + 1] = tfirst[T - S.T0] + (thi[T] - T + 1);
        auto at = [&](int64_t T) { return hroff[(size_t)(128 * (T - S.T0))]; };
        for (int64_t Ta = S.T0; Ta < S.T1;) {
            int64_t Tb = Ta + 1;
            while (Tb < S.T1 && at(Tb + 1) - at(Ta) <= pcap) ++Tb;
            Range R;
            R.a0 = trow0[Ta];
            R.a1 = trow0[Tb];
            R.n = at(Tb) - at(Ta);
            R.off.resize((size_t)(R.a1 - R.a0 + 1));
            for (int64_t i = R.a0; i < R.a1; ++i) R.off[i - R.a0] = hroff[(size_t)(prow[i] - S.R0)] - at(Ta);
            R.off.back() = R.n;
            R.on = true;
            if (R.n > 0) {
                R.x = (int)(n_ranges++ % 2);
                cudaEvent_t* e = ev.e + 2 + 3 * R.x;
                a.tiles = (const LdTile*)(dev + S.o_tiles) + tfirst[Ta - S.T0];
                a.n_tiles = (int32_t)(tfirst[Tb - S.T0] - tfirst[Ta - S.T0]);
                p.off = d_off;
                p.rowoff = d_roff;
                p.base = at(Ta);
                p.rid = (const int32_t*)(dev + S.o_rid);
                p.b = d_pb;
                p.r = d_pr;
                p.err = d_err;
                p.nmiss = d_nmiss;
                CU_TRY(h, cudaEventRecord(e[0], st));
                CU_TRY(h, launch_ld_pairs(tmap, a, p, true, h->n_sm, st));
                CU_TRY(h, cudaEventRecord(e[1], st));
                uint8_t* pin = (uint8_t*)h->ld_pin[R.x].p;
                CU_TRY(h, cudaMemcpyAsync(pin, d_pb, sizeof(int32_t) * (size_t)R.n, cudaMemcpyDeviceToHost, st));
                CU_TRY(h, cudaMemcpyAsync(pin + o_pr, d_pr, sizeof(double) * (size_t)R.n, cudaMemcpyDeviceToHost, st));
                CU_TRY(h, cudaMemcpyAsync(pin + o_flag, d_err, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
                CU_TRY(h, cudaEventRecord(e[2], st));
            }
            r = flush();                                // the previous range's sink runs while this one is emitted
            if (r != DBSLMM_B200_OK) return r;
            pend = std::move(R);
            Ta = Tb;
        }
        return DBSLMM_B200_OK;
    };
    rc = stream_chunks(h, (int64_t)segs.size(), max_bytes, n1, [&](int64_t k) { return segs[k].bytes; }, gather2, launch2);
    if (rc == DBSLMM_B200_OK) rc = flush();
    if (rc != DBSLMM_B200_OK) {
        cudaStreamSynchronize(st);                      // no copy may still be bound for the pinned buffers
        return rc;
    }
    unsigned long long nm = 0;
    CU_TRY(h, cudaMemcpyAsync(&nm, d_nmiss, sizeof(nm), cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaStreamSynchronize(st));
    n_miss = (int64_t)nm;
    if (n_pairs_out) *n_pairs_out = n_pairs;
    if (n_miss_pairs_out) *n_miss_pairs_out = n_miss;
    if (kernel_ms_out) *kernel_ms_out = ms;
    return DBSLMM_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// inspection hooks
// ---------------------------------------------------------------------------------------------
int dbslmm_b200_get_row_codes(dbslmm_b200_handle* h, int32_t block, int32_t j, int32_t plane, int8_t* codes_out, int32_t n_out) {
    if (!h || !codes_out) return DBSLMM_B200_ERR_ARG;
    if (!h->plan.valid) return fail(h, DBSLMM_B200_ERR_STATE, "no fit yet");
    if (block < 0 || block >= h->plan.n_blocks || n_out > h->n_pad || n_out < 0 || plane < 0 || plane > 1)
        return fail(h, DBSLMM_B200_ERR_ARG, "row out of range");
    const BlockDesc& bd = h->plan.blocks[block];
    if (j < 0 || j >= bd.m) return fail(h, DBSLMM_B200_ERR_ARG, "row out of range");
    const int64_t row = (int64_t)bd.croff + (plane ? bd.m : 0) + j;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaMemcpy(codes_out, (const int8_t*)h->codes.p + (size_t)row * h->n_pad, (size_t)n_out, cudaMemcpyDeviceToHost));
    return DBSLMM_B200_OK;
}

// The first mp + extra_rows rows (stride ld) of block `block`'s matrix in device buffer `dev` -> tmp.
static int fetch_block(dbslmm_b200_handle* h, int32_t block, const void* dev, size_t esz, std::vector<uint8_t>& tmp,
                       const BlockDesc** bd_out, int extra_rows = 0) {
    if (!h->plan.valid) return fail(h, DBSLMM_B200_ERR_STATE, "no fit yet");
    if (block < 0 || block >= h->plan.n_blocks) return fail(h, DBSLMM_B200_ERR_ARG, "block out of range");
    const BlockDesc& bd = h->plan.blocks[block];
    *bd_out = &bd;
    if (bd.m == 0) return DBSLMM_B200_OK;
    tmp.resize((size_t)(bd.mp + extra_rows) * bd.ld * esz);
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaMemcpy(tmp.data(), (const uint8_t*)dev + (size_t)bd.moff * esz, tmp.size(), cudaMemcpyDeviceToHost));
    return DBSLMM_B200_OK;
}

int dbslmm_b200_get_block_sigma(dbslmm_b200_handle* h, int32_t block, double* sigma_out) {
    if (!h || !sigma_out) return DBSLMM_B200_ERR_ARG;
    std::vector<uint8_t> tmp;
    const BlockDesc* bd = nullptr;
    int rc = fetch_block(h, block, h->sigma.p, sizeof(double), tmp, &bd);
    if (rc != DBSLMM_B200_OK) return rc;
    const double* s = (const double*)tmp.data();
    const bool full = (h->last_flags & DBSLMM_B200_FLAG_FULL_SIGMA) != 0;
    for (int i = 0; i < bd->m; ++i)
        for (int j = 0; j < bd->m; ++j) {
            const double v = (j <= i || full) ? s[(size_t)i * bd->ld + j] : s[(size_t)j * bd->ld + i];
            sigma_out[(size_t)i * bd->m + j] = v;
        }
    return DBSLMM_B200_OK;
}

int dbslmm_b200_get_block_factor(dbslmm_b200_handle* h, int32_t block, double* l_out, double* y_out) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (h->plan.valid && (h->last_solver != DBSLMM_B200_SOLVER_CHOLESKY || h->last_quad))
        return fail(h, DBSLMM_B200_ERR_STATE, "last fit did not factor (PCG solver or quadform)");
    std::vector<uint8_t> tmp;
    const BlockDesc* bd = nullptr;
    // rows 0..mp-1 hold L (lower triangle; W_kk^T in the upper triangles of the diagonal tiles), row mp holds y = L^-1 z
    int rc = fetch_block(h, block, h->lbuf.p, sizeof(double), tmp, &bd, 1);
    if (rc != DBSLMM_B200_OK) return rc;
    const double* s = (const double*)tmp.data();
    const int m = bd->m;
    if (l_out)
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) l_out[(size_t)i * m + j] = (j <= i) ? s[(size_t)i * bd->ld + j] : 0.0;
    if (y_out)
        for (int j = 0; j < m; ++j) y_out[j] = s[(size_t)bd->mp * bd->ld + j];
    return DBSLMM_B200_OK;
}

int dbslmm_b200_get_block_gram(dbslmm_b200_handle* h, int32_t block, int32_t* q_out, int32_t* a_out, int32_t* n_out) {
    if (!h || !q_out) return DBSLMM_B200_ERR_ARG;
    if (!(h->last_flags & DBSLMM_B200_FLAG_KEEP_INT_GRAM)) return fail(h, DBSLMM_B200_ERR_STATE, "last fit did not keep the integer Gram");
    std::vector<uint8_t> tmp;
    const BlockDesc* bd = nullptr;
    int rc = fetch_block(h, block, h->intQ.p, sizeof(int32_t), tmp, &bd);
    if (rc != DBSLMM_B200_OK) return rc;
    const int m = bd->m;
    auto copy_plane = [&](int32_t* out) {
        const int32_t* s = (const int32_t*)tmp.data();
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) out[(size_t)i * m + j] = s[(size_t)i * bd->ld + j];
    };
    copy_plane(q_out);
    if (h->miss_flags.size() > (size_t)block && h->miss_flags[block]) {
        if (a_out) { rc = fetch_block(h, block, h->intA.p, sizeof(int32_t), tmp, &bd); if (rc) return rc; copy_plane(a_out); }
        if (n_out) { rc = fetch_block(h, block, h->intN.p, sizeof(int32_t), tmp, &bd); if (rc) return rc; copy_plane(n_out); }
    } else {
        // no missing calls: A_ij = S_i, N_ij = n_ref (the fast path never forms them)
        std::vector<int32_t> S(std::max(m, 1));
        if (m) CU_TRY(h, cudaMemcpy(S.data(), (const int32_t*)h->rowS.p + bd->goff, sizeof(int32_t) * (size_t)m, cudaMemcpyDeviceToHost));
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) {
                if (a_out) a_out[(size_t)i * m + j] = S[i];
                if (n_out) n_out[(size_t)i * m + j] = h->n_ref;
            }
    }
    return DBSLMM_B200_OK;
}

int dbslmm_b200_get_block_iters(dbslmm_b200_handle* h, int32_t block) {
    if (!h) return DBSLMM_B200_ERR_ARG;
    if (!h->plan.valid || block < 0 || block >= h->plan.n_blocks) return fail(h, DBSLMM_B200_ERR_ARG, "block out of range");
    if (h->last_solver != DBSLMM_B200_SOLVER_PCG) return fail(h, DBSLMM_B200_ERR_STATE, "last fit was not a PCG fit");
    const int32_t* hs = (const int32_t*)((const uint8_t*)h->h_out.p +
                                         sizeof(double) * (size_t)(h->plan.tot_s + h->plan.tot_l) * (size_t)h->last_nfolds);
    return hs[h->plan.n_blocks + block];
}

}  // extern "C"
