// Stage 3: EM vanishing-point localisation as bulk-synchronous supersteps over
// the whole batch.
//
// Replaces vp_localisation.expectation_maximisation (reference
// vp_localisation.py:168-450) and everything it calls in
// probability_functions.py / coordinate_conversion.py.  Every image owns a slot
// (its VP state, <= 64 hypotheses, plus a workspace slice in HBM).  The
// per-image control flow of the reference is a state machine (em_core.cuh); the
// data-parallel work of all active images is spread over the whole GPU:
//
//   em_pair   : once per image, CTA = (image, 64-column slab).  All N^2 segment
//               pairs: similarity matrix lsim (E3, stored slab-major so that the
//               W kernel streams contiguous memory), its column sums, and the
//               kNN line rating (E4) from the same distances.
//   em_init   : once per image: unit lines, prior mixture, initial VPs (E0-E2).
//   superstep : em_estep (CTA = 64 lines of an image; E5) ->
//               em_wmat  (CTA = (image, slab): the (M x N)(N x N) weight-matrix
//                         product E6 on the FP64 tensor cores, lsim streamed by bulk
//                         async copies through a 4-stage shared-memory ring) ->
//               em_post  (CTA = image: reductions over the lines, 3x3
//                         eigen-solves, prune / split / merge / convergence
//                         decisions E7-E12, choice of the next superstep).
//   The superstep loop runs in one of three forms (plan_wave): the images of a wave dealt to groups, every
//   group driven by a device-side loop (CUDA graph of conditional WHILE nodes) on its own stream, so that
//   the latency-bound POST of one group overlaps the tensor/HBM-bound W of the others (default); the same
//   kernels launched by the host (profiling, VPK_EM_HOST_LOOP=1); or ONE persistent kernel with a cluster
//   per image that keeps the slot state in shared memory from the first E-step to the result (em_fused,
//   VPK_EM_MODE=fused).  All three produce bit-identical results.
//
// Arithmetic is float64 throughout: the reference is float64, its discrete
// decisions (counts < 3, argmax, err > 1.5, angle < thresh) sit on float values
// and the parity gate is 1e-4 rad on the refined VPs.
#include <algorithm>
#include <vector>
#include <chrono>
#include <cstdio>
#include <cstring>
#include "em_core.cuh"
#include "vpk_internal.cuh"

namespace vpk {

using namespace em;

static constexpr int kInitThreads = 512;
static constexpr int kPairThreads = 256;
static constexpr int kEThreads = 256;
static constexpr int kWThreads = 256;
static constexpr int kJR = 32;             // lsim rows per pipeline stage of the W kernel
static constexpr int kStages = 4;            // ring depth of the W kernel when the GPU is full (2 CTAs / SM)
static constexpr int kStagesTail = 8;        // ... when fewer CTAs than SMs are left: per-CTA streaming is latency bound
static constexpr int kChunkSteps = 4;      // supersteps enqueued between two host polls

struct SlotDesc {
    int32_t img, N, base, pad;
    unsigned long long ws_off;
};

struct EmParams {
    const double* lines;
    const double* segs;
    const float* resp32;
    const double* resp64;
    const uint8_t* sphere;
    int S;
    const double* init_vp;
    const int32_t* init_off;
    vpk_em_config cfg;
    EmSlot* slots;
    const SlotDesc* desc;
    double* ws;
    int* lists;            // 2 x n_slots: active slot ids of the current / next superstep, in slot order (heaviest image first)
    int* alive;            // n_slots flags: the slot takes part in the next superstep
    int* ctl;              // [0],[1]: list lengths; [3]: supersteps done (parity = current list);
                           // [4]: POST ticket counter; [5]: superstep limit hit
    int* ovlock;           // lock of the overflow scratch (shared by all groups of a wave)
    unsigned long long* stats;   // nullable (profiling): [0] algorithmic bytes, [1] flops of the W products, [2] slot-products,
                                 // [3] algorithmic bytes of POST, [4] of the E-step
    int n_slots;
    double* overflow;
    size_t overflow_cap;
    EmOut out;
};

// Loop control of the device-driven superstep loop (CUDA graph with conditional WHILE nodes, one per
// tier of grid sizes): after every superstep the last POST block sets each tier's condition to
// "more than thr[j] slots are still active".  n = 0: host-driven loop, nothing to set.
constexpr int kMaxTiers = 8;
struct TierCtl {
    int n, max_steps;
    int thr[kMaxTiers];
    cudaGraphConditionalHandle h[kMaxTiers];
};
constexpr int kCtlInts = 8;

// ---- PTX wrappers: mbarrier + 1-D bulk async copy (TMA engine, no tensor map) ----
__device__ __forceinline__ uint32_t em_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void em_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void em_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool em_mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps instead of hanging the GPU (the host then reports the failing launch by name,
// check_launch / KernelScope).  The bound is wall time on the device (20 s of %globaltimer once 2^24 polls have
// failed), not a poll count alone, so a time-sliced or preempted context is not mistaken for one.  No printf: the
// call costs the W kernel registers (measured 1.74 -> 1.765 ms per YUD batch).
__device__ __forceinline__ unsigned long long em_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void em_mbar_wait(uint32_t bar, uint32_t parity) {
    for (uint32_t i = 0; i < (1u << 24); ++i)
        if (em_mbar_try_wait(bar, parity)) return;
    // not reached in a run that is neither broken nor descheduled for long: now bound the wait by time
    const unsigned long long t0 = em_globaltimer();
    while (!em_mbar_try_wait(bar, parity))
        if (em_globaltimer() - t0 > 20000000000ull) __trap();
}
__device__ __forceinline__ void em_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// Stores of the per-superstep planes (lvsq, pvl, wt, w): kept in the L2 (evict-last) so that the next
// kernel of the superstep reads them there although the similarity matrices stream through in between.
__device__ __forceinline__ uint64_t em_policy_keep() {
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
    return policy;
}
__device__ __forceinline__ void em_st_keep(double* p, double v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(policy) : "memory");
}

__device__ __forceinline__ void copy_slot(EmSlot* dst, const EmSlot* src, const Team& T) {
    const int* s = reinterpret_cast<const int*>(src);
    int* d = reinterpret_cast<int*>(dst);
    for (int i = T.tid; i < (int)(sizeof(EmSlot) / sizeof(int)); i += T.nthreads) d[i] = s[i];
}

// ---------------------------------------------------------------------------
// em_pair: E3 (calc_lsim, vp_localisation.py:87-108) + E4 (line_rating_knn, :34-84)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kPairThreads) em_pair_kernel(EmParams P) {
    __shared__ double s_kd[kK1 * kPairThreads];
    __shared__ int s_kj[kK1 * kPairThreads];
    __shared__ int s_cnt[kPairThreads];
    __shared__ double s_part[kPairThreads];
    constexpr int JB = 128;
    __shared__ SegPre s_seg[JB];                     // per-segment constants of the current block of rows
    const SlotDesc d = P.desc[blockIdx.y];
    const int N = d.N, t = blockIdx.x;
    if (t * kTK >= N) return;
    const Img im = make_img(N, P.ws + d.ws_off, P.segs + 4 * (size_t)d.base);
    const int tid = threadIdx.x, col = tid & (kTK - 1), g = tid / kTK;
    constexpr int G = kPairThreads / kTK;
    const int k = t * kTK + col;
    const bool live = k < N;
    const SegPre sk = seg_pre(load_seg(im.lp, live ? k : 0));
    double* slab = im.lsim + (size_t)t * N * kTK;
    double part = 0.0;
    int cnt = 0;
    for (int jb = 0; jb < N; jb += JB) {
        __syncthreads();
        if (tid < JB && jb + tid < N) s_seg[tid] = seg_pre(load_seg(im.lp, jb + tid));
        __syncthreads();
        const int jn = min(JB, N - jb);
        // two rows per trip: the arithmetic of both pairs first (independent chains for the FP64 pipe), then the
        // candidate-list updates, stores and column sums in row order (the same order as one row per trip)
        for (int jj = g; jj < jn; jj += 2 * G) {
            const int ja = jb + jj, jc = ja + G;
            const bool two = jj + G < jn;
            double d2a = 16.0, vala = 0.0, d2c = 16.0, valc = 0.0;          // diagonal: ldist = 4 (:82), lsim = 0 (:105)
            if (live) {
                if (ja != k) { const SegPre& sj = s_seg[jj]; d2a = seg_distance2(sj, sk); vala = similarity_pre(sj, sk, d2a); }
                if (two && jc != k) { const SegPre& sj = s_seg[jj + G]; d2c = seg_distance2(sj, sk); valc = similarity_pre(sj, sk, d2c); }
                knn_insert(s_kd + tid, s_kj + tid, kPairThreads, cnt, d2a, ja);
            }
            slab[(size_t)ja * kTK + lsim_swz(ja, col)] = vala;
            part += vala;
            if (two) {
                if (live) knn_insert(s_kd + tid, s_kj + tid, kPairThreads, cnt, d2c, jc);
                slab[(size_t)jc * kTK + lsim_swz(jc, col)] = valc;
                part += valc;
            }
        }
    }
    s_cnt[tid] = cnt;
    s_part[tid] = part;
    __syncthreads();
    if (g == 0 && live) {
        double cs = 0.0;
        for (int q = 0; q < G; ++q) cs += s_part[q * kTK + col];
        im.colsum[k] = cs;
        // merge the G partial candidate lists (ascending (distance, index)) and rate the line
        double cd[kK1];
        int cj[kK1];
        int n = 0;
        for (int q = 0; q < G; ++q) {
            const int src = q * kTK + col;
            for (int e = 0; e < s_cnt[src]; ++e) knn_insert(cd, cj, 1, n, s_kd[e * kPairThreads + src], s_kj[e * kPairThreads + src]);
        }
        im.lweight[k] = rate_line(im.lp, k, cj, cd, n, N);
    }
}

// Closing of a kernel with one CTA per slot: every CTA has written alive[slot]; the last one to
// arrive compacts the flags into list `next` IN SLOT ORDER (slots are sorted heaviest image first, so the
// CTAs of the big images of the next E / W launches start first) and returns the number of active slots
// to its thread 0 (-1 in every other CTA).  Block-wide; thread 0 of the last CTA resets the ticket.
__device__ int close_slot_list(const EmParams& P, int next, const Team& T, int participants = -1) {
    __shared__ int s_last, s_warp[32], s_base;
    if (participants < 0) participants = (int)gridDim.x;
    __syncthreads();
    if (T.tid == 0) {
        __threadfence();
        s_last = atomicAdd(P.ctl + 4, 1) == participants - 1;
        s_base = 0;
    }
    __syncthreads();
    if (!s_last) return -1;
    __threadfence();
    int* list = P.lists + next * P.n_slots;
    for (int c0 = 0; c0 < P.n_slots; c0 += T.nthreads) {
        const int i = c0 + T.tid;
        const bool f = i < P.n_slots && *reinterpret_cast<volatile int*>(P.alive + i) != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        if (T.lane == 0) s_warp[T.warp] = __popc(bal);
        __syncthreads();
        int off = s_base, tot = 0;
        for (int w = 0; w < T.nwarps; ++w) { if (w < T.warp) off += s_warp[w]; tot += s_warp[w]; }
        if (f) list[off + __popc(bal & ((1u << T.lane) - 1u))] = i;
        __syncthreads();
        if (T.tid == 0) s_base += tot;
        __syncthreads();
    }
    const int live = s_base;
    if (T.tid == 0) { P.ctl[4] = 0; P.ctl[next] = live; }
    return T.tid == 0 ? live : -1;
}

// ---------------------------------------------------------------------------
// em_init: per-line constants, prior mixture, initial VPs, first E-step request
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kInitThreads) em_init_kernel(EmParams P) {
    __shared__ __align__(16) EmSlot st;
    __shared__ InitScratch isc;
    const Team T = make_team();
    const int slot = blockIdx.x;
    const SlotDesc d = P.desc[slot];
    const int N = d.N, b = d.img;
    for (int i = T.tid; i < (int)(sizeof(EmSlot) / sizeof(int)); i += T.nthreads) reinterpret_cast<int*>(&st)[i] = 0;
    __syncthreads();
    if (T.tid == 0) { st.img = b; st.N = N; st.base = d.base; st.ws_off = d.ws_off; st.phase = PH_DONE; }
    const Img im = make_img(N, P.ws + d.ws_off, P.segs + 4 * (size_t)d.base);
    line_constants(im, P.lines + 3 * (size_t)d.base, T);
    if (!P.cfg.use_weights)
        for (int n = T.tid; n < N; n += T.nthreads) { im.lweight[n] = 1.0; im.colsum[n] = 0.0; }
    for (int c = T.tid; c < kCells; c += T.nthreads)
        isc.resp[c] = P.resp64 ? P.resp64[(size_t)b * kCells + c] : (double)P.resp32[(size_t)b * kCells + c];
    __syncthreads();
    const double* iv = nullptr;
    int n_init = 0;
    if (P.init_vp) { iv = P.init_vp + 3 * (size_t)P.init_off[b]; n_init = P.init_off[b + 1] - P.init_off[b]; }
    const uint8_t* sph = P.sphere ? P.sphere + (size_t)b * P.S * P.S : nullptr;
    const bool active = init_slot(st, isc, im, P.out, P.cfg, sph, P.S, iv, n_init, T);
    __syncthreads();
    copy_slot(P.slots + slot, &st, T);
    if (T.tid == 0) P.alive[slot] = active ? 1 : 0;
    close_slot_list(P, 0, T);
}

// ---------------------------------------------------------------------------
// em_estep: E5 for 32 lines of one active slot.  lane = line, warp w = VP rows
// w, w+8, ...; the per-line normaliser p(l) is the sum of the 8 warp partials in
// warp order; the W operand tile is staged in shared memory and written with
// contiguous stores.
// ---------------------------------------------------------------------------
constexpr int kEL = 64;                      // lines per E-step tile
struct ESmem {
    double c_pv[kMaxM], c_vx[kMaxM], c_vy[kMaxM], c_inv2s[kMaxM], c_coef[kMaxM];
    double s_pl[8][kEL];
    double s_wt[kMaxM / kMP][kEL][kMP + 1];      // +1: conflict-free column writes (rows of a pass: 8 * tiles <= kMP)
};

// the constants of the E-step on the slot's selected VP set (prepare_estep) -> shared memory
__device__ __forceinline__ void estep_load_constants(ESmem& es, const EmSlot& st) {
    for (int m = threadIdx.x; m < st.M; m += blockDim.x) {
        es.c_pv[m] = st.pv[m]; es.c_vx[m] = st.vx[m]; es.c_vy[m] = st.vy[m]; es.c_inv2s[m] = st.inv2s[m]; es.c_coef[m] = st.coef[m];
    }
}

// E5 for lines n0 .. n0+63 of one image (block-wide, kEThreads = 256 threads; es.c_* loaded and synchronised).
// Thread (line = tid & 63, q = tid >> 6) evaluates the VP rows m = q, q + 4, q + 8, ...; the per-line normaliser
// p(l) is the sum of eight partials -- rows m = r (mod 8), r = 0 .. 7, in that order -- whatever the tiling.
__device__ __forceinline__ void estep_tile(ESmem& es, const Img& im, int N, int M, int n0, uint64_t keep) {
    constexpr int NQ = kEThreads / kEL, kMI = kMaxM / NQ;      // 4 row classes per line, 16 rows per thread
    const int tid = threadIdx.x, q = tid / kEL, ln = tid % kEL;
    const int n = n0 + ln;
    const bool live = n < N;
    const LineGeom g = line_geom(im.lp, live ? n : 0);
    double plv[kMI];
    double part[2] = {0.0, 0.0};                               // rows m = q (mod 8) and m = q + 4 (mod 8)
#pragma unroll
    for (int mi = 0; mi < kMI; ++mi) {
        const int m = q + NQ * mi;
        plv[mi] = 0.0;
        if (m < M) {
            double lvsq;
            estep_nm(g, es.c_vx[m], es.c_vy[m], es.c_inv2s[m], es.c_coef[m], lvsq, plv[mi]);
            if (live) em_st_keep(im.lvsq + (size_t)m * N + n, lvsq, keep);
            part[mi & 1] += plv[mi] * es.c_pv[m];
        }
    }
    es.s_pl[q][ln] = part[0];
    es.s_pl[q + NQ][ln] = part[1];
    __syncthreads();
    double pl = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) pl += es.s_pl[w][ln];
    if (pl < 1e-12) pl = 1e-12;                                         // :117 (NaN stays NaN)
    const double inv_pl = 1.0 / pl;
    const double lw = live ? im.lweight[n] : 0.0;
    const int passes = (M + kMP - 1) / kMP;
#pragma unroll
    for (int mi = 0; mi < kMI; ++mi) {
        const int m = q + NQ * mi, p = m / kMP, mm = m % kMP;
        if (p < passes && mm < 8 * wpass_tiles(M, p)) {
            double x = 0.0;
            if (m < M) {
                x = plv[mi] * es.c_pv[m] * inv_pl;                      // calc_pvl (:128)
                if (live) em_st_keep(im.pvl + (size_t)m * N + n, x, keep);
                x *= lw;                                                // weight_matrix :517
            }
            es.s_wt[p][ln][mm] = x;
        }
    }
    __syncthreads();
    const int nl = min(kEL, N - n0);
    for (int p = 0; p < passes; ++p) {
        const int ws = wpass_stride(M, p), rows = ws - 4;                  // the 4 padding doubles of a line are never read
        double* dst = im.wt + (size_t)p * N * kMPS + (size_t)n0 * ws;
        for (int e = tid; e < nl * rows; e += kEThreads) em_st_keep(dst + (size_t)(e / rows) * ws + (e % rows), es.s_wt[p][e / rows][e % rows], keep);
    }
}

__global__ void __launch_bounds__(kEThreads) em_estep_kernel(EmParams P) {
    __shared__ ESmem es;
    const int cur = P.ctl[3] & 1;
    if ((int)blockIdx.y >= P.ctl[cur]) return;
    const int slot = P.lists[cur * P.n_slots + blockIdx.y];
    const EmSlot& st = P.slots[slot];
    if (!st.run_e) return;
    const int N = st.N, M = st.M, n0 = blockIdx.x * kEL;
    if (n0 >= N) return;
    // algorithmic bytes of this slot's E-step: segments + line weights in, the planes lvsq, pvl, wt out
    if (P.stats && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(P.stats + 4, 8ull * (5ull * N + 3ull * M * N));
    estep_load_constants(es, st);
    __syncthreads();
    const Img im = make_img(N, P.ws + st.ws_off, P.segs + 4 * (size_t)st.base);
    estep_tile(es, im, N, M, n0, em_policy_keep());
}

// ---------------------------------------------------------------------------
// em_wmat: E6, w[m,k] = (wt[k,m] + b lw[k] sum_j wt[j,m] lsim[j,k]) / (1 + b lw[k] colsum[k])
// (vp_localisation.py:515-524).
//
// A cluster of CS CTAs owns (slot, 64-column slab); CTA rank r of the cluster
// streams the rows of chunk range r of the slab (N x 64 doubles, contiguous) and
// the matching rows of wt through a 4-stage ring of shared-memory buffers filled
// by cp.async.bulk (full/empty mbarriers, no CTA-wide barrier in the loop: warp
// 0 re-arms a stage as soon as all 8 warps have released it).  Lane l of a warp
// accumulates columns 2l, 2l+1; a pass covers up to 32 VP rows as G groups of
// warps x R rows per thread.  Partial sums are combined in a fixed order: the
// warps of a CTA through shared memory, then the CTAs of the cluster in rank
// order through distributed shared memory.  CS depends on N only, so an image's
// result does not depend on what else is in the batch.
// ---------------------------------------------------------------------------
template <int STAGES>
struct WSmemT {
    double a[STAGES][kJR * kTK];           // lsim rows
    double b[STAGES][kJR * kMPS];          // wt rows; b[0..1] reused for the per-CTA partial result (kMP x kTK)
    unsigned long long full[STAGES], empty[STAGES];
};

// CTAs per slab: only very tall slabs are split (the cluster barriers cost ~20 % of a short CTA's time)
__host__ __device__ inline int wmat_split(int N) { return N <= 1536 ? 1 : (N <= 3072 ? 2 : 4); }

// Threads per arrival on a ring stage's "empty" barrier.  Every thread releases the stage itself after its own fragment
// reads.  One arrival per warp (lane 0 after __syncwarp()) is equally ordered and measured equally fast, but
// compute-sanitizer's racecheck does not follow that delegation and reports the refill of a stage against the other
// lanes' reads; with one arrival per thread it reports no hazard (profiles/r2_sanitize_summary.txt).
constexpr int kArriveGroup = 1;
__device__ __forceinline__ void em_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void em_bulk_g2s_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ uint32_t em_cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void em_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ double em_ld_dsmem(const double* local, uint32_t rank) {
    uint32_t addr = em_smem_u32(local), remote;
    double v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(addr), "r"(rank));
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(remote) : "memory");
    return v;
}

// D (8 x 8) += A (8 x 4, row) * B (4 x 8, col) on the FP64 tensor-core path.  Lane l = 4 g + t holds A[g][t], B[t][g]
// and D[g][2t], D[g][2t + 1].
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// main loop of one pass of MT 8-row tiles of VP rows: chunks [c0, c1) of the slab.  The (8 MT x 32)(32 x 64) product
// of a chunk runs on the FP64 tensor cores: warp w takes the 16 columns 16 (w & 3) .. and the row half (w >> 2) of the
// chunk, i.e. 4 k-steps x MT x 2 instructions.  The fragments are read straight from the bulk-copied rows (both
// layouts are bank-conflict free, see lsim_swz / wpass_stride).  The two row halves are added (first + second) at the
// end; the result lands in part[row * 64 + column].
template <int MT, int kStages>
__device__ __forceinline__ void wmat_pass(WSmemT<kStages>& sm, const double* slab, const double* wtp, int ws, int N, int c0, int c1,
                                          int& ring, uint64_t policy, bool keep, double* red, double* part) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3, wn = warp & 3, wk = warp >> 2;
    double acc[MT][2][2];
#pragma unroll
    for (int m = 0; m < MT; ++m) acc[m][0][0] = acc[m][0][1] = acc[m][1][0] = acc[m][1][1] = 0.0;
    const int nch = c1 - c0;
    int next_issue = 0;                              // warp 0 only
    auto issue = [&](int i) {                        // chunk c0 + i into ring slot (ring + i) % kStages
        const int j0 = (c0 + i) * kJR, jn = min(kJR, N - j0), s = (ring + i) % kStages;
        const uint32_t bar = em_smem_u32(&sm.full[s]);
        em_mbar_expect_tx(bar, (uint32_t)(jn * (kTK + ws) * sizeof(double)));
        if (keep) em_bulk_g2s(em_smem_u32(sm.a[s]), slab + (size_t)j0 * kTK, (uint32_t)(jn * kTK * sizeof(double)), bar);
        else em_bulk_g2s_hint(em_smem_u32(sm.a[s]), slab + (size_t)j0 * kTK, (uint32_t)(jn * kTK * sizeof(double)), bar, policy);
        em_bulk_g2s(em_smem_u32(sm.b[s]), wtp + (size_t)j0 * ws, (uint32_t)(jn * ws * sizeof(double)), bar);
    };
    const int colb0 = (16 * wn + g) ^ (t << 2), colb1 = (16 * wn + 8 + g) ^ (t << 2);
    for (int i = 0; i < nch; ++i) {
        const int pos = ring + i, s = pos % kStages;
        if (warp == 0) {
            // keep the ring full: chunk q may be issued once ring position (ring + q - kStages) was released
            while (next_issue < nch && next_issue < i + kStages) {
                const int q = ring + next_issue;
                if (q >= kStages) {
                    const uint32_t eb = em_smem_u32(&sm.empty[q % kStages]);
                    const uint32_t par = (uint32_t)(((q / kStages) - 1) & 1);
                    if (next_issue == i) em_mbar_wait(eb, par);
                    else if (!em_mbar_try_wait(eb, par)) break;
                }
                if (lane == 0) issue(next_issue);
                ++next_issue;
            }
            __syncwarp();
        }
        em_mbar_wait(em_smem_u32(&sm.full[s]), (uint32_t)((pos / kStages) & 1));
        const int jn = min(kJR, N - (c0 + i) * kJR);
        const double* Bs = sm.a[s];
        const double* As = sm.b[s];
        if (jn == kJR) {
#pragma unroll
            for (int ks = 0; ks < kJR / 8; ++ks) {
                const int j = (kJR / 2) * wk + 4 * ks + t;
                const double b0 = Bs[j * kTK + colb0], b1 = Bs[j * kTK + colb1];
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const double a = As[j * ws + 8 * m + g];
                    dmma884(acc[m][0][0], acc[m][0][1], a, b0);
                    dmma884(acc[m][1][0], acc[m][1][1], a, b1);
                }
            }
        } else {
            // last chunk of the image: rows >= jn are stale shared memory and must not contribute
#pragma unroll
            for (int ks = 0; ks < kJR / 8; ++ks) {
                const int j = (kJR / 2) * wk + 4 * ks + t;
                const bool ok = j < jn;
                const double b0 = ok ? Bs[j * kTK + colb0] : 0.0, b1 = ok ? Bs[j * kTK + colb1] : 0.0;
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const double a = ok ? As[j * ws + 8 * m + g] : 0.0;
                    dmma884(acc[m][0][0], acc[m][0][1], a, b0);
                    dmma884(acc[m][1][0], acc[m][1][1], a, b1);
                }
            }
        }
        em_mbar_arrive(em_smem_u32(&sm.empty[s]));      // this thread is done with stage s (see kArriveGroup)
    }
    ring += nch;
    __syncthreads();                                 // every warp has finished reading the ring
    // the two row halves of the chunks, in the (now idle) ring: first half -> part, second half -> red
    double* dst = wk ? red : part;
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int n = 0; n < 2; ++n)
            *reinterpret_cast<double2*>(&dst[(8 * m + g) * kTK + 16 * wn + 8 * n + 2 * t]) = make_double2(acc[m][n][0], acc[m][n][1]);
    __syncthreads();
    for (int e = tid; e < 8 * MT * kTK; e += kWThreads) part[e] = part[e] + red[e];
}

// keep: the similarity matrices of the slots still active fit the L2, so they are loaded with the
// default policy and stay resident from one superstep to the next (evict-first otherwise).
template <int kStages>
__global__ void __launch_bounds__(kWThreads, 2) em_wmat_kernel(EmParams P, int csl, int keep, int want_split) {
    extern __shared__ __align__(128) unsigned char w_smem_raw[];
    WSmemT<kStages>& sm = *reinterpret_cast<WSmemT<kStages>*>(w_smem_raw);
    const int cur = P.ctl[3] & 1;
    if ((int)blockIdx.y >= P.ctl[cur]) return;
    const int slot = P.lists[cur * P.n_slots + blockIdx.y];
    const EmSlot& st = P.slots[slot];
    if (!st.run_w) return;
    const int N = st.N, M = st.M, t = blockIdx.x / csl;
    if (t * kTK >= N) return;                       // uniform over the cluster
    // Tall slabs (N > 1536) are shared by the CTAs of a cluster, all others take one CTA: two launches per superstep,
    // each skipping the other's slots, so that no idle cluster rank holds shared memory next to a short slab.
    if ((wmat_split(N) > 1) != (want_split != 0)) return;
    const int rank = csl > 1 ? (int)em_cluster_ctarank() : 0;
    const int cs = min(wmat_split(N), csl);         // CTAs of the cluster that share this slab
    const Img im = make_img(N, P.ws + st.ws_off, P.segs + 4 * (size_t)st.base);
    const int tid = threadIdx.x;
    const bool stream = P.cfg.use_weights != 0;
    const double bias = P.cfg.wbias;
    if (P.stats && blockIdx.x == 0 && tid == 0) {
        // algorithmic work of this slot's product: the N x N similarity matrix once, 2 M N^2 flops
        atomicAdd(P.stats + 0, (unsigned long long)N * N * sizeof(double));
        atomicAdd(P.stats + 1, 2ull * M * N * N);
        atomicAdd(P.stats + 2, 1ull);
    }
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) {
            em_mbar_init(em_smem_u32(&sm.full[s]), 1);
            em_mbar_init(em_smem_u32(&sm.empty[s]), kWThreads / kArriveGroup);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    const uint64_t keep_policy = em_policy_keep();
    const int nchunks = (N + kJR - 1) / kJR;
    const int passes = (M + kMP - 1) / kMP;
    const double* slab = im.lsim + (size_t)t * N * kTK;
    double* red = &sm.a[0][0];
    double* part = &sm.b[0][0];
    // chunk range of this CTA
    int c0 = 0, c1 = 0;
    if (stream && rank < cs) { c0 = (int)((long long)nchunks * rank / cs); c1 = (int)((long long)nchunks * (rank + 1) / cs); }
    int ring = 0;                                   // ring position, carries over passes
    for (int pass = 0; pass < passes; ++pass) {
        const int mt = wpass_tiles(M, pass), ws = 8 * mt + 4;
        const double* wtp = im.wt + (size_t)pass * N * kMPS;
        switch (mt) {
        case 1: wmat_pass<1, kStages>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep != 0, red, part); break;
        case 2: wmat_pass<2, kStages>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep != 0, red, part); break;
        case 3: wmat_pass<3, kStages>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep != 0, red, part); break;
        default: wmat_pass<4, kStages>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep != 0, red, part); break;
        }
        if (csl > 1) em_cluster_sync(); else __syncthreads();          // partial results are complete
        if (rank == 0) {
            for (int e = tid; e < 8 * mt * kTK; e += kWThreads) {
                const int mm = e / kTK, col = e % kTK, k = t * kTK + col, m = pass * kMP + mm;
                if (k < N && m < M) {
                    double sum = part[e];
                    for (int r = 1; r < cs; ++r) sum += em_ld_dsmem(part + e, (uint32_t)r);
                    em_st_keep(im.w + (size_t)m * N + k,
                               wmat_finish(im.wt[(size_t)pass * N * kMPS + (size_t)k * ws + mm], im.lweight[k], im.colsum[k], sum, bias),
                               keep_policy);
                }
            }
        }
        // the ring (generic-proxy writes of red / part) is refilled by the async proxy in the next pass;
        // remote CTAs must not leave (or overwrite part) while rank 0 still reads their shared memory
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (csl > 1) em_cluster_sync(); else __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// em_post: one CTA per active slot
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kPostThreads, 2) em_post_kernel(EmParams P, TierCtl tc) {
    __shared__ __align__(16) EmSlot st;
    __shared__ PostScratch sc;
    const int step = P.ctl[3], cur = step & 1;
    const Team T = make_team();
#if defined(VPK_EM_MARKS)
    if (T.tid == 0) { for (auto& m : sc.mark) m = 0; sc.mark_t = clock64(); }
#endif
    if ((int)blockIdx.x < P.ctl[cur]) {
        const int slot = P.lists[cur * P.n_slots + blockIdx.x];
        copy_slot(&st, P.slots + slot, T);
        __syncthreads();
        // algorithmic bytes of this slot's POST: the planes w, lvsq, pvl and the unit lines + weights once
        if (P.stats && T.tid == 0) atomicAdd(P.stats + 3, 8ull * (3ull * st.M * st.N + 5ull * st.N));
        const Img im = make_img(st.N, P.ws + st.ws_off, P.segs + 4 * (size_t)st.base);
        post_slot(st, sc, im, P.out, P.cfg, P.overflow, P.overflow_cap, P.ovlock, T);
        __syncthreads();
        VPK_MARK(sc, T, 6);
        copy_slot(P.slots + slot, &st, T);
        if (T.tid == 0) P.alive[slot] = st.done ? 0 : 1;
        __syncthreads();
        VPK_MARK(sc, T, 7);
#if defined(VPK_EM_MARKS)
        if (P.stats && T.tid == 0) {
            for (int k = 0; k < 10; ++k) atomicAdd(P.stats + 8 + k, (unsigned long long)sc.mark[k]);
            atomicAdd(P.stats + 18, 1ull);
            if (sc.mark[15] > 0) {                              // split_best_vp ran to its end: marks 11..15 of the split
                for (int k = 11; k < 16; ++k) atomicAdd(P.stats + 8 + k, (unsigned long long)sc.mark[k]);
                atomicAdd(P.stats + 24, 1ull);
                unsigned long long tot = 0;
                for (int k = 11; k < 16; ++k) tot += (unsigned long long)sc.mark[k];
                if (atomicMax(P.stats + 25, tot) < tot) {        // phases of the slowest split (diagnostic; not race-free)
                    for (int k = 11; k < 16; ++k) P.stats[15 + k] = (unsigned long long)sc.mark[k];
                    P.stats[31] = (unsigned long long)st.N;
                }
            }
        }
#endif
    }
    // the last block to finish closes the superstep: the other list becomes current, this one is emptied
    const int live = close_slot_list(P, cur ^ 1, T);
    if (live >= 0) {
        P.ctl[cur] = 0;
        P.ctl[3] = step + 1;
        const bool stop = step + 1 >= tc.max_steps;
        if (stop && live > 0) P.ctl[5] = 1;
        for (int j = 0; j < tc.n; ++j) cudaGraphSetConditional(tc.h[j], (!stop && live > tc.thr[j]) ? 1u : 0u);
    }
}

// ---------------------------------------------------------------------------
// em_fused: the whole superstep loop of an image inside ONE persistent kernel.
//
// A thread-block cluster owns an image from its first E-step to its result: the
// slot state lives in the shared memory of the cluster's CTA 0 (the other CTAs
// mirror the few words they need through distributed shared memory), and the
// three phases of a superstep are separated by cluster barriers instead of
// kernel boundaries:
//     E     : CTA r takes the 32-line tiles r, r + C, ...
//     W     : CTA r takes the 64-column slabs r, r + C, ... (the same bulk-copy ring,
//             the same chunk ranges and summation order as em_wmat: bit-identical w)
//     POST  : CTA 0 runs the state machine (post_slot); the sums of the M-step,
//             one warp per hypothesis, are spread over the warps of ALL CTAs first
//     (E + W + POST of one image never wait for another image)
// Clusters pull images from a queue (heaviest first) until it is empty, two CTAs
// per SM, so the POST of one image overlaps the W of the image that shares its SMs,
// and the similarity matrices of the ~40-70 images in flight stay in the L2.
// ---------------------------------------------------------------------------
constexpr int kFThreads = 256;
static_assert(kFThreads == kEThreads && kFThreads == kWThreads, "the fused kernel runs E, W and POST with one block size");

struct FusedSmem {
    union U {
        WSmemT<kStages> w;       // ring + its mbarriers (the barriers lie beyond the other two members)
        PostScratch sc;
        ESmem es;
    } u;
    __align__(16) EmSlot st;
    RefitAcc tmp[kFThreads / 32];    // per-warp staging of the M-step sums before they are shipped to CTA 0
    int idx, flag;
    long long mark[8];
};
static_assert(sizeof(PostScratch) <= offsetof(WSmemT<kStages>, full), "POST scratch must not reach the ring's barriers");
static_assert(sizeof(ESmem) <= offsetof(WSmemT<kStages>, full), "E scratch must not reach the ring's barriers");
static_assert(sizeof(FusedSmem) <= 113 * 1024, "two CTAs per SM");

__device__ __forceinline__ uint32_t em_cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t em_ld_dsmem_u32(const void* local, uint32_t rank) {
    uint32_t addr = em_smem_u32(local), remote, v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(addr), "r"(rank));
    asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(remote) : "memory");
    return v;
}
__device__ __forceinline__ void em_st_dsmem_f64(double* local, uint32_t rank, double v) {
    uint32_t addr = em_smem_u32(local), remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(addr), "r"(rank));
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(remote), "d"(v) : "memory");
}
__device__ __forceinline__ void em_st_dsmem_u32(void* local, uint32_t rank, uint32_t v) {
    uint32_t addr = em_smem_u32(local), remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(addr), "r"(rank));
    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(remote), "r"(v) : "memory");
}

// E6 for slab t of one image by ONE CTA: the chunk ranges a cluster of em_wmat CTAs would share are run one
// after the other and their partial sums added in the same (rank) order, so w is bit-identical to em_wmat's.
template <int kSt>
__device__ void wmat_slab(WSmemT<kSt>& sm, const Img& im, int N, int M, int t, int& ring, uint64_t policy, bool keep,
                          uint64_t keep_policy, double bias, bool stream) {
    const int tid = threadIdx.x;
    const int nchunks = (N + kJR - 1) / kJR, passes = (M + kMP - 1) / kMP, cs = wmat_split(N);
    const double* slab = im.lsim + (size_t)t * N * kTK;
    double* red = &sm.a[0][0];
    double* part = &sm.b[0][0];
    for (int pass = 0; pass < passes; ++pass) {
        const int mt = wpass_tiles(M, pass), ws = 8 * mt + 4;
        const double* wtp = im.wt + (size_t)pass * N * kMPS;
        for (int r = 0; r < cs; ++r) {
            int c0 = 0, c1 = 0;
            if (stream) { c0 = (int)((long long)nchunks * r / cs); c1 = (int)((long long)nchunks * (r + 1) / cs); }
            switch (mt) {
            case 1: wmat_pass<1, kSt>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep, red, part); break;
            case 2: wmat_pass<2, kSt>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep, red, part); break;
            case 3: wmat_pass<3, kSt>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep, red, part); break;
            default: wmat_pass<4, kSt>(sm, slab, wtp, ws, N, c0, c1, ring, policy, keep, red, part); break;
            }
            __syncthreads();                                         // the partial sums of this range are complete
            for (int e = tid; e < 8 * mt * kTK; e += kFThreads) {
                const int mm = e / kTK, col = e % kTK, k = t * kTK + col, m = pass * kMP + mm;
                if (k < N && m < M) {
                    double* dst = im.w + (size_t)m * N + k;
                    // running sum of the ranges parked in the output element itself (this thread owns it)
                    const double sum = r == 0 ? part[e] : *dst + part[e];
                    if (r + 1 < cs) *dst = sum;
                    else em_st_keep(dst, wmat_finish(im.wt[(size_t)pass * N * kMPS + (size_t)k * ws + mm], im.lweight[k], im.colsum[k], sum, bias),
                                    keep_policy);
                }
            }
            // the ring (generic-proxy writes of red / part) is refilled by the async proxy next
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
        }
    }
}

// M-step sums (refit_sums) of hypothesis rows spread over the warps of the whole cluster; results land in the
// RefitAcc array of CTA 0 (distributed shared memory).  Only for the plain M-step phase.
__device__ void cluster_presum(RefitAcc* acc0, RefitAcc* s_tmp, const Img& im, int N, int M, uint32_t rank, uint32_t C, const Team& T) {
    // acc0: the RefitAcc array of the POST scratch (same shared-memory offset in every CTA of the cluster)
    const int gw = (int)rank * T.nwarps + T.warp, tw = (int)C * T.nwarps;
    for (int m = gw; m < M; m += tw) {
        refit_sums(im, im.w + (size_t)m * N, nullptr, -1, m, -1, s_tmp[T.warp], T);
        __syncwarp();
        // ship the accumulator to CTA 0, 4 bytes per lane and round
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&s_tmp[T.warp]);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&acc0[m]);
        for (int i = T.lane; i < (int)(sizeof(RefitAcc) / 4); i += 32) em_st_dsmem_u32(dst + i, 0, src[i]);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kFThreads, 2) em_fused_kernel(EmParams P, int max_steps, int keep) {
    extern __shared__ __align__(128) unsigned char f_smem_raw[];
    FusedSmem& S = *reinterpret_cast<FusedSmem*>(f_smem_raw);
    const Team T = make_team();
    const int tid = T.tid;
    const uint32_t rank = em_cluster_ctarank(), C = em_cluster_nctarank();
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) {
            em_mbar_init(em_smem_u32(&S.u.w.full[s]), 1);
            em_mbar_init(em_smem_u32(&S.u.w.empty[s]), kFThreads / kArriveGroup);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (auto& m : S.mark) m = 0;
    }
    __syncthreads();
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    const uint64_t keep_policy = em_policy_keep();
    const bool stream = P.cfg.use_weights != 0;
    const double bias = P.cfg.wbias;
    int ring = 0;                                    // position in the bulk-copy ring, carried over slabs, supersteps and images
    long long t_mark = 0;
    auto mark = [&](int k) {                          // cycles of CTA 0 per phase (profiling runs)
        if (P.stats && rank == 0 && tid == 0) { const long long c = clock64(); S.mark[k] += c - t_mark; t_mark = c; }
    };
    for (;;) {
        if (rank == 0 && tid == 0) S.idx = atomicAdd(P.ctl + 6, 1);
        em_cluster_sync();
        const int slot = (int)em_ld_dsmem_u32(&S.idx, 0);
        em_cluster_sync();                           // CTA 0 may overwrite idx only after every CTA has read it
        if (slot >= P.n_slots) break;
        copy_slot(&S.st, P.slots + slot, T);         // every CTA: the state em_init left in HBM
        __syncthreads();
        const int N = S.st.N;
        const Img im = make_img(N, P.ws + S.st.ws_off, P.segs + 4 * (size_t)S.st.base);
        const int ntile = (N + kEL - 1) / kEL, tiles = (N + kTK - 1) / kTK;
        int steps = 0;
        if (P.stats && rank == 0 && tid == 0) t_mark = clock64();
        while (!S.st.done) {                         // identical in every CTA of the cluster
            const int M = S.st.M;
            // ---- E ----------------------------------------------------------------------------
            estep_load_constants(S.u.es, S.st);
            __syncthreads();
            for (int b = (int)rank; b < ntile; b += (int)C) estep_tile(S.u.es, im, N, M, b * kEL, keep_policy);
            // wt is read through the async proxy (bulk copies) by the other CTAs
            asm volatile("fence.proxy.async;" ::: "memory");
            mark(0);
            em_cluster_sync();
            mark(1);
            // ---- W ----------------------------------------------------------------------------
            asm volatile("fence.proxy.async;" ::: "memory");
            for (int t = (int)rank; t < tiles; t += (int)C)
                wmat_slab<kStages>(S.u.w, im, N, M, t, ring, policy, keep != 0, keep_policy, bias, stream);
            mark(2);
            em_cluster_sync();
            mark(3);
            // ---- POST -------------------------------------------------------------------------
            const bool presum = S.st.phase == PH_MSTEP && P.cfg.do_iterations && C > 1;
            if (presum) {
                cluster_presum(refit_acc(S.u.sc), S.tmp, im, N, M, rank, C, T);
                em_cluster_sync();
            }
            mark(4);
            if (rank == 0) {
                if (P.stats && tid == 0) {
                    atomicAdd(P.stats + 0, (unsigned long long)N * N * sizeof(double));
                    atomicAdd(P.stats + 1, 2ull * M * N * N);
                    atomicAdd(P.stats + 2, 1ull);
                    atomicAdd(P.stats + 3, 8ull * (3ull * M * N + 5ull * N));
                    atomicAdd(P.stats + 4, 8ull * (5ull * N + 3ull * M * N));
                }
#if defined(VPK_EM_MARKS)
                if (tid == 0) { for (auto& m : S.u.sc.mark) m = 0; S.u.sc.mark_t = clock64(); }
#endif
                post_slot(S.st, S.u.sc, im, P.out, P.cfg, P.overflow, P.overflow_cap, P.ovlock, T, presum);
                __syncthreads();
#if defined(VPK_EM_MARKS)
                if (P.stats && tid == 0) {
                    for (int k = 0; k < 10; ++k) atomicAdd(P.stats + 16 + k, (unsigned long long)S.u.sc.mark[k]);
                    atomicAdd(P.stats + 26, 1ull);
                }
#endif
                ++steps;
                if (tid == 0 && steps >= max_steps && !S.st.done) { P.ctl[5] = 1; S.st.done = 1; }     // runaway guard
            }
            mark(5);
            em_cluster_sync();
            if (rank != 0) {
                // mirror what E and W need: the header and the E-step constants
                constexpr int kHead = (int)(offsetof(EmSlot, cur) / 4);
                constexpr int kC0 = (int)(offsetof(EmSlot, pv) / 4), kC1 = (int)(offsetof(EmSlot, cw) / 4);
                uint32_t* d = reinterpret_cast<uint32_t*>(&S.st);
                for (int i = tid; i < kHead; i += kFThreads) d[i] = em_ld_dsmem_u32(d + i, 0);
                for (int i = kC0 + tid; i < kC1; i += kFThreads) d[i] = em_ld_dsmem_u32(d + i, 0);
            }
            __syncthreads();
            mark(6);
        }
        if (P.stats && rank == 0 && tid == 0) atomicMax(P.stats + 5, (unsigned long long)steps);
        if (rank == 0 && steps > 0) copy_slot(P.slots + slot, &S.st, T);      // the final state (vpk_em_distribution reads it)
    }
    if (P.stats && rank == 0 && tid == 0)
        for (int k = 0; k < 7; ++k) atomicAdd(P.stats + 8 + k, (unsigned long long)S.mark[k]);
}

// ---------------------------------------------------------------------------
// em_poste: POST of superstep s and the E-step of superstep s + 1 of every active slot in one launch, one
// CLUSTER of kPC CTAs per slot: the line sweeps of the M-step (one warp per hypothesis) are spread over the warps
// of the whole cluster, CTA 0 runs the state machine (post_slot) on the slot state in its shared memory, the other
// CTAs mirror the new E-step constants through distributed shared memory and all of them share the E-step tiles.
// Replaces em_post + em_estep in the kernel-per-phase loops: a superstep is W -> POSTE (two launches, not three).
// ---------------------------------------------------------------------------
struct PosteSmem {
    union U {
        PostScratch sc;
        ESmem es;
    } u;
    __align__(16) EmSlot st;
    RefitAcc tmp[kFThreads / 32];
};

__global__ void __launch_bounds__(kFThreads) em_poste_kernel(EmParams P, TierCtl tc) {
    extern __shared__ __align__(128) unsigned char p_smem_raw[];
    PosteSmem& S = *reinterpret_cast<PosteSmem*>(p_smem_raw);
    const Team T = make_team();
    const int tid = T.tid;
    const uint32_t rank = em_cluster_ctarank(), C = em_cluster_nctarank();
    const int cid = (int)(blockIdx.x / C);
    const int step = P.ctl[3], cur = step & 1;
    const int n_active = P.ctl[cur];
    // every CTA of the cluster has read the control words before its leading CTA can take part in closing the
    // superstep (the closing CTA rewrites them)
    em_cluster_sync();
    if (cid < n_active) {                                          // uniform over the cluster
        const int slot = P.lists[cur * P.n_slots + cid];
        copy_slot(&S.st, P.slots + slot, T);
        __syncthreads();
        const int N = S.st.N, M = S.st.M;
        const Img im = make_img(N, P.ws + S.st.ws_off, P.segs + 4 * (size_t)S.st.base);
        const bool presum = S.st.phase == PH_MSTEP && P.cfg.do_iterations && C > 1;
        if (presum) {
            cluster_presum(refit_acc(S.u.sc), S.tmp, im, N, M, rank, C, T);
            em_cluster_sync();
        }
        if (rank == 0) {
            if (P.stats && tid == 0) atomicAdd(P.stats + 3, 8ull * (3ull * M * N + 5ull * N));
#if defined(VPK_EM_MARKS)
            if (tid == 0) { for (auto& m : S.u.sc.mark) m = 0; S.u.sc.mark_t = clock64(); }
#endif
            post_slot(S.st, S.u.sc, im, P.out, P.cfg, P.overflow, P.overflow_cap, P.ovlock, T, presum);
            __syncthreads();
#if defined(VPK_EM_MARKS)
            if (P.stats && tid == 0) {
                for (int k = 0; k < 10; ++k) atomicAdd(P.stats + 8 + k, (unsigned long long)S.u.sc.mark[k]);
                atomicAdd(P.stats + 18, 1ull);
            }
#endif
            copy_slot(P.slots + slot, &S.st, T);                   // the W kernel and the next POSTE read the state from HBM
            if (tid == 0) P.alive[slot] = S.st.done ? 0 : 1;
        }
        em_cluster_sync();
        if (rank != 0) {
            constexpr int kHead = (int)(offsetof(EmSlot, cur) / 4);
            constexpr int kC0 = (int)(offsetof(EmSlot, pv) / 4), kC1 = (int)(offsetof(EmSlot, cw) / 4);
            uint32_t* d = reinterpret_cast<uint32_t*>(&S.st);
            for (int i = tid; i < kHead; i += kFThreads) d[i] = em_ld_dsmem_u32(d + i, 0);
            for (int i = kC0 + tid; i < kC1; i += kFThreads) d[i] = em_ld_dsmem_u32(d + i, 0);
        }
        __syncthreads();
        em_cluster_sync();                                         // CTA 0 keeps its shared memory until everybody has read it
        // ---- E-step of the next superstep on the VP set POST selected
        if (!S.st.done && S.st.run_e) {
            const int M2 = S.st.M, ntile = (N + kEL - 1) / kEL;
            if (P.stats && rank == 0 && tid == 0) atomicAdd(P.stats + 4, 8ull * (5ull * N + 3ull * M2 * N));
            estep_load_constants(S.u.es, S.st);
            __syncthreads();
            const uint64_t keep = em_policy_keep();
            for (int b = (int)rank; b < ntile; b += (int)C) estep_tile(S.u.es, im, N, M2, b * kEL, keep);
        }
    }
    // the last leading CTA to finish POST closes the superstep: the other list becomes current, this one is emptied
    if (rank == 0) {
        const int live = close_slot_list(P, cur ^ 1, T, (int)(gridDim.x / C));
        if (live >= 0) {
            P.ctl[cur] = 0;
            P.ctl[3] = step + 1;
            const bool stop = step + 1 >= tc.max_steps;
            if (stop && live > 0) P.ctl[5] = 1;
            for (int j = 0; j < tc.n; ++j) cudaGraphSetConditional(tc.h[j], (!stop && live > tc.thr[j]) ? 1u : 0u);
        }
    }
}

// ---------------------------------------------------------------------------
// 'distribution' of the reference's result dict (vp_localisation.py:441-442: the PDF namedtuple of
// probability_functions.py:5, :99-120 for the last E-step) from the planes the last superstep left in the slot
// workspace.  out (doubles): p_v (M) | angles (M,2) | p_l (N) | p_lv (N,M) | lvsq (N,M) | p_vl (M,N)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) em_distribution_kernel(const EmSlot* __restrict__ slot, const double* __restrict__ ws, double* __restrict__ out) {
    const EmSlot& st = *slot;
    const int N = st.N, M = st.M;
    const Img im = make_img(N, const_cast<double*>(ws) + st.ws_off, nullptr);
    double* p_v = out;
    double* angles = p_v + M;
    double* p_l = angles + 2 * (size_t)M;
    double* p_lv = p_l + N;
    double* lvsq = p_lv + (size_t)N * M;
    double* p_vl = lvsq + (size_t)N * M;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < M) {
        const int m = n;
        p_v[m] = st.pv[m];
        const double* v = st.nxt[m];                                  // the final E-step runs on v[i + 1] (:415)
        const double beta = asin(v[1]);
        double inner = v[0] / cos(beta);
        const bool isn = isnan(inner);
        inner = fmax(fmin(inner, 1.0), -1.0);
        if (isn) inner = nan("");
        angles[2 * m] = asin(inner);                                  // calc_angles (probability_functions.py:252-259)
        angles[2 * m + 1] = beta;
    }
    if (n >= N) return;
    double pl = 0.0, part[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int m = 0; m < M; ++m) {
        const double lv = im.lvsq[(size_t)m * N + n];
        const double plv = exp(-(lv * st.inv2s[m])) * st.coef[m];    // calc_plv (:140-145), as the E-step evaluates it
        lvsq[(size_t)n * M + m] = lv;
        p_lv[(size_t)n * M + m] = plv;
        part[m & 7] += plv * st.pv[m];                                // the E-step's own summation order (estep_tile)
        p_vl[(size_t)m * N + n] = im.pvl[(size_t)m * N + n];
    }
    for (int w = 0; w < 8; ++w) pl += part[w];
    p_l[n] = pl < 1e-12 ? 1e-12 : pl;                                 // :117
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
// Device-driven loop: a CUDA graph of conditional WHILE nodes, one per tier of grid sizes
// (n, n/4, n/16, ... slots); tier j repeats the superstep while more than bound[j+1] slots are
// active (POST sets the conditions), so neither the host nor empty CTAs sit on the critical path.
struct EmLoopGraph {
    EmParams key;
    int n = 0, nmax = 0, nbig = 0;
    int supersteps_per_iter = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    void destroy() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        exec = nullptr; graph = nullptr;
    }
};

// A wave's slots are dealt to up to kMaxGroups groups, each running its own device-driven superstep
// loop on its own stream: POST (one CTA per image, latency bound) of one group overlaps the W product
// (HBM bound) of the others, and a group's tail of slow images does not hold the other groups back.
constexpr int kMaxGroups = 8;
constexpr int kPosteCluster = 4;      // CTAs per image of em_poste (408 CTAs for the 102 images of the YUD batch: one wave)
constexpr int kGroupSlots = 26;       // images per group (default; VPK_EM_GROUPS overrides the group count)

struct GroupRun { EmParams P; cudaStream_t s; int n, nmax, nbig, bound, step; bool done; };
enum { MODE_FUSED = 0, MODE_GRAPH = 1, MODE_HOST = 2 };
struct EmWave {
    bool begun = false;                    // wave_begin done, wave_run pending
    bool device_loop = true;
    int mode = MODE_FUSED, cluster = 8, keep = 0;
    int waves_run = 0;                     // waves of the current / last batch that have run (1: its planes are still in the workspace)
    int begin = 0, end = 0, n = 0, G = 0;
    size_t budget = 0;
    std::vector<int32_t> order;
    EmParams P, key_P;
    GroupRun R[kMaxGroups];
    int key_B = 0;
    const int32_t* key_off = nullptr;
};

struct EmState {
    EmWave wave;
    DBuf ws, slots, desc, lists, alive, ctl, stats, overflow, resp, out_small, out_assoc, out_dm, init_vp, init_off, sphere;
    HBuf h_desc, h_cnt;
    bool attr_set = false;
    EmLoopGraph* loop[kMaxGroups] = {};
    cudaStream_t gstream[kMaxGroups] = {};
    cudaEvent_t gdone[kMaxGroups] = {};
    cudaEvent_t gev[kMaxGroups][8] = {};
    cudaEvent_t fork = nullptr, ready = nullptr;
    int last_supersteps = 0;
    unsigned long long totals[6] = {0, 0, 0, 0, 0, 0};   // accumulated W-product statistics + supersteps (profiling runs)
    unsigned long long phase_cycles[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // fused kernel, CTA 0 of every cluster (profiling runs)
    int max_clusters[17] = {};             // co-resident clusters of em_fused_kernel per cluster size (0 = not asked yet)
};

void em_free(vpk_ctx* ctx) {
    if (!ctx->em) return;
    EmState* e = ctx->em;
    e->ws.release(); e->slots.release(); e->desc.release(); e->lists.release(); e->alive.release(); e->ctl.release(); e->stats.release(); e->overflow.release();
    e->resp.release(); e->out_small.release(); e->out_assoc.release(); e->out_dm.release(); e->init_vp.release();
    e->init_off.release(); e->sphere.release(); e->h_desc.release(); e->h_cnt.release();
    for (auto& l : e->loop) if (l) { l->destroy(); delete l; }
    for (auto& g : e->gstream) if (g) cudaStreamDestroy(g);
    for (auto& g : e->gdone) if (g) cudaEventDestroy(g);
    for (auto& r : e->gev) for (auto& g : r) if (g) cudaEventDestroy(g);
    if (e->fork) cudaEventDestroy(e->fork);
    if (e->ready) cudaEventDestroy(e->ready);
    delete e;
    ctx->em = nullptr;
}

// VPK_EM_POSTE=1: a superstep is W -> POSTE (POST and the next E-step in one cluster-per-image kernel) instead of
// E -> W -> POST.  Measured slower on full batches (its mostly idle CTAs compete with W for the SMs), kept for comparison.
static bool use_poste() {
    static const bool v = getenv("VPK_EM_POSTE") != nullptr;
    return v;
}

// one superstep on the stream (direct launch or stream capture): E -> W -> POST over `bound` slots
// nbig: slots of the group whose slabs are split over a cluster (N > 1536); they are the first slots of the group
// (heaviest first), hence the first entries of every active list.
static int enqueue_superstep(vpk_ctx* ctx, cudaStream_t sm, const EmParams& P, int bound, int nmax, int nbig, int n_group,
                             const TierCtl& tc, bool scoped) {
    const bool poste = use_poste();
    if (!poste) {
        KernelScope ks(ctx, "em_estep", scoped);
        em_estep_kernel<<<dim3((nmax + kEL - 1) / kEL, bound), kEThreads, 0, sm>>>(P);
        VPK_TRY(check_launch("em_estep"));
    }
    auto launch_w = [&](int csl, int slots, int n_cols, int want_split) -> int {
        KernelScope ks(ctx, "em_wmat", scoped);
        const int tiles = (n_cols + kTK - 1) / kTK;
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3(tiles * csl, slots);
        lc.blockDim = dim3(kWThreads);
        // fewer CTAs than SMs: deeper ring; similarity matrices of the active slots within half the L2: keep them there
        const bool tail = (long long)tiles * csl * slots <= (long long)ctx->num_sms;
        const int keep = 8.0 * n_cols * n_cols * slots <= 0.5 * (double)ctx->l2_bytes ? 1 : 0;
        lc.dynamicSmemBytes = tail ? sizeof(WSmemT<kStagesTail>) : sizeof(WSmemT<kStages>);
        lc.stream = sm;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = csl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        lc.attrs = at; lc.numAttrs = 1;
        if (tail) VPK_CUDA(cudaLaunchKernelEx(&lc, em_wmat_kernel<kStagesTail>, P, csl, keep, want_split));
        else VPK_CUDA(cudaLaunchKernelEx(&lc, em_wmat_kernel<kStages>, P, csl, keep, want_split));
        return check_launch("em_wmat");
    };
    if (nbig > 0) VPK_TRY(launch_w(wmat_split(nmax), std::min(bound, nbig), nmax, 1));
    if (nbig < n_group) VPK_TRY(launch_w(1, bound, std::min(nmax, 1536), 0));
    if (!poste) {
        KernelScope ks(ctx, "em_post", scoped);
        em_post_kernel<<<bound, kPostThreads, 0, sm>>>(P, tc);
        VPK_TRY(check_launch("em_post"));
    } else {
        KernelScope ks(ctx, "em_poste", scoped);
        static const int pc_env = getenv("VPK_EM_POSTE_CLUSTER") ? atoi(getenv("VPK_EM_POSTE_CLUSTER")) : 0;
        const int pc = (pc_env == 1 || pc_env == 2 || pc_env == 4 || pc_env == 8) ? pc_env : kPosteCluster;
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3(bound * pc);
        lc.blockDim = dim3(kFThreads);
        lc.dynamicSmemBytes = sizeof(PosteSmem);
        lc.stream = sm;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = pc; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        lc.attrs = at; lc.numAttrs = 1;
        VPK_CUDA(cudaLaunchKernelEx(&lc, em_poste_kernel, P, tc));
        VPK_TRY(check_launch("em_poste"));
    }
    return VPK_OK;
}

// the E-step of the first superstep (every later one is the tail of em_poste)
static int enqueue_first_estep(vpk_ctx* ctx, cudaStream_t sm, const EmParams& P, int n, int nmax) {
    KernelScope ks(ctx, "em_estep");
    em_estep_kernel<<<dim3((nmax + kEL - 1) / kEL, n), kEThreads, 0, sm>>>(P);
    return check_launch("em_estep");
}

static int build_loop_graph(vpk_ctx* ctx, cudaStream_t sm, EmLoopGraph& G, const EmParams& P, int n, int nmax, int nbig, int max_steps) {
    G.destroy();
    VPK_CUDA(cudaGraphCreate(&G.graph, 0));
    TierCtl tc;
    memset(&tc, 0, sizeof(tc));
    tc.max_steps = max_steps;
    int bound[kMaxTiers + 1];
    int nt = 0;
    bound[0] = n;
    while (nt + 1 < kMaxTiers && bound[nt] > 8) { bound[nt + 1] = (bound[nt] + 3) / 4; ++nt; }
    ++nt;                                         // tiers 0 .. nt-1
    tc.n = nt;
    for (int j = 0; j < nt; ++j) {
        tc.thr[j] = j + 1 < nt ? bound[j + 1] : 0;
        VPK_CUDA(cudaGraphConditionalHandleCreate(&tc.h[j], G.graph, 1, cudaGraphCondAssignDefault));
    }
    cudaGraphNode_t prev = nullptr;
    for (int j = 0; j < nt; ++j) {
        cudaGraphNodeParams np = {};
        np.type = cudaGraphNodeTypeConditional;
        np.conditional.handle = tc.h[j];
        np.conditional.type = cudaGraphCondTypeWhile;
        np.conditional.size = 1;
        cudaGraphNode_t node;
        VPK_CUDA(cudaGraphAddNode(&node, G.graph, prev ? &prev : nullptr, prev ? 1 : 0, &np));
        cudaGraph_t body = np.conditional.phGraph_out[0];
        VPK_CUDA(cudaStreamBeginCaptureToGraph(sm, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
        int rc = enqueue_superstep(ctx, sm, P, bound[j], nmax, nbig, n, tc, false);
        cudaGraph_t dummy = nullptr;
        cudaError_t e = cudaStreamEndCapture(sm, &dummy);
        if (rc != VPK_OK) return rc;
        VPK_CUDA(e);
        prev = node;
    }
    VPK_CUDA(cudaGraphInstantiate(&G.exec, G.graph, 0));
    G.key = P; G.n = n; G.nmax = nmax; G.nbig = nbig;
    return VPK_OK;
}

// ---- one wave = the images (heaviest first) that fit the workspace.  Group g = slots
// [gstart[g], gstart[g+1]) runs its supersteps on its own stream, driven by a device-side loop graph
// (the default) or by the host (VPK_EM_HOST_LOOP=1 and profiling runs: supersteps enqueued in chunks,
// the active count read LA chunks behind).  wave_begin needs the segments only (slot layout, pair
// pass); wave_run needs the CNN response and the sphere images (initial hypotheses, supersteps).

// plan of wave [begin, end) of `order`: buffers, slot descriptors, groups, kernel parameters
static int plan_wave(vpk_ctx* ctx, EmState* st, const EmParams& P0, const int32_t* h_offsets, int B) {
    EmWave& W = st->wave;
    const int begin = W.begin;
    size_t doubles = 0;
    int end = begin;
    const int nmax = std::max(1, h_offsets[W.order[begin] + 1] - h_offsets[W.order[begin]]);
    while (end < B && end - begin < 32768) {
        const int N = h_offsets[W.order[end] + 1] - h_offsets[W.order[end]];
        const size_t need = slot_doubles(N);
        if (end > begin && doubles + need > W.budget) break;
        doubles += need;
        ++end;
    }
    const int n = end - begin;
    VPK_TRY(st->ws.ensure(doubles * sizeof(double)));
    VPK_TRY(st->slots.ensure(sizeof(EmSlot) * (size_t)n));
    VPK_TRY(st->desc.ensure(sizeof(SlotDesc) * (size_t)n));
    VPK_TRY(st->lists.ensure(2 * sizeof(int) * (size_t)n));
    VPK_TRY(st->alive.ensure(sizeof(int) * (size_t)n));
    const size_t ov = (size_t)nmax * nmax + 6 * (size_t)nmax + 16;
    VPK_TRY(st->overflow.ensure(ov * sizeof(double)));
    VPK_TRY(st->h_desc.ensure(sizeof(SlotDesc) * (size_t)n));
    SlotDesc* hd = st->h_desc.as<SlotDesc>();
    // groups: the wave's images (heaviest first) are dealt round-robin, so every group gets the same
    // mix of sizes; a group's slots are contiguous.  One group per ~kGroupSlots images.
    static const int env_groups = getenv("VPK_EM_GROUPS") ? atoi(getenv("VPK_EM_GROUPS")) : 0;
    // How the superstep loop runs (read per call: smoke() and the tests toggle it):
    //   graph (default) : W / POSTE kernels in a CUDA graph of conditional WHILE nodes, several groups in flight
    //   host            : the same kernels launched by the host (VPK_EM_HOST_LOOP=1, profiling runs)
    //   fused           : one persistent kernel, a cluster per image (em_fused_kernel, VPK_EM_MODE=fused): measured
    //                     slower on full batches (the CTAs of a cluster idle while its leading CTA runs POST), see DESIGN.md
    const char* mode_env = getenv("VPK_EM_MODE");
    const char* cl_env = getenv("VPK_EM_CLUSTER");
    int cluster = cl_env ? atoi(cl_env) : (nmax > 3072 ? 16 : 8);
    if (cluster != 1 && cluster != 2 && cluster != 4 && cluster != 8 && cluster != 16) cluster = 8;
    int mode = MODE_GRAPH;
    if (getenv("VPK_EM_HOST_LOOP")) mode = MODE_HOST;
    else if (mode_env && !strcmp(mode_env, "fused")) mode = MODE_FUSED;
    else if (mode_env && !strcmp(mode_env, "host")) mode = MODE_HOST;
    if (mode == MODE_GRAPH && ctx->profiling) mode = MODE_HOST;      // no per-kernel events inside a graph
    W.mode = mode; W.cluster = cluster;
    W.device_loop = mode == MODE_GRAPH;
    int G = env_groups > 0 ? env_groups : (n + kGroupSlots - 1) / kGroupSlots;
    G = std::max(1, std::min(G, std::min(n, kMaxGroups)));
    if (ctx->profiling || mode == MODE_FUSED) G = 1;   // per-kernel events are recorded on the context's stream; the fused
                                                       // kernel takes the images from one queue, heaviest first
    EmParams P;
    memcpy(&P, &P0, sizeof(EmParams));
    P.slots = st->slots.as<EmSlot>(); P.desc = st->desc.as<SlotDesc>(); P.ws = st->ws.as<double>();
    P.lists = st->lists.as<int>(); P.alive = st->alive.as<int>(); P.ctl = st->ctl.as<int>();
    P.ovlock = st->ctl.as<int>() + kMaxGroups * kCtlInts;
    P.stats = ctx->profiling ? st->stats.as<unsigned long long>() : nullptr;
    P.overflow = st->overflow.as<double>(); P.overflow_cap = ov;
    P.n_slots = n;
    size_t off = 0;
    int i = 0;
    for (int g = 0; g < G; ++g) {
        GroupRun& r = W.R[g];
        const int g0 = i;
        r.nmax = 1; r.nbig = 0;
        for (int k = g; k < n; k += G, ++i) {
            const int b = W.order[begin + k];
            hd[i].img = b; hd[i].base = h_offsets[b]; hd[i].N = h_offsets[b + 1] - h_offsets[b]; hd[i].pad = 0;
            hd[i].ws_off = off;
            off += slot_doubles(hd[i].N);
            r.nmax = std::max(r.nmax, hd[i].N);
            r.nbig += wmat_split(hd[i].N) > 1 ? 1 : 0;
        }
        r.s = ctx->profiling ? ctx->stream : st->gstream[g];
        memcpy(&r.P, &P, sizeof(EmParams));      // padding included: the loop graph is keyed on the bytes
        r.n = i - g0; r.bound = r.n; r.step = 0; r.done = false;
        r.P.slots = P.slots + g0; r.P.desc = P.desc + g0; r.P.lists = P.lists + 2 * (size_t)g0; r.P.alive = P.alive + g0;
        r.P.ctl = P.ctl + g * kCtlInts; r.P.n_slots = r.n;
    }
    memcpy(&W.P, &P, sizeof(EmParams));
    W.n = n; W.G = G; W.end = end;
    return VPK_OK;
}

// descriptors, control words, pair pass (E3 + E4) of every group on its stream
static int wave_begin(vpk_ctx* ctx, EmState* st) {
    EmWave& W = st->wave;
    cudaStream_t sm = ctx->stream;
    VPK_CUDA(cudaMemcpyAsync(st->desc.p, st->h_desc.p, sizeof(SlotDesc) * (size_t)W.n, cudaMemcpyHostToDevice, sm));
    VPK_CUDA(cudaMemsetAsync(st->ctl.p, 0, (kMaxGroups + 1) * kCtlInts * sizeof(int), sm));
    if (W.P.stats) VPK_CUDA(cudaMemsetAsync(W.P.stats, 0, 32 * sizeof(unsigned long long), sm));
    VPK_CUDA(cudaEventRecord(st->fork, sm));
    for (int g = 0; g < W.G; ++g) {
        GroupRun& r = W.R[g];
        if (r.s != sm) VPK_CUDA(cudaStreamWaitEvent(r.s, st->fork, 0));
        if (r.P.cfg.use_weights) {
            KernelScope ks(ctx, "em_pair");
            em_pair_kernel<<<dim3((r.nmax + kTK - 1) / kTK, r.n), kPairThreads, 0, r.s>>>(r.P);
            VPK_TRY(check_launch("em_pair"));
        }
    }
    W.begun = true;
    return VPK_OK;
}

// initial hypotheses and the superstep loops; returns when every slot of the wave is finished
static int wave_run(vpk_ctx* ctx, EmState* st) {
    EmWave& W = st->wave;
    cudaStream_t sm = ctx->stream;
    const int G = W.G;
    const int max_steps = 64 * (W.P.cfg.num_iter + 8);
    int* h_cnt = st->h_cnt.as<int>();
    static const bool trace = getenv("VPK_EM_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    int rebuilt = 0;
    W.begun = false;
    VPK_CUDA(cudaEventRecord(st->ready, sm));          // CNN response and sphere images are complete
    auto join = [&](int g) {
        if (W.R[g].s == sm) return cudaSuccess;
        cudaError_t e = cudaEventRecord(st->gdone[g], W.R[g].s);
        return e != cudaSuccess ? e : cudaStreamWaitEvent(sm, st->gdone[g], 0);
    };
    for (int g = 0; g < G; ++g) {
        GroupRun& r = W.R[g];
        if (r.s != sm) VPK_CUDA(cudaStreamWaitEvent(r.s, st->ready, 0));
        {
            KernelScope ks(ctx, "em_init");
            em_init_kernel<<<r.n, kInitThreads, 0, r.s>>>(r.P);
            VPK_TRY(check_launch("em_init"));
        }
        if (W.mode == MODE_FUSED) {
            const int C = W.cluster;
            if (!st->max_clusters[C]) {
                cudaLaunchConfig_t oc = {};
                oc.gridDim = dim3(C * 64); oc.blockDim = dim3(kFThreads); oc.dynamicSmemBytes = sizeof(FusedSmem);
                cudaLaunchAttribute oa[1];
                oa[0].id = cudaLaunchAttributeClusterDimension;
                oa[0].val.clusterDim.x = C; oa[0].val.clusterDim.y = 1; oa[0].val.clusterDim.z = 1;
                oc.attrs = oa; oc.numAttrs = 1;
                int nc = 0;
                VPK_CUDA(cudaOccupancyMaxActiveClusters(&nc, em_fused_kernel, &oc));
                if (nc <= 0) { set_error("vpk_em: a cluster of %d CTAs of em_fused_kernel does not fit this device", C); return VPK_ERR_STATE; }
                st->max_clusters[C] = nc;
            }
            const int nclusters = std::max(1, std::min(r.n, st->max_clusters[C]));
            // similarity matrices of the images in flight (the heaviest ones come first) within 60 % of the L2: default
            // cache policy, they stay resident from one superstep to the next (evict-first otherwise)
            double inflight = 0.0;
            const SlotDesc* hd = st->h_desc.as<SlotDesc>();
            for (int i = 0; i < nclusters; ++i) inflight += 8.0 * hd[i].N * hd[i].N;
            W.keep = inflight <= 0.6 * (double)ctx->l2_bytes ? 1 : 0;
            KernelScope ks(ctx, "em_fused");
            cudaLaunchConfig_t lc = {};
            lc.gridDim = dim3(nclusters * C);
            lc.blockDim = dim3(kFThreads);
            lc.dynamicSmemBytes = sizeof(FusedSmem);
            lc.stream = r.s;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            lc.attrs = at; lc.numAttrs = 1;
            VPK_CUDA(cudaLaunchKernelEx(&lc, em_fused_kernel, r.P, max_steps, W.keep));
            VPK_TRY(check_launch("em_fused"));
            VPK_CUDA(join(g));
        }
        if (W.mode != MODE_FUSED && use_poste()) VPK_TRY(enqueue_first_estep(ctx, r.s, r.P, r.n, r.nmax));
        if (W.device_loop) {
            EmLoopGraph& L = *st->loop[g];
            if (!L.exec || L.n != r.n || L.nmax != r.nmax || L.nbig != r.nbig || memcmp(&L.key, &r.P, sizeof(EmParams)) != 0) {
                VPK_TRY(build_loop_graph(ctx, r.s, L, r.P, r.n, r.nmax, r.nbig, max_steps));
                ++rebuilt;
            }
            VPK_CUDA(cudaGraphLaunch(L.exec, r.s));
            VPK_CUDA(join(g));
        }
    }
    int steps = 0;
    if (W.mode == MODE_FUSED) {
        VPK_CUDA(cudaMemcpyAsync(h_cnt, W.P.ctl, kCtlInts * sizeof(int), cudaMemcpyDeviceToHost, sm));
        VPK_CUDA(cudaStreamSynchronize(sm));
        if (h_cnt[5]) { set_error("vpk_em: supersteps did not terminate"); return VPK_ERR_STATE; }
    } else if (W.device_loop) {
        VPK_CUDA(cudaMemcpyAsync(h_cnt, W.P.ctl, G * kCtlInts * sizeof(int), cudaMemcpyDeviceToHost, sm));
        VPK_CUDA(cudaStreamSynchronize(sm));
        for (int g = 0; g < G; ++g) {
            const int* c = h_cnt + g * kCtlInts;
            ctx->launches += ((use_poste() ? 2 : 3) + ((W.R[g].nbig > 0 && W.R[g].nbig < W.R[g].n) ? 1 : 0)) * (int64_t)c[3];
            steps = std::max(steps, c[3]);
            if (c[5]) { set_error("vpk_em: supersteps did not terminate"); return VPK_ERR_STATE; }
        }
    } else {
        TierCtl tc;
        memset(&tc, 0, sizeof(tc));
        tc.max_steps = max_steps;
        static const int LA = getenv("VPK_EM_LOOKAHEAD") ? std::max(1, std::min(7, atoi(getenv("VPK_EM_LOOKAHEAD")))) : 3;
        int active = G;
        for (int chunk = 0; active > 0; ++chunk) {
            for (int g = 0; g < G; ++g) {
                GroupRun& r = W.R[g];
                if (r.done) continue;
                int* ring = h_cnt + g * 8;
                if (chunk >= LA) {
                    VPK_CUDA(cudaEventSynchronize(st->gev[g][(chunk - LA) & 7]));
                    r.bound = ring[(chunk - LA) & 7];     // upper bound of the number of active slots (they only ever finish)
                    if (r.bound <= 0) {
                        r.done = true;
                        --active;
                        VPK_CUDA(join(g));
                        continue;
                    }
                }
                for (int k = 0; k < kChunkSteps; ++k, ++r.step)
                    VPK_TRY(enqueue_superstep(ctx, r.s, r.P, r.bound, r.nmax, r.nbig, r.n, tc, true));
                // length of the list the next superstep will read
                VPK_CUDA(cudaMemcpyAsync(ring + (chunk & 7), r.P.ctl + (r.step & 1), sizeof(int), cudaMemcpyDeviceToHost, r.s));
                VPK_CUDA(cudaEventRecord(st->gev[g][chunk & 7], r.s));
                if (r.step > max_steps) { set_error("vpk_em: supersteps did not terminate"); return VPK_ERR_STATE; }
            }
        }
        VPK_CUDA(cudaStreamSynchronize(sm));
        for (int g = 0; g < G; ++g) steps = std::max(steps, W.R[g].step);
    }
    if (trace) {
        const auto t_end = std::chrono::steady_clock::now();
        fprintf(stderr, "[vpk_em] wave n=%d groups=%d %s, cluster=%d keep=%d, graphs rebuilt=%d, supersteps %d, %.3f ms\n", W.n, G,
                W.mode == MODE_FUSED ? "fused kernel" : (W.device_loop ? "device loop" : "host loop"), W.cluster, W.keep, rebuilt, steps,
                std::chrono::duration<double, std::milli>(t_end - t_begin).count());
    }
    st->last_supersteps = steps;
    if (W.P.stats) {
        unsigned long long h[16] = {};
        VPK_CUDA(cudaMemcpy(h, W.P.stats, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (int k = 0; k < 3; ++k) st->totals[k] += h[k];
        if (W.mode == MODE_FUSED) {
            steps = (int)h[5];                                   // supersteps of the slowest image
            st->last_supersteps = steps;
            for (int k = 0; k < 7; ++k) st->phase_cycles[k] += h[8 + k];
        }
        st->totals[3] += (unsigned long long)steps;
        st->totals[4] += h[3];
        st->totals[5] += h[4];
#if defined(VPK_EM_MARKS)
        unsigned long long mk[11];
        VPK_CUDA(cudaMemcpy(mk, W.P.stats + (W.mode == MODE_FUSED ? 16 : 8), 11 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        fprintf(stderr, "[vpk_em] POST cycles per slot-superstep (%llu):", mk[10]);
        for (int k = 0; k < 10; ++k) fprintf(stderr, " m%d=%.0f", k, (double)mk[k] / (double)std::max<unsigned long long>(mk[10], 1));
        fprintf(stderr, "\n");
        if (W.mode != MODE_FUSED) {
            unsigned long long sp[6];
            VPK_CUDA(cudaMemcpy(sp, W.P.stats + 19, 6 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            fprintf(stderr, "[vpk_em] split cycles per completed split (%llu): stats=%.0f pick=%.0f distances=%.0f linkage=%.0f refit=%.0f\n", sp[5],
                    (double)sp[0] / std::max<unsigned long long>(sp[5], 1), (double)sp[1] / std::max<unsigned long long>(sp[5], 1),
                    (double)sp[2] / std::max<unsigned long long>(sp[5], 1), (double)sp[3] / std::max<unsigned long long>(sp[5], 1),
                    (double)sp[4] / std::max<unsigned long long>(sp[5], 1));
            unsigned long long mx[7];
            VPK_CUDA(cudaMemcpy(mx, W.P.stats + 25, 7 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            fprintf(stderr, "[vpk_em] slowest split (N = %llu): %llu cycles: stats=%llu pick=%llu distances=%llu linkage=%llu refit=%llu\n", mx[6], mx[0],
                    mx[1], mx[2], mx[3], mx[4], mx[5]);
        }
#endif
    }
    return VPK_OK;
}

// phase EM_ALL: the whole stage.  EM_EARLY: only what needs the segments (layout and pair pass of the
// first wave, on the group streams: overlaps whatever the caller enqueues on the context's stream
// afterwards, i.e. sphere mapping and the CNN); the matching EM_ALL call then continues from there.
int em_dev(vpk_ctx* ctx, const double* d_lines, const double* d_segments, const int32_t* d_offsets,
           const int32_t* h_offsets, int32_t B, const float* d_resp_f32, const double* d_resp_f64,
           const uint8_t* d_sphere, int32_t S, const double* d_init_vp, const int32_t* d_init_off,
           const vpk_em_config* cfg, const EmDeviceOut& out, int phase) {
    (void)d_offsets;
    if (B <= 0) return VPK_OK;
    if (!ctx->em) ctx->em = new EmState();
    EmState* st = ctx->em;
    if (!st->attr_set) {
        VPK_CUDA(cudaFuncSetAttribute(em_wmat_kernel<kStages>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WSmemT<kStages>)));
        VPK_CUDA(cudaFuncSetAttribute(em_wmat_kernel<kStagesTail>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WSmemT<kStagesTail>)));
        VPK_CUDA(cudaFuncSetAttribute(em_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
        VPK_CUDA(cudaFuncSetAttribute(em_poste_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PosteSmem)));
        VPK_CUDA(cudaFuncSetAttribute(em_fused_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        for (auto& ev : st->gdone) VPK_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        for (auto& r : st->gev) for (auto& ev : r) VPK_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        VPK_CUDA(cudaEventCreateWithFlags(&st->fork, cudaEventDisableTiming));
        VPK_CUDA(cudaEventCreateWithFlags(&st->ready, cudaEventDisableTiming));
        for (auto& g : st->gstream) VPK_CUDA(cudaStreamCreateWithFlags(&g, cudaStreamNonBlocking));
        for (auto& l : st->loop) l = new EmLoopGraph();
        st->attr_set = true;
    }
    EmWave& W = st->wave;

    EmParams P;
    memset(&P, 0, sizeof(P));                   // padding included: the loop graph is keyed on the bytes
    P.lines = d_lines; P.segs = d_segments;
    P.resp32 = d_resp_f32; P.resp64 = d_resp_f64; P.sphere = d_sphere; P.S = S;
    P.init_vp = d_init_vp; P.init_off = d_init_off;
    P.cfg = *cfg;
    P.out.status = out.status; P.out.n_vp = out.n_vp; P.out.iterations = out.iterations; P.out.vp = out.vp;
    P.out.sigma = out.sigma; P.out.counts = out.counts; P.out.counts_weighted = out.counts_weighted;
    P.out.vp_assoc = out.vp_assoc; P.out.decision_metric = out.decision_metric;

    // continue a wave begun by an EM_EARLY call with the same arguments?
    const bool resume = W.begun && phase == EM_ALL && W.key_B == B && W.key_off == h_offsets && memcmp(&W.key_P, &P, sizeof(EmParams)) == 0;
    if (W.begun && !resume) {
        // an early pair pass nobody continued: drain it before its buffers are reused
        for (int g = 0; g < W.G; ++g) VPK_CUDA(cudaStreamSynchronize(W.R[g].s));
        W.begun = false;
    }
    if (!resume) {
        // heaviest images first
        W.order.resize(B);
        for (int b = 0; b < B; ++b) W.order[b] = b;
        std::stable_sort(W.order.begin(), W.order.end(), [&](int a, int b) {
            return (h_offsets[a + 1] - h_offsets[a]) > (h_offsets[b + 1] - h_offsets[b]);
        });
        // workspace budget of a wave: the whole batch if the workspace already holds it (no driver query on
        // the steady-state path), else half of what is free
        size_t all_doubles = 0;
        for (int b = 0; b < B; ++b) all_doubles += slot_doubles(h_offsets[b + 1] - h_offsets[b]);
        W.budget = all_doubles;
        if (all_doubles * sizeof(double) > st->ws.cap) {
            size_t free_b = 0, total_b = 0;
            VPK_CUDA(cudaMemGetInfo(&free_b, &total_b));
            W.budget = std::max<size_t>((free_b + st->ws.cap) / 2, (size_t)1 << 28) / sizeof(double);
        }
        // test knob: cap the workspace of a wave (MiB) so that small batches run in several waves
        if (const char* cap_mb = getenv("VPK_EM_WAVE_MB")) W.budget = std::min<size_t>(W.budget, (size_t)std::max(1, atoi(cap_mb)) * ((size_t)1 << 20) / sizeof(double));
        VPK_TRY(st->h_cnt.ensure(kMaxGroups * 8 * sizeof(int)));
        VPK_TRY(st->ctl.ensure((kMaxGroups + 1) * kCtlInts * sizeof(int)));
        VPK_TRY(st->stats.ensure(32 * sizeof(unsigned long long)));
        W.begin = 0;
        W.waves_run = 0;
        W.key_B = B; W.key_off = h_offsets;
        memcpy(&W.key_P, &P, sizeof(EmParams));
    }
    while (W.begin < B) {
        if (!W.begun) {
            VPK_TRY(plan_wave(ctx, st, P, h_offsets, B));
            VPK_TRY(wave_begin(ctx, st));
        }
        if (phase == EM_EARLY) return VPK_OK;
        VPK_TRY(wave_run(ctx, st));
        ++W.waves_run;
        W.begin = W.end;
    }
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_em_stats(vpk_ctx* ctx, uint64_t out[6], int reset) {
    if (!ctx || !out) { set_error("vpk_em_stats: bad argument"); return VPK_ERR_ARG; }
    for (int k = 0; k < 6; ++k) out[k] = ctx->em ? ctx->em->totals[k] : 0;
    if (reset && ctx->em) for (auto& t : ctx->em->totals) t = 0;
    return VPK_OK;
}

int vpk_em_distribution(vpk_ctx* ctx, int32_t image, int32_t n_vp, int32_t n_lines, double* p_v, double* p_lv, double* p_vl,
                        double* p_l, double* lvsq, double* angles) {
    if (!ctx || !ctx->em || image < 0 || !p_v || !p_lv || !p_vl || !p_l || !lvsq || !angles) { set_error("vpk_em_distribution: bad argument"); return VPK_ERR_ARG; }
    EmState* st = ctx->em;
    EmWave& W = st->wave;
    if (W.begun || W.n <= 0 || W.waves_run != 1 || W.n != W.key_B) {
        set_error("vpk_em_distribution: the planes of the last E-step are kept for batches that ran in one workspace wave only");
        return VPK_ERR_STATE;
    }
    const SlotDesc* hd = st->h_desc.as<SlotDesc>();
    int slot = -1;
    for (int i = 0; i < W.n; ++i) if (hd[i].img == image) { slot = i; break; }
    if (slot < 0) { set_error("vpk_em_distribution: image %d is not part of the last batch", image); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    EmSlot hs;
    VPK_CUDA(cudaMemcpy(&hs, st->slots.as<EmSlot>() + slot, sizeof(EmSlot), cudaMemcpyDeviceToHost));
    if (hs.status != VPK_EM_OK || hs.M != n_vp || hs.N != n_lines) {
        set_error("vpk_em_distribution: image %d finished with status %d, %d hypotheses, %d lines (caller expects %d, %d)", image, hs.status,
                  hs.M, hs.N, n_vp, n_lines);
        return VPK_ERR_ARG;
    }
    const size_t M = (size_t)hs.M, N = (size_t)hs.N, total = 3 * M + N + 3 * N * M;
    VPK_TRY(ctx->d_misc.ensure(total * sizeof(double)));
    double* d = ctx->d_misc.as<double>();
    {
        KernelScope ks(ctx, "em_distribution");
        const unsigned blocks = (unsigned)((std::max(N, M) + 255) / 256);
        em_distribution_kernel<<<blocks, 256, 0, ctx->stream>>>(st->slots.as<EmSlot>() + slot, st->ws.as<double>(), d);
        VPK_TRY(check_launch("em_distribution"));
    }
    auto D2H = [&](double* dst, const double* src, size_t n) { return cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream); };
    VPK_CUDA(D2H(p_v, d, M));
    VPK_CUDA(D2H(angles, d + M, 2 * M));
    VPK_CUDA(D2H(p_l, d + 3 * M, N));
    VPK_CUDA(D2H(p_lv, d + 3 * M + N, N * M));
    VPK_CUDA(D2H(lvsq, d + 3 * M + N + N * M, N * M));
    VPK_CUDA(D2H(p_vl, d + 3 * M + N + 2 * N * M, N * M));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

int vpk_em_debug_fetch(vpk_ctx* ctx, int32_t image, int32_t which, double* out, int64_t capacity, int64_t* count) {
    if (count) *count = 0;
    if (!ctx || image < 0 || which < 0 || which >= VPK_EM_NBUF || capacity < 0 || (capacity > 0 && !out)) {
        set_error("vpk_em_debug_fetch: bad argument");
        return VPK_ERR_ARG;
    }
    EmState* st = ctx->em;
    if (!st || st->wave.begun || st->wave.n <= 0 || st->wave.waves_run != 1 || st->wave.n != st->wave.key_B) {
        set_error("vpk_em_debug_fetch: the EM workspace is kept for the last batch only, and only if it ran in one workspace wave");
        return VPK_ERR_STATE;
    }
    const EmWave& W = st->wave;
    const SlotDesc* hd = st->h_desc.as<SlotDesc>();
    int slot = -1;
    for (int i = 0; i < W.n; ++i) if (hd[i].img == image) { slot = i; break; }
    if (slot < 0) { set_error("vpk_em_debug_fetch: image %d is not part of the last batch", image); return VPK_ERR_ARG; }
    if (which == VPK_EM_BUF_LSIM && !W.key_P.cfg.use_weights) {
        set_error("vpk_em_debug_fetch: the last batch ran with use_weights = 0, the pair pass did not compute lsim");
        return VPK_ERR_STATE;
    }
    VPK_CUDA(cudaSetDevice(ctx->device));
    const int N = hd[slot].N;
    const Img im = make_img(N, st->ws.as<double>() + hd[slot].ws_off, nullptr);
    const double* src = nullptr;
    size_t n = 0;
    EmSlot hs;
    if (which >= VPK_EM_BUF_LVSQ) {
        VPK_CUDA(cudaMemcpy(&hs, st->slots.as<EmSlot>() + slot, sizeof(EmSlot), cudaMemcpyDeviceToHost));
        if (hs.status != VPK_EM_OK) {
            set_error("vpk_em_debug_fetch: image %d finished with status %d, its last E-step planes are not kept", image, hs.status);
            return VPK_ERR_STATE;
        }
    }
    const size_t M = which >= VPK_EM_BUF_LVSQ ? (size_t)hs.M : 0;
    switch (which) {
    case VPK_EM_BUF_LSIM: src = im.lsim; n = lsim_doubles(N); break;
    case VPK_EM_BUF_COLSUM: src = im.colsum; n = N; break;
    case VPK_EM_BUF_LWEIGHT: src = im.lweight; n = N; break;
    case VPK_EM_BUF_LVSQ: src = im.lvsq; n = M * N; break;
    case VPK_EM_BUF_PVL: src = im.pvl; n = M * N; break;
    case VPK_EM_BUF_W: src = im.w; n = M * N; break;
    case VPK_EM_BUF_WT: src = im.wt; n = (M + kMP - 1) / kMP * (size_t)N * kMPS; break;
    default: n = 5 * M; break;                                            // VPK_EM_BUF_ESTEP: from the slot state
    }
    if (count) *count = (int64_t)n;
    if (!out) return VPK_OK;                                              // size query
    if ((size_t)capacity < n) { set_error("vpk_em_debug_fetch: %zu doubles needed, room for %lld", n, (long long)capacity); return VPK_ERR_ARG; }
    if (which == VPK_EM_BUF_ESTEP) {
        const double* c[5] = {hs.pv, hs.vx, hs.vy, hs.inv2s, hs.coef};
        for (int r = 0; r < 5; ++r) memcpy(out + r * M, c[r], M * sizeof(double));
        return VPK_OK;
    }
    if (n) {
        VPK_CUDA(cudaMemcpyAsync(out, src, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return VPK_OK;
}

int vpk_em_phase_cycles(vpk_ctx* ctx, uint64_t out[8], int reset) {
    if (!ctx || !out) { set_error("vpk_em_phase_cycles: bad argument"); return VPK_ERR_ARG; }
    for (int k = 0; k < 8; ++k) out[k] = ctx->em ? ctx->em->phase_cycles[k] : 0;
    if (reset && ctx->em) for (auto& t : ctx->em->phase_cycles) t = 0;
    return VPK_OK;
}

void vpk_em_default_config(vpk_em_config* c) {
    if (!c) return;
    c->num_iter = 100; c->num_init_vp = 25; c->split_merge_freq = 10; c->num_min_lines = 3;
    c->do_merge = 1; c->do_split = 1; c->do_iterations = 1; c->use_weights = 1;
    c->wbias = 1.0; c->merge_thresh = 1e-3; c->outlier_thresh = 1.96 * 1.96; c->final_convergence = 5e-3;
    c->s_thresh = 1e-200;
}

int vpk_em(vpk_ctx* ctx, const double* lines, const double* segments, const int32_t* offsets, int32_t B,
           const double* responses, const uint8_t* sphere_images, int32_t S, const double* init_vp,
           const int32_t* init_vp_offsets, const vpk_em_config* cfg_in, vpk_em_result* out) {
    if (!ctx || !offsets || !out || B < 0 || S <= 0) { set_error("vpk_em: bad argument"); return VPK_ERR_ARG; }
    if (B == 0) return VPK_OK;
    if (!responses || (!sphere_images && !init_vp)) { set_error("vpk_em: responses and sphere_images (or init_vp) are required"); return VPK_ERR_ARG; }
    if (!out->status || !out->n_vp || !out->iterations || !out->vp || !out->sigma || !out->counts || !out->counts_weighted ||
        !out->vp_assoc) { set_error("vpk_em: result arrays must be allocated by the caller"); return VPK_ERR_ARG; }
    vpk_em_config cfg;
    if (cfg_in) cfg = *cfg_in; else vpk_em_default_config(&cfg);
    if (cfg.split_merge_freq <= 0 || cfg.num_iter < 0 || cfg.num_init_vp < 0) { set_error("vpk_em: bad config"); return VPK_ERR_ARG; }
    if (offsets[0] != 0) { set_error("vpk_em: offsets[0] must be 0"); return VPK_ERR_ARG; }
    for (int b = 0; b < B; ++b) if (offsets[b + 1] < offsets[b]) { set_error("vpk_em: offsets must be non-decreasing"); return VPK_ERR_ARG; }
    const int64_t sumN = offsets[B];
    if (sumN > 0 && (!lines || !segments)) { set_error("vpk_em: lines/segments are NULL"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->em) ctx->em = new EmState();
    EmState* st = ctx->em;
    const size_t plane = (size_t)S * S;
    VPK_TRY(ctx->d_lines.ensure((sumN + 1) * 3 * sizeof(double)));
    VPK_TRY(ctx->d_segments.ensure((sumN + 1) * 4 * sizeof(double)));
    VPK_TRY(st->resp.ensure((size_t)B * kCells * sizeof(double)));
    if (sphere_images) VPK_TRY(st->sphere.ensure(plane * B));
    // small outputs packed: vp | sigma | cw | status,n_vp,iterations (3B int32) | counts (B*64 int32)
    const size_t n_i32 = 3 * (size_t)B + (size_t)B * kMaxM;
    const size_t n_f64 = (size_t)B * kMaxM * 5;
    VPK_TRY(st->out_small.ensure(n_f64 * sizeof(double) + n_i32 * sizeof(int32_t) + 64));
    VPK_TRY(st->out_assoc.ensure((sumN + 1) * sizeof(int32_t)));
    if (out->decision_metric) VPK_TRY(st->out_dm.ensure(((size_t)kMaxM * sumN + 1) * sizeof(double)));
    if (sumN) {
        VPK_CUDA(cudaMemcpyAsync(ctx->d_lines.p, lines, sumN * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        VPK_CUDA(cudaMemcpyAsync(ctx->d_segments.p, segments, sumN * 4 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    VPK_CUDA(cudaMemcpyAsync(st->resp.p, responses, (size_t)B * kCells * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (sphere_images) VPK_CUDA(cudaMemcpyAsync(st->sphere.p, sphere_images, plane * B, cudaMemcpyHostToDevice, ctx->stream));
    const double* d_init = nullptr;
    const int32_t* d_ioff = nullptr;
    if (init_vp) {
        if (!init_vp_offsets) { set_error("vpk_em: init_vp needs init_vp_offsets"); return VPK_ERR_ARG; }
        if (init_vp_offsets[0] != 0) { set_error("vpk_em: init_vp_offsets[0] must be 0"); return VPK_ERR_ARG; }
        for (int b = 0; b < B; ++b)
            if (init_vp_offsets[b + 1] < init_vp_offsets[b]) { set_error("vpk_em: init_vp_offsets must be non-decreasing (B + 1 entries)"); return VPK_ERR_ARG; }
        size_t nv = init_vp_offsets[B];
        VPK_TRY(st->init_vp.ensure((nv + 1) * 3 * sizeof(double)));
        VPK_TRY(st->init_off.ensure((B + 1) * sizeof(int32_t)));
        VPK_CUDA(cudaMemcpyAsync(st->init_vp.p, init_vp, nv * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        VPK_CUDA(cudaMemcpyAsync(st->init_off.p, init_vp_offsets, (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        d_init = st->init_vp.as<double>();
        d_ioff = st->init_off.as<int32_t>();
    }
    EmDeviceOut d;
    double* f = st->out_small.as<double>();
    d.vp = f; f += (size_t)B * kMaxM * 3;
    d.sigma = f; f += (size_t)B * kMaxM;
    d.counts_weighted = f; f += (size_t)B * kMaxM;
    int32_t* ip = reinterpret_cast<int32_t*>(f);
    d.status = ip; ip += B;
    d.n_vp = ip; ip += B;
    d.iterations = ip; ip += B;
    d.counts = ip;
    d.vp_assoc = st->out_assoc.as<int32_t>();
    d.decision_metric = out->decision_metric ? st->out_dm.as<double>() : nullptr;
    VPK_TRY(em_dev(ctx, ctx->d_lines.as<double>(), ctx->d_segments.as<double>(), nullptr, offsets, B,
                   nullptr, st->resp.as<double>(), sphere_images ? st->sphere.as<uint8_t>() : nullptr, S, d_init, d_ioff,
                   &cfg, d));
    auto D2H = [&](void* dst, const void* src, size_t bytes) {
        return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
    };
    VPK_CUDA(D2H(out->vp, d.vp, (size_t)B * kMaxM * 3 * sizeof(double)));
    VPK_CUDA(D2H(out->sigma, d.sigma, (size_t)B * kMaxM * sizeof(double)));
    VPK_CUDA(D2H(out->counts_weighted, d.counts_weighted, (size_t)B * kMaxM * sizeof(double)));
    VPK_CUDA(D2H(out->status, d.status, (size_t)B * sizeof(int32_t)));
    VPK_CUDA(D2H(out->n_vp, d.n_vp, (size_t)B * sizeof(int32_t)));
    VPK_CUDA(D2H(out->iterations, d.iterations, (size_t)B * sizeof(int32_t)));
    VPK_CUDA(D2H(out->counts, d.counts, (size_t)B * kMaxM * sizeof(int32_t)));
    if (sumN) VPK_CUDA(D2H(out->vp_assoc, d.vp_assoc, sumN * sizeof(int32_t)));
    if (out->decision_metric && sumN) VPK_CUDA(D2H(out->decision_metric, d.decision_metric, (size_t)kMaxM * sumN * sizeof(double)));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

}  // extern "C"
