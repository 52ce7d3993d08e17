// bls_host.cu — host driver + C ABI of the batch BLS verification path.
//
// Mirrors bls::verify_signature_sets (crypto/bls/src/impls/blst.rs:37-119) at the batch level: the caller (the
// Rust shim in INTEGRATION.md, or lighthouse_b200/bls.py) flattens SignatureSets into SoA buffers
//   sigs  n x 96 B  compressed G2            (AggregateSignature::serialize, generic_aggregate_signature.rs:153-160)
//   msgs  n x 32 B  signing roots            (generic_signature_set.rs:70)
//   pks   K x 96 B  uncompressed affine G1   (validator_pubkey_cache.rs:195-199 format), CSR offsets n+1
// and gets back the batch verdict.  All arithmetic runs on the device; there is no CPU fallback.
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <mutex>
#include <errno.h>
#include <sys/random.h>
#include <vector>
#include "bls/debug.cuh"
#include "bls/groups.cuh"
#include <condition_variable>
#include <thread>
#include "ctx.h"

namespace lhb200 {

using namespace bls;

static inline uint32_t cdiv(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

int32_t bls_init() { return LHB200_OK; }
void bls_shutdown();

}  // namespace lhb200

using namespace lhb200;

struct lhb200_pubkey_table {
    G1Mont* d_keys = nullptr;
    uint64_t capacity = 0, len = 0;
};

struct lhb200_bls_batch {
    // indexed mode: keys come from a device-resident table
    const lhb200_pubkey_table* table = nullptr;
    uint32_t* d_indices = nullptr;
    uint64_t cap_indices = 0;
    const uint32_t* in_indices = nullptr;
    uint32_t cap_sets = 0;
    uint64_t cap_keys = 0;
    uint32_t n = 0;
    // inputs (owned copies, or caller's device buffers)
    uint8_t *d_sigs = nullptr, *d_msgs = nullptr, *d_pks = nullptr;
    uint32_t* d_offsets = nullptr;
    uint64_t* d_rands = nullptr;
    const uint8_t *in_sigs = nullptr, *in_msgs = nullptr, *in_pks = nullptr;
    const uint32_t* in_offsets = nullptr;
    const uint64_t* in_rands = nullptr;
    // intermediates
    G2Jac* d_sigr = nullptr;      // r_i * sig_i
    G2Jac* d_sig_tmp[2] = {nullptr, nullptr};
    G1Proj3* d_p = nullptr;       // r_i * apk_i (projective evaluation point)
    G2Jac* d_h = nullptr;         // H(m_i), Jacobian
    Fp12* d_f = nullptr;          // Miller loop values
    Fp12* d_f_tmp[2] = {nullptr, nullptr};
    Fp12* d_flast = nullptr;
    Fp12* d_gt = nullptr;
    uint8_t* d_status = nullptr;
    uint32_t* d_fail = nullptr;
    uint8_t* d_ok = nullptr;
    uint8_t* h_res = nullptr;     // pinned: ok + status
    cudaStream_t s_main = nullptr;   // the stream lhb200_verify_signature_sets drives this handle on (one per handle)
    cudaStream_t s2 = nullptr, s3 = nullptr;
    cudaEvent_t e_h2c = nullptr, e_sig = nullptr;
    cudaEvent_t e_fork = nullptr, e_join = nullptr;
    cudaEvent_t e_k0 = nullptr, e_k1 = nullptr;  // around the dominant kernel (k_miller_multi), for the roofline
    cudaEvent_t e_done = nullptr;                // cudaEventBlockingSync: the host wait of long steps
    uint64_t launches_last = 0;
    // cooperative Miller kernel (bls/miller_coop.cuh): parking area for T / Q between rounds, the -g1 argument
    uint32_t* d_mc_scratch = nullptr;
    size_t mc_scratch_words = 0;
    G1Proj3* d_neg_g1 = nullptr;
    const G2Jac* d_sig_sum = nullptr;
    // small / medium batches: slice sums of the key lists (k_pk_partial -> k_pk_combine), PK_SLICES per set
    G1Jac* d_pk_part = nullptr;
    uint8_t* d_pk_part_bad = nullptr;
    // streamed key upload (lhb200_bls_batch_upload_async): the key copy is cut into chunks of whole sets on its own
    // stream; k_pk_aggregate runs per chunk as it lands while the signature / hash-to-curve kernels already compute
    static constexpr int MAX_CHUNKS = 16;
    static constexpr int N_PK_STREAMS = 4;
    cudaStream_t s_pk[N_PK_STREAMS] = {};    // high priority: chunk c is copied AND aggregated on s_pk[c % 4]
    cudaEvent_t e_pk[N_PK_STREAMS] = {};
    cudaEvent_t e_small = nullptr, e_copy_free = nullptr;
    uint32_t chunk_lo[MAX_CHUNKS + 1] = {};  // set ranges
    uint64_t chunk_key[MAX_CHUNKS + 1] = {}; // key ranges
    const uint8_t* h_pks = nullptr;          // caller's host keys (valid until result)
    int n_chunks = 0;                        // 0: inputs already complete on the device
    std::vector<uint64_t> rbuf;              // scalars drawn by the library (must outlive the async copy)
    // grouped verification (lhb200_verify_signature_set_groups): set for the duration of one grouped call; its buffers
    // are allocated on the first grouped call, so a handle that only runs plain verifications never holds them
    const groups::Plan* grp = nullptr;
    uint32_t* d_gwords = nullptr;            // the plan's tables (groups.cuh)
    Fp12* d_pf = nullptr;                    // one Miller value per pair: n sets, then one (-g1, sum r sig) per group
    G2Jac* d_gsum[2] = {nullptr, nullptr};   // levels of the segmented signature sums
    Fp12* d_gfold[2] = {nullptr, nullptr};   // levels of the segmented Miller products
    uint8_t* d_gok = nullptr;                // per-group verdicts
    uint64_t cap_gwords = 0, cap_pf = 0, cap_gsum[2] = {}, cap_gfold[2] = {}, cap_gok = 0;
};

static void batch_free(lhb200_bls_batch* b) {
    if (!b) return;
    if (b->d_indices) cudaFree(b->d_indices);
    void* ptrs[] = {b->d_sigs, b->d_msgs, b->d_pks, b->d_offsets, b->d_rands, b->d_sigr, b->d_sig_tmp[0],
                    b->d_sig_tmp[1], b->d_p, b->d_h, b->d_f, b->d_f_tmp[0], b->d_f_tmp[1], b->d_flast, b->d_gt,
                    b->d_status, b->d_fail, b->d_ok, b->d_mc_scratch, b->d_neg_g1, b->d_pk_part, b->d_pk_part_bad,
                    b->d_gwords, b->d_pf, b->d_gsum[0], b->d_gsum[1], b->d_gfold[0], b->d_gfold[1], b->d_gok};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (b->h_res) cudaFreeHost(b->h_res);
    if (b->s_main) cudaStreamDestroy(b->s_main);
    if (b->s2) cudaStreamDestroy(b->s2);
    if (b->s3) cudaStreamDestroy(b->s3);
    if (b->e_h2c) cudaEventDestroy(b->e_h2c);
    if (b->e_sig) cudaEventDestroy(b->e_sig);
    if (b->e_fork) cudaEventDestroy(b->e_fork);
    if (b->e_join) cudaEventDestroy(b->e_join);
    if (b->e_k0) cudaEventDestroy(b->e_k0);
    if (b->e_k1) cudaEventDestroy(b->e_k1);
    if (b->e_done) cudaEventDestroy(b->e_done);
    for (cudaStream_t st : b->s_pk)
        if (st) cudaStreamDestroy(st);
    for (cudaEvent_t e : b->e_pk)
        if (e) cudaEventDestroy(e);
    if (b->e_small) cudaEventDestroy(b->e_small);
    if (b->e_copy_free) cudaEventDestroy(b->e_copy_free);
    delete b;
}

constexpr uint32_t REDUCE_CHUNK = 8;
// latency modes of the per-set stages (batches that do not fill the GPU): slice-parallel key sums, two threads per hash
constexpr uint32_t PK_SPLIT_MAX_SETS = 8192;
constexpr uint32_t HASH_PAIR_MAX_SETS = 4096;    // (measured: 10 000 sets 16.4 ms with the plain kernel, 17.6 ms with the paired one)
constexpr uint32_t FINAL_WARP_TAIL = 160;             // Miller block products k_final_warp takes directly (one per SM + slack)
constexpr uint32_t BLOCKING_WAIT_MIN_SETS = 16384;   // lhb200_bls_batch_result: blocking wait for steps of >= ~15 ms

// ---- pool of batch handles behind lhb200_verify_signature_sets -------------------------------------------------
namespace {
// ---------------------------------------------------------------------------------------------------------
// Pageable key buffers (what a Rust Vec is).  cudaMemcpyAsync from pageable memory is staged by the driver through its
// own bounce buffer on the calling thread (~8.5 GB/s here: 145 ms for the 1.24 GB of a 100 k-set batch against 85 ms
// from pinned memory).  For big pageable key buffers the library stages them itself: a ring of pinned blocks filled by
// a few copy threads (memcpy scales with threads, the DMA engine reads pinned memory at link speed) and drained by
// cudaMemcpyAsync on the chunk's stream, so the CPU copy of block i + 1 overlaps the DMA of block i.
constexpr size_t STAGE_BLOCK = 16u << 20;
constexpr int STAGE_SLOTS = 4, STAGE_THREADS = 4;
constexpr uint64_t STAGE_MIN_BYTES = 64ull << 20;   // below this the driver's own staging is as good
struct KeyStager {
    uint8_t* slot[STAGE_SLOTS] = {};
    cudaEvent_t free_ev[STAGE_SLOTS] = {};
    bool used[STAGE_SLOTS] = {};
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    const uint8_t* src = nullptr;
    uint8_t* dst = nullptr;
    size_t bytes = 0;
    uint64_t generation = 0;
    int pending = 0;
    bool quit = false, ok = false;
    uint64_t next = 0;

    bool init() {
        if (ok) return true;
        for (int i = 0; i < STAGE_SLOTS; i++) {
            if (cudaHostAlloc(reinterpret_cast<void**>(&slot[i]), STAGE_BLOCK, cudaHostAllocDefault) != cudaSuccess ||
                cudaEventCreateWithFlags(&free_ev[i], cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) {
                cudaGetLastError();
                return false;
            }
        }
        for (int t = 0; t < STAGE_THREADS; t++) workers.emplace_back([this, t] { run(t); });
        ok = true;
        return true;
    }
    void run(int t) {
        uint64_t seen = 0;
        for (;;) {
            std::unique_lock<std::mutex> lk(mu);
            cv_work.wait(lk, [&] { return quit || generation != seen; });
            if (quit) return;
            seen = generation;
            const uint8_t* s_ = src; uint8_t* d_ = dst; const size_t n = bytes;
            lk.unlock();
            const size_t per = (n + STAGE_THREADS - 1) / STAGE_THREADS, lo = std::min(n, per * t), hi = std::min(n, lo + per);
            if (hi > lo) memcpy(d_ + lo, s_ + lo, hi - lo);
            lk.lock();
            if (--pending == 0) cv_done.notify_one();
        }
    }
    void parallel_copy(uint8_t* d_, const uint8_t* s_, size_t n) {
        std::unique_lock<std::mutex> lk(mu);
        src = s_; dst = d_; bytes = n; pending = STAGE_THREADS; generation++;
        cv_work.notify_all();
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    // host -> device copy of `n` bytes on `st`, staged block by block; returns when the LAST block has been queued
    cudaError_t copy(uint8_t* d_dev, const uint8_t* h_src, size_t n, cudaStream_t st) {
        for (size_t off = 0; off < n; off += STAGE_BLOCK) {
            const int k = (int)(next++ % STAGE_SLOTS);
            if (used[k]) {
                cudaError_t e = cudaEventSynchronize(free_ev[k]);   // the DMA that read this block has finished
                if (e != cudaSuccess) return e;
            }
            const size_t len = std::min(STAGE_BLOCK, n - off);
            parallel_copy(slot[k], h_src + off, len);
            cudaError_t e = cudaMemcpyAsync(d_dev + off, slot[k], len, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaEventRecord(free_ev[k], st);
            if (e != cudaSuccess) return e;
            used[k] = true;
        }
        return cudaSuccess;
    }
    void shutdown() {
        if (!ok) return;
        { std::lock_guard<std::mutex> g(mu); quit = true; }
        cv_work.notify_all();
        for (std::thread& w : workers) w.join();
        workers.clear();
        for (int i = 0; i < STAGE_SLOTS; i++) {
            if (free_ev[i]) cudaEventDestroy(free_ev[i]);
            if (slot[i]) cudaFreeHost(slot[i]);
            free_ev[i] = nullptr; slot[i] = nullptr; used[i] = false;
        }
        quit = false; ok = false;
    }
};
// heap-allocated and never destroyed: its worker threads must not meet a static destructor at process exit
// (lhb200_shutdown joins them and frees the ring)
KeyStager& g_stager = *new KeyStager;
std::mutex g_stager_use;   // one staged upload at a time (the ring is shared); concurrent big pageable uploads queue here

static bool host_pointer_is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

std::mutex g_pool_mu;
std::vector<lhb200_bls_batch*> g_pool_free;
constexpr size_t POOL_MAX_IDLE = 64;   // idle handles kept (a 64-set handle is ~0.5 MB of device memory)

lhb200_bls_batch* pool_acquire(uint32_t n_sets, uint64_t n_keys) {
    lhb200_bls_batch* b = nullptr;
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        // best fit: the smallest idle handle that is large enough
        size_t best = SIZE_MAX;
        for (size_t i = 0; i < g_pool_free.size(); i++) {
            lhb200_bls_batch* c = g_pool_free[i];
            if (c->cap_sets >= n_sets && c->cap_keys >= n_keys &&
                (best == SIZE_MAX || c->cap_keys < g_pool_free[best]->cap_keys)) best = i;
        }
        if (best != SIZE_MAX) {
            b = g_pool_free[best];
            g_pool_free.erase(g_pool_free.begin() + best);
        } else if (g_pool_free.size() >= POOL_MAX_IDLE) {   // recycle the oldest handle's slot
            lhb200_bls_batch* victim = g_pool_free.front();
            g_pool_free.erase(g_pool_free.begin());
            cudaStreamSynchronize(victim->s_main);
            batch_free(victim);
        }
    }
    if (b) return b;
    const uint32_t cap_sets = std::max<uint32_t>(n_sets + n_sets / 4, 256);
    const uint64_t cap_keys = std::max<uint64_t>(n_keys + n_keys / 4, 4096);
    if (lhb200_bls_batch_create(cap_sets, cap_keys, &b) != LHB200_OK) return nullptr;
    return b;
}
void pool_release(lhb200_bls_batch* b) {
    std::lock_guard<std::mutex> g(g_pool_mu);
    g_pool_free.push_back(b);
}
}  // namespace
namespace lhb200 {
void bls_shutdown() {
    g_stager.shutdown();
    std::lock_guard<std::mutex> g(g_pool_mu);
    for (lhb200_bls_batch* b : g_pool_free) batch_free(b);
    g_pool_free.clear();
}
}  // namespace lhb200

// ---- grouped verification (lhb200_verify_signature_set_groups) -------------------------------------------------------
// The per-set stages run as in a plain call; from the sum of r sig on, every group is its own batch:
//   s2: k_g2_sum_seg_warp levels -> one sum r sig per group
//   s:  k_miller_warp_pairs      -> one Miller value per pair (n sets + one (-g1, sum) pair per group)
//       k_fp12_reduce_seg levels -> at most groups::FOLD_MAX values per group (only for groups larger than that)
//       k_final_groups_warp      -> one warp per group: fold, final exponentiation, ok[g]
template <class T>
static cudaError_t grow(T*& p, uint64_t& cap, uint64_t need) {
    if (need <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    need += need / 4;
    const cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), need * sizeof(T));
    if (e == cudaSuccess) cap = need;
    return e;
}

// Buffers of a grouped call of n sets on an idle handle.
static int32_t group_reserve(lhb200_bls_batch* b, const groups::Plan& gp, uint32_t n) {
    const uint32_t G = gp.n_groups;
    LHB_CUDA(grow(b->d_gwords, b->cap_gwords, gp.words.size()));
    LHB_CUDA(grow(b->d_pf, b->cap_pf, (uint64_t)n + G));
    LHB_CUDA(grow(b->d_gok, b->cap_gok, G));
    for (int k = 0; k < 2; k++) {
        LHB_CUDA(grow(b->d_gsum[k], b->cap_gsum[k], gp.sum.max_out));
        LHB_CUDA(grow(b->d_gfold[k], b->cap_gfold[k], gp.fold.max_out));
    }
    return LHB200_OK;
}

// Everything after the per-set stages of a grouped call (called by lhb200_bls_batch_verify_enqueue on stream s, once
// the key sums, hashes and statuses are in place).
static int32_t enqueue_group_tail(lhb200_bls_batch* b, cudaStream_t s, uint32_t n, uint64_t launches) {
    const groups::Plan& gp = *b->grp;
    const uint32_t G = gp.n_groups, n_pairs = n + G;
    static const bool attr_ok = [] {
        return cudaFuncSetAttribute(mw::k_miller_warp_pairs, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)mw::smem_bytes(mc::MC_WARPS)) == cudaSuccess &&
               cudaFuncSetAttribute(fe::k_final_groups_warp, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)fe::groups_smem_bytes()) == cudaSuccess;
    }();
    if (!attr_ok) { set_error("grouped verification kernels: cannot reserve shared memory"); return LHB200_ECUDA; }
    // four warps per block (one per scheduler) while the pairs are few, eight above (as k_miller_warp)
    const uint32_t wpb = n_pairs <= 4 * COOP_TAIL ? 4 : mc::MC_WARPS;
    LHB_CUDA(cudaStreamWaitEvent(s, b->e_join, 0));   // the group sums
    LHB_CUDA(cudaEventRecord(b->e_k0, s));
    mw::k_miller_warp_pairs<<<cdiv(n_pairs, wpb), 32 * wpb, mw::smem_bytes((int)wpb), s>>>(b->d_p, b->d_h, b->d_status, n,
                                                                                            b->d_sig_sum, G, b->d_neg_g1, b->d_pf);
    LHB_CUDA(cudaEventRecord(b->e_k1, s));
    launches++;
    const Fp12* cur = b->d_pf;
    for (size_t l = 0; l < gp.fold.n_out.size(); l++) {
        const uint32_t mo = gp.fold.n_out[l];
        k_fp12_reduce_seg<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, s>>>(cur, b->d_gwords + gp.fold.at[l], mo, b->d_gfold[l & 1]);
        launches++;
        cur = b->d_gfold[l & 1];
    }
    fe::k_final_groups_warp<<<cdiv(G, fe::FG_WARPS), 32 * fe::FG_WARPS, fe::groups_smem_bytes(), s>>>(
        cur, b->d_gwords + gp.val_off_at, b->d_pf + n, b->d_status, b->d_gwords, G, b->d_gok);
    launches++;
    LHB_CUDA(cudaGetLastError());
    count_launch(launches);
    b->launches_last = launches;
    return LHB200_OK;
}

extern "C" {

int32_t lhb200_bls_batch_create(uint32_t max_sets, uint64_t max_keys, lhb200_bls_batch** out) {
    LHB_REQUIRE_READY();
    if (!out || max_sets == 0) { set_error("bls_batch_create: bad arguments"); return LHB200_EINVAL; }
    lhb200_bls_batch* b = new lhb200_bls_batch();
    b->cap_sets = max_sets;
    b->cap_keys = max_keys;
    // sum-tree buffers: sized for the narrowest chunk in use (4 points per warp in latency mode, REDUCE_CHUNK otherwise)
    const uint64_t n = max_sets, n1 = cdiv(n, 4) + 1, n2 = cdiv(n1, 4) + 1;
    // Miller values: one per set (old kernels) or 5 per warp of the cooperative kernel (<= ceil((n+1)/6) + 40 warps)
    const uint64_t nf = std::max<uint64_t>(n, (cdiv(n + 1, 6) + 48) * 5), nf1 = cdiv(nf, REDUCE_CHUNK) + 1,
                   nf2 = cdiv(nf1, REDUCE_CHUNK) + 1;
#define ALLOC(p, bytes)                                                         \
    do {                                                                        \
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&(p)), (bytes));    \
        if (e != cudaSuccess) { batch_free(b); return cuda_fail(e, "cudaMalloc(" #p ")"); } \
    } while (0)
    ALLOC(b->d_sigs, n * 96 + 16);
    ALLOC(b->d_msgs, n * 32 + 16);
    ALLOC(b->d_pks, std::max<uint64_t>(max_keys, 1) * 96 + 16);
    ALLOC(b->d_offsets, (n + 1) * 4);
    ALLOC(b->d_rands, n * 8);
    ALLOC(b->d_sigr, n * sizeof(G2Jac));
    ALLOC(b->d_sig_tmp[0], n1 * sizeof(G2Jac));
    ALLOC(b->d_sig_tmp[1], n2 * sizeof(G2Jac));
    ALLOC(b->d_p, n * sizeof(G1Proj3));
    ALLOC(b->d_h, n * sizeof(G2Jac));
    ALLOC(b->d_f, nf * sizeof(Fp12));
    ALLOC(b->d_f_tmp[0], nf1 * sizeof(Fp12));
    ALLOC(b->d_f_tmp[1], nf2 * sizeof(Fp12));
    ALLOC(b->d_flast, sizeof(Fp12));
    ALLOC(b->d_gt, sizeof(Fp12));
    ALLOC(b->d_status, n);
    ALLOC(b->d_fail, 4);
    ALLOC(b->d_ok, 4);
    ALLOC(b->d_neg_g1, sizeof(G1Proj3));
    ALLOC(b->d_pk_part, std::min<uint64_t>(n, PK_SPLIT_MAX_SETS) * PK_SLICES * sizeof(G1Jac));
    ALLOC(b->d_pk_part_bad, std::min<uint64_t>(n, PK_SPLIT_MAX_SETS) * PK_SLICES);
#undef ALLOC
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&b->h_res), n + 64 + sizeof(Fp12), cudaHostAllocDefault);
    if (e != cudaSuccess) { batch_free(b); return cuda_fail(e, "cudaHostAlloc(result)"); }
    if ((e = cudaStreamCreateWithFlags(&b->s_main, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&b->s2, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&b->s3, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_h2c, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_sig, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_fork, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_join, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreate(&b->e_k0)) != cudaSuccess || (e = cudaEventCreate(&b->e_k1)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_done, cudaEventBlockingSync | cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_small, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->e_copy_free, cudaEventDisableTiming)) != cudaSuccess) {
        batch_free(b);
        return cuda_fail(e, "stream/event create");
    }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);  // the key chunks must not queue behind the 1563-CTA kernels
    for (int j = 0; j < lhb200_bls_batch::N_PK_STREAMS; j++)
        if ((e = cudaStreamCreateWithPriority(&b->s_pk[j], cudaStreamNonBlocking, prio_hi)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&b->e_pk[j], cudaEventDisableTiming)) != cudaSuccess) {
            batch_free(b);
            return cuda_fail(e, "stream create");
        }
    k_init_neg_g1<<<1, 32, 0, b->s_main>>>(b->d_neg_g1);
    if ((e = cudaStreamSynchronize(b->s_main)) != cudaSuccess) { batch_free(b); return cuda_fail(e, "k_init_neg_g1"); }
    *out = b;
    return LHB200_OK;
}

int32_t lhb200_bls_batch_destroy(lhb200_bls_batch* b) {
    if (ctx().ready) cudaDeviceSynchronize();
    batch_free(b);
    return LHB200_OK;
}

// ---- blinding scalars (blst.rs:46-68: `rand::thread_rng()`, a ChaCha CSPRNG seeded from the OS) ----------------
// Same construction: a ChaCha20 keystream (RFC 8439 block function) keyed with 256 bits from getrandom(2) per thread,
// re-keyed every 2^20 blocks; every 64-bit word is used as one scalar, zeros are skipped (blst.rs:60-64).
namespace {
struct ChaChaRng {
    uint32_t key[8];
    uint32_t nonce[3];
    uint32_t counter = 0;
    bool keyed = false;
    uint64_t buf[8];
    int have = 0;
    static inline uint32_t rotl(uint32_t v, int c) { return (v << c) | (v >> (32 - c)); }
    static inline void qr(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
        a += b; d ^= a; d = rotl(d, 16);
        c += d; b ^= c; b = rotl(b, 12);
        a += b; d ^= a; d = rotl(d, 8);
        c += d; b ^= c; b = rotl(b, 7);
    }
    bool rekey() {
        uint8_t seed[44];
        size_t got = 0;
        while (got < sizeof seed) {
            const ssize_t k = getrandom(seed + got, sizeof seed - got, 0);
            if (k < 0) { if (errno == EINTR) continue; return false; }
            got += (size_t)k;
        }
        memcpy(key, seed, 32);
        memcpy(nonce, seed + 32, 12);
        counter = 0;
        keyed = true;
        return true;
    }
    bool refill() {
        if (!keyed || counter >= (1u << 20)) { if (!rekey()) return false; }
        uint32_t st[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u, key[0], key[1], key[2], key[3],
                           key[4], key[5], key[6], key[7], counter, nonce[0], nonce[1], nonce[2]};
        uint32_t x[16];
        memcpy(x, st, sizeof x);
        for (int i = 0; i < 10; i++) {
            qr(x[0], x[4], x[8], x[12]); qr(x[1], x[5], x[9], x[13]); qr(x[2], x[6], x[10], x[14]); qr(x[3], x[7], x[11], x[15]);
            qr(x[0], x[5], x[10], x[15]); qr(x[1], x[6], x[11], x[12]); qr(x[2], x[7], x[8], x[13]); qr(x[3], x[4], x[9], x[14]);
        }
        for (int i = 0; i < 16; i++) x[i] += st[i];
        memcpy(buf, x, sizeof buf);
        counter++;
        have = 8;
        return true;
    }
    bool next(uint64_t& v) {
        do {
            if (have == 0 && !refill()) return false;
            v = buf[--have];
        } while (v == 0);
        return true;
    }
};
}  // namespace
static bool gen_rands(uint64_t* r, uint32_t n) {
    static thread_local ChaChaRng rng;
    for (uint32_t i = 0; i < n; i++)
        if (!rng.next(r[i])) return false;
    return true;
}
// Test hook: n scalars from the generator above (statistical / distinctness tests without a device).
extern "C" LHB200_API int32_t lhb200_debug_rand_scalars(uint64_t* out, uint32_t n) {
    if (!out) return LHB200_EINVAL;
    return gen_rands(out, n) ? LHB200_OK : LHB200_ECUDA;
}

// Copy host inputs into the batch's device buffers.  rands == NULL: drawn here.
int32_t lhb200_bls_batch_upload(lhb200_bls_batch* b, const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets) {
    LHB_REQUIRE_READY();
    if (!b || n_sets == 0 || n_sets > b->cap_sets || !sigs || !msgs || !pk_offsets) {
        set_error("bls_batch_upload: bad arguments");
        return LHB200_EINVAL;
    }
    const uint64_t n_keys = pk_offsets[n_sets];
    if (n_keys > b->cap_keys || (n_keys && !pks)) { set_error("bls_batch_upload: key buffer too small"); return LHB200_EINVAL; }
    for (uint32_t i = 0; i < n_sets; i++)
        if (pk_offsets[i] > pk_offsets[i + 1]) { set_error("bls_batch_upload: offsets not monotone"); return LHB200_EINVAL; }
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    cudaStream_t s = c.stream;
    std::vector<uint64_t> rbuf;
    if (!rands) {
        rbuf.resize(n_sets);
        if (!gen_rands(rbuf.data(), n_sets)) { set_error("getrandom(2) failed"); return LHB200_ECUDA; }
        rands = rbuf.data();
    } else {
        for (uint32_t i = 0; i < n_sets; i++)
            if (rands[i] == 0) { set_error("bls_batch_upload: zero random scalar"); return LHB200_EINVAL; }
    }
    LHB_CUDA(cudaMemcpyAsync(b->d_sigs, sigs, (size_t)n_sets * 96, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_msgs, msgs, (size_t)n_sets * 32, cudaMemcpyHostToDevice, s));
    if (n_keys) LHB_CUDA(cudaMemcpyAsync(b->d_pks, pks, (size_t)n_keys * 96, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_offsets, pk_offsets, (size_t)(n_sets + 1) * 4, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_rands, rands, (size_t)n_sets * 8, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaStreamSynchronize(s));  // rbuf / caller buffers may go away
    b->n = n_sets;
    b->n_chunks = 0;
    b->in_sigs = b->d_sigs; b->in_msgs = b->d_msgs; b->in_pks = b->d_pks;
    b->in_offsets = b->d_offsets; b->in_rands = b->d_rands;
    b->table = nullptr;
    return LHB200_OK;
}

// Streamed form of lhb200_bls_batch_upload: queues the small arrays and BINDS the host key buffer; the key chunks are
// copied by lhb200_bls_batch_verify_enqueue, interleaved with their aggregation kernels.  The host buffers must stay
// valid and unchanged until lhb200_bls_batch_result returns.  The small arrays go first; the keys (96 B x K, 1.2 GB at
// 100 k x 128) follow in chunks of whole sets on a copy stream, and lhb200_bls_batch_verify_enqueue aggregates each
// chunk as it lands while k_sig_prepare / k_hash_to_g2 already run — the host link hides behind the ALU-bound kernels.
int32_t lhb200_bls_batch_upload_async(lhb200_bls_batch* b, const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                      const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets, void* stream) {
    LHB_REQUIRE_READY();
    if (!b || n_sets == 0 || n_sets > b->cap_sets || !sigs || !msgs || !pk_offsets) {
        set_error("bls_batch_upload_async: bad arguments");
        return LHB200_EINVAL;
    }
    const uint64_t n_keys = pk_offsets[n_sets];
    if (n_keys > b->cap_keys || (n_keys && !pks)) { set_error("bls_batch_upload_async: key buffer too small"); return LHB200_EINVAL; }
    for (uint32_t i = 0; i < n_sets; i++)
        if (pk_offsets[i] > pk_offsets[i + 1]) { set_error("bls_batch_upload_async: offsets not monotone"); return LHB200_EINVAL; }
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx().stream;
    if (!rands) {
        b->rbuf.resize(n_sets);
        if (!gen_rands(b->rbuf.data(), n_sets)) { set_error("getrandom(2) failed"); return LHB200_ECUDA; }
        rands = b->rbuf.data();
    } else {
        for (uint32_t i = 0; i < n_sets; i++)
            if (rands[i] == 0) { set_error("bls_batch_upload_async: zero random scalar"); return LHB200_EINVAL; }
    }
    // the previous verify on this batch may still be reading d_pks: order the new copies behind it
    LHB_CUDA(cudaEventRecord(b->e_copy_free, s));
    for (cudaStream_t st : b->s_pk) LHB_CUDA(cudaStreamWaitEvent(st, b->e_copy_free, 0));
    LHB_CUDA(cudaMemcpyAsync(b->d_sigs, sigs, (size_t)n_sets * 96, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_msgs, msgs, (size_t)n_sets * 32, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_offsets, pk_offsets, (size_t)(n_sets + 1) * 4, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_rands, rands, (size_t)n_sets * 8, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaEventRecord(b->e_small, s));
    // chunks of whole sets, ~equal key counts
    int nc = (int)std::min<uint64_t>(lhb200_bls_batch::MAX_CHUNKS, std::max<uint64_t>(1, n_keys * 96 / (32u << 20)));
    nc = std::min<int>(nc, (int)n_sets);
    b->chunk_lo[0] = 0;
    uint32_t lo = 0;
    for (int c = 0; c < nc; c++) {
        uint32_t hi;
        if (c == nc - 1) hi = n_sets;
        else {
            const uint64_t target = n_keys * (uint64_t)(c + 1) / nc;
            hi = (uint32_t)(std::lower_bound(pk_offsets + lo, pk_offsets + n_sets + 1, target) - pk_offsets);
            hi = std::min<uint32_t>(std::max<uint32_t>(hi, lo), n_sets);
        }
        b->chunk_key[c] = pk_offsets[lo];
        b->chunk_key[c + 1] = pk_offsets[hi];
        b->chunk_lo[c + 1] = hi;
        lo = hi;
    }
    b->n_chunks = nc;
    b->h_pks = pks;
    b->n = n_sets;
    b->in_sigs = b->d_sigs; b->in_msgs = b->d_msgs; b->in_pks = b->d_pks;
    b->in_offsets = b->d_offsets; b->in_rands = b->d_rands;
    b->table = nullptr;
    return LHB200_OK;
}

// ---- device-resident pubkey table (SURVEY §8f-1; mirror of ValidatorPubkeyCache) ---------------------------
int32_t lhb200_pubkey_table_create(uint64_t capacity, lhb200_pubkey_table** out) {
    LHB_REQUIRE_READY();
    if (!out || capacity == 0) return LHB200_EINVAL;
    lhb200_pubkey_table* t = new lhb200_pubkey_table();
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&t->d_keys), capacity * sizeof(G1Mont));
    if (e != cudaSuccess) { delete t; return cuda_fail(e, "cudaMalloc(pubkey table)"); }
    t->capacity = capacity;
    *out = t;
    return LHB200_OK;
}
int32_t lhb200_pubkey_table_destroy(lhb200_pubkey_table* t) {
    if (!t) return LHB200_OK;
    if (ctx().ready) cudaDeviceSynchronize();
    if (t->d_keys) cudaFree(t->d_keys);
    delete t;
    return LHB200_OK;
}
uint64_t lhb200_pubkey_table_len(const lhb200_pubkey_table* t) { return t ? t->len : 0; }

// Append n validated keys (96-byte uncompressed, the validator_pubkey_cache.rs:195-199 format) at indices
// [len, len+n).  Malformed / off-curve / infinity entries make the call fail with LHB200_EDECODE (nothing appended).
int32_t lhb200_pubkey_table_append(lhb200_pubkey_table* t, const uint8_t* pks96, uint64_t n) {
    LHB_REQUIRE_READY();
    if (!t || (n && !pks96)) return LHB200_EINVAL;
    if (t->len + n > t->capacity) { set_error("pubkey table full"); return LHB200_EINVAL; }
    if (n == 0) return LHB200_OK;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch(n * 96 + 256));
    if (!d) return LHB200_ENOMEM;
    uint32_t* d_bad = reinterpret_cast<uint32_t*>(d + ((n * 96 + 15) / 16) * 16);
    LHB_CUDA(cudaMemcpyAsync(d, pks96, n * 96, cudaMemcpyHostToDevice, c.stream));
    LHB_CUDA(cudaMemsetAsync(d_bad, 0, 4, c.stream));
    k_table_import<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, (uint32_t)n, t->d_keys + t->len, d_bad);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    uint32_t bad = 0;
    LHB_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    if (bad) { set_error("%u of %llu keys are malformed, off-curve or at infinity", bad, (unsigned long long)n); return LHB200_EDECODE; }
    t->len += n;
    return LHB200_OK;
}

// Like lhb200_bls_batch_upload, but the signing keys are given as indices into a resident table
// (what signature_sets.rs:315-320 gathers from the pubkey cache): key_indices[K], CSR offsets as before.
int32_t lhb200_bls_batch_upload_indexed(lhb200_bls_batch* b, const lhb200_pubkey_table* table, const uint8_t* sigs,
                                        const uint8_t* msgs, const uint32_t* key_indices, const uint32_t* pk_offsets,
                                        const uint64_t* rands, uint32_t n_sets) {
    LHB_REQUIRE_READY();
    if (!b || !table || n_sets == 0 || n_sets > b->cap_sets || !sigs || !msgs || !pk_offsets) {
        set_error("bls_batch_upload_indexed: bad arguments");
        return LHB200_EINVAL;
    }
    const uint64_t n_keys = pk_offsets[n_sets];
    if (n_keys && !key_indices) return LHB200_EINVAL;
    for (uint32_t i = 0; i < n_sets; i++)
        if (pk_offsets[i] > pk_offsets[i + 1]) { set_error("bls_batch_upload_indexed: offsets not monotone"); return LHB200_EINVAL; }
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    cudaStream_t s = c.stream;
    if (n_keys > b->cap_indices) {
        if (b->d_indices) { cudaStreamSynchronize(s); cudaFree(b->d_indices); b->d_indices = nullptr; }
        LHB_CUDA(cudaMalloc(reinterpret_cast<void**>(&b->d_indices), std::max<uint64_t>(n_keys, 1) * 4));
        b->cap_indices = n_keys;
    }
    std::vector<uint64_t> rbuf;
    if (!rands) {
        rbuf.resize(n_sets);
        if (!gen_rands(rbuf.data(), n_sets)) { set_error("getrandom(2) failed"); return LHB200_ECUDA; }
        rands = rbuf.data();
    }
    else for (uint32_t i = 0; i < n_sets; i++) if (rands[i] == 0) { set_error("zero random scalar"); return LHB200_EINVAL; }
    LHB_CUDA(cudaMemcpyAsync(b->d_sigs, sigs, (size_t)n_sets * 96, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_msgs, msgs, (size_t)n_sets * 32, cudaMemcpyHostToDevice, s));
    if (n_keys) LHB_CUDA(cudaMemcpyAsync(b->d_indices, key_indices, (size_t)n_keys * 4, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_offsets, pk_offsets, (size_t)(n_sets + 1) * 4, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaMemcpyAsync(b->d_rands, rands, (size_t)n_sets * 8, cudaMemcpyHostToDevice, s));
    LHB_CUDA(cudaStreamSynchronize(s));
    b->n = n_sets;
    b->in_sigs = b->d_sigs; b->in_msgs = b->d_msgs; b->in_pks = nullptr;
    b->in_offsets = b->d_offsets; b->in_rands = b->d_rands; b->in_indices = b->d_indices;
    b->n_chunks = 0;
    b->table = table;
    return LHB200_OK;
}

// Use caller-owned device buffers (16-byte aligned) as the inputs: nothing is copied.
int32_t lhb200_bls_batch_set_device_inputs(lhb200_bls_batch* b, const void* d_sigs, const void* d_msgs,
                                           const void* d_pks, const void* d_offsets, const void* d_rands,
                                           uint32_t n_sets) {
    LHB_REQUIRE_READY();
    if (!b || n_sets == 0 || n_sets > b->cap_sets || !d_sigs || !d_msgs || !d_offsets || !d_rands ||
        ((uintptr_t)d_sigs & 15) || ((uintptr_t)d_msgs & 15) || ((uintptr_t)d_pks & 15)) {
        set_error("bls_batch_set_device_inputs: bad arguments (buffers must be 16-byte aligned)");
        return LHB200_EINVAL;
    }
    b->n = n_sets;
    b->in_sigs = static_cast<const uint8_t*>(d_sigs);
    b->in_msgs = static_cast<const uint8_t*>(d_msgs);
    b->in_pks = static_cast<const uint8_t*>(d_pks);
    b->in_offsets = static_cast<const uint32_t*>(d_offsets);
    b->in_rands = static_cast<const uint64_t*>(d_rands);
    b->n_chunks = 0;
    b->table = nullptr;
    return LHB200_OK;
}

int32_t lhb200_bls_batch_verify_enqueue(lhb200_bls_batch* b, void* stream) {
    LHB_REQUIRE_READY();
    if (!b || b->n == 0 || !b->in_sigs) { set_error("bls_batch_verify_enqueue: no inputs"); return LHB200_EINVAL; }
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx().stream;
    const uint32_t n = b->n;
    // Resident CTAs per SM are capped (grid-stride kernels): fewer threads keep their 1-4 KB stacks in L1/L2.
    // LHB_BLS_CTAS_PER_SM overrides (tuning knob; 0 = one CTA per BLS_BLOCK sets, i.e. no cap).
    static const int ctas_per_sm = [] { const char* e = getenv("LHB_BLS_CTAS_PER_SM"); return e ? atoi(e) : 12; }();
    static const int n_sm = [] { int v = 148; cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, ctx().device); return v; }();
    uint32_t grid = cdiv(n, BLS_BLOCK);
    if (ctas_per_sm > 0 && grid > (uint32_t)(n_sm * ctas_per_sm)) {
        const uint32_t max_thr = (uint32_t)(n_sm * ctas_per_sm) * BLS_BLOCK;
        const uint32_t per_thread = cdiv(n, max_thr);            // sets per thread, balanced across the grid
        grid = cdiv(n, (uint64_t)per_thread * BLS_BLOCK);
    }
    uint64_t launches = 0;
    // key ingest through the TMA unit (bulk async copies into a shared-memory ring); needs 16-byte aligned keys
    // Only for batches that fill the GPU by themselves: the ring needs a shared-memory carve-out, and an SM that is
    // running blocks of the (shared-memory-free, full-L1) k_sig_prepare / k_hash_to_g2 cannot take a block with a
    // different carve-out until it drains — on the 5 216-set block-import batch that serialised the three stages
    // (32.5 ms against 19.9 ms with the plain kernel, which also copes better with ragged 1 ... 512-key lists).
    // LHB_PK_TMA=0 / 1 forces the choice (tuning, tests).
    static const int pk_tma_env = [] { const char* e = getenv("LHB_PK_TMA"); return e ? atoi(e) : -1; }();
    const bool pk_tma_fit = b->in_pks && ((uintptr_t)b->in_pks & 15) == 0;
    const bool pk_tma = pk_tma_fit && (pk_tma_env < 0 ? n >= 4u * BLS_BLOCK * (uint32_t)n_sm : pk_tma_env != 0);
    if (b->n_chunks) LHB_CUDA(cudaStreamWaitEvent(s, b->e_small, 0));  // streamed upload: small arrays first
    LHB_CUDA(cudaMemsetAsync(b->d_status, 0, n, s));
    LHB_CUDA(cudaMemsetAsync(b->d_fail, 0, 4, s));
    LHB_CUDA(cudaMemsetAsync(b->d_ok, 0, 4, s));
    // Three independent per-set stages run concurrently (they matter for small batches, where each kernel is a
    // latency-bound handful of warps): s2 = signatures (+ their sum tree + the last Miller loop), s3 = hash_to_g2,
    // s = key aggregation; the Miller kernel joins s and s3, k_final joins s2.
    LHB_CUDA(cudaEventRecord(b->e_fork, s));
    LHB_CUDA(cudaStreamWaitEvent(b->s2, b->e_fork, 0));
    LHB_CUDA(cudaStreamWaitEvent(b->s3, b->e_fork, 0));
    // latency mode of the two G2 stages (bls/g2_warp.cuh): one warp per signature / message while the batch is small
    // enough for the warps of one wave (four per block, at most two blocks per SM)
    static const int g2_warp_env = [] { const char* e = getenv("LHB_G2_WARP"); return e ? atoi(e) : 1; }();
    const bool g2_warp = g2_warp_env && n <= 6u * (uint32_t)n_sm;   // measured crossover with the lane-per-set kernels: ~1 000 sets
    constexpr uint32_t GW_WPB = 4;
    const size_t gw_smem = gw::smem_bytes(GW_WPB);
    if (g2_warp) {   // working sets + a shared-memory copy of the phase tables: above the 48 KB default
        static const bool gw_attr_ok = [&] {
            return cudaFuncSetAttribute(gw::k_sig_prepare_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gw_smem) == cudaSuccess &&
                   cudaFuncSetAttribute(gw::k_hash_to_g2_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gw_smem) == cudaSuccess &&
                   cudaFuncSetAttribute(gw::k_g2_sum_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gw_smem) == cudaSuccess;
        }();
        if (!gw_attr_ok) { set_error("g2 warp kernels: cannot reserve %zu B of shared memory", gw_smem); return LHB200_ECUDA; }
    }
    if (g2_warp)
        gw::k_sig_prepare_warp<<<cdiv(n, GW_WPB), 32 * GW_WPB, gw_smem, b->s2>>>(b->in_sigs, b->in_rands, n, b->d_sigr,
                                                                               b->d_status, b->d_fail);
    else
        k_sig_prepare<<<grid, BLS_BLOCK, 0, b->s2>>>(b->in_sigs, b->in_rands, n, b->d_sigr, b->d_status, b->d_fail);
    launches++;
    LHB_CUDA(cudaEventRecord(b->e_sig, b->s2));
    if (b->grp) {
        // grouped: one sum r sig per group, segmented levels of four points per warp (no level when every group has one
        // set: the set's own point is the sum)
        const groups::Levels& L = b->grp->sum;
        const G2Jac* cur = b->d_sigr;
        if (!L.n_out.empty()) {
            static const bool seg_attr_ok = [&] {
                return cudaFuncSetAttribute(gw::k_g2_sum_seg_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gw_smem) == cudaSuccess;
            }();
            if (!seg_attr_ok) { set_error("k_g2_sum_seg_warp: cannot reserve %zu B of shared memory", gw_smem); return LHB200_ECUDA; }
        }
        for (size_t l = 0; l < L.n_out.size(); l++) {
            gw::k_g2_sum_seg_warp<<<cdiv(L.n_out[l], GW_WPB), 32 * GW_WPB, gw_smem, b->s2>>>(cur, b->d_gwords + L.at[l], L.n_out[l],
                                                                                          b->d_gsum[l & 1]);
            launches++;
            cur = b->d_gsum[l & 1];
        }
        b->d_sig_sum = cur;
        LHB_CUDA(cudaEventRecord(b->e_join, b->s2));
    } else {
        const G2Jac* cur = b->d_sigr;
        uint32_t m = n;
        int flip = 0;
        while (m > 1) {
            if (g2_warp) {   // latency mode: warp-wide additions, four points per warp and level
                constexpr uint32_t CH = 4;
                const uint32_t mo = cdiv(m, CH);
                gw::k_g2_sum_warp<<<cdiv(mo, GW_WPB), 32 * GW_WPB, gw_smem, b->s2>>>(cur, m, CH, b->d_sig_tmp[flip]);
                launches++;
                cur = b->d_sig_tmp[flip];
                flip ^= 1;
                m = mo;
                continue;
            }
            const uint32_t mo = cdiv(m, REDUCE_CHUNK);
            k_g2_reduce<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, b->s2>>>(cur, m, REDUCE_CHUNK, b->d_sig_tmp[flip]);
            launches++;
            cur = b->d_sig_tmp[flip];
            flip ^= 1;
            m = mo;
        }
        b->d_sig_sum = cur;
        static const int miller_coop_s2 = [] { const char* e = getenv("LHB_MILLER_COOP"); return e ? atoi(e) : 1; }();
        if (!miller_coop_s2) {
            k_last_miller<<<1, 32, 0, b->s2>>>(cur, b->d_flast);
            launches++;
        }
        LHB_CUDA(cudaEventRecord(b->e_join, b->s2));
    }
    if (g2_warp)
        gw::k_hash_to_g2_warp<<<cdiv(n, GW_WPB), 32 * GW_WPB, gw_smem, b->s3>>>(b->in_msgs, n, b->d_h);
    else if (n <= HASH_PAIR_MAX_SETS)   // latency mode: two threads per message (one SSWU map each)
        k_hash_to_g2_pair<<<cdiv(2 * n, BLS_BLOCK), BLS_BLOCK, 0, b->s3>>>(b->in_msgs, n, b->d_h);
    else
        k_hash_to_g2<<<grid, BLS_BLOCK, 0, b->s3>>>(b->in_msgs, n, b->d_h);
    launches++;
    LHB_CUDA(cudaEventRecord(b->e_h2c, b->s3));
    // explicit keys, sets [lo, lo + cnt): TMA ring for GPU-filling batches, slice-parallel sums for small and medium
    // ones (a 512-key list is 64 + 8 additions deep instead of 512), one thread per set in between
    auto launch_pk = [&](uint32_t lo, uint32_t cnt, cudaStream_t st) {
        if (pk_tma) {
            k_pk_aggregate_tma<<<cdiv(cnt, BLS_BLOCK), BLS_BLOCK, 0, st>>>(b->in_pks, b->in_offsets + lo, b->in_rands + lo, cnt,
                                                                          b->d_p + lo, b->d_status + lo, b->d_fail);
        } else if (n <= PK_SPLIT_MAX_SETS) {
            k_pk_partial<<<cdiv(cnt * PK_SLICES, BLS_BLOCK), BLS_BLOCK, 0, st>>>(
                b->in_pks, b->in_offsets + lo, cnt, b->d_pk_part + (size_t)lo * PK_SLICES, b->d_pk_part_bad + (size_t)lo * PK_SLICES);
            k_pk_combine<<<cdiv(cnt, BLS_BLOCK), BLS_BLOCK, 0, st>>>(
                b->d_pk_part + (size_t)lo * PK_SLICES, b->d_pk_part_bad + (size_t)lo * PK_SLICES, b->in_offsets + lo,
                b->in_rands + lo, cnt, b->d_p + lo, b->d_status + lo, b->d_fail);
            launches++;
        } else {
            k_pk_aggregate<<<std::min<uint32_t>(grid, cdiv(cnt, BLS_BLOCK)), BLS_BLOCK, 0, st>>>(
                b->in_pks, b->in_offsets + lo, b->in_rands + lo, cnt, b->d_p + lo, b->d_status + lo, b->d_fail);
        }
        launches++;
    };
    if (b->table) {
        launches++;
        k_pk_aggregate_indexed<<<grid, BLS_BLOCK, 0, s>>>(b->table->d_keys, (uint32_t)b->table->len, b->in_indices,
                                                         b->in_offsets, b->in_rands, n, b->d_p, b->d_status, b->d_fail);
    } else if (b->n_chunks) {
        // big pageable key buffers go through the library's pinned ring (see KeyStager)
        static const int stage_env = [] { const char* e = getenv("LHB_STAGE_PAGEABLE"); return e ? atoi(e) : 1; }();
        const uint64_t key_bytes = (b->chunk_key[b->n_chunks] - b->chunk_key[0]) * 96;
        std::unique_lock<std::mutex> stage_lock(g_stager_use, std::defer_lock);
        bool stage_keys = false;
        if (stage_env && key_bytes >= STAGE_MIN_BYTES && host_pointer_is_pageable(b->h_pks)) {
            stage_lock.lock();
            stage_keys = g_stager.init();
            if (!stage_keys) stage_lock.unlock();
        }
        // aggregate each chunk of sets on the (high-priority) stream that copies it, as soon as its keys have landed
        for (int j = 0; j < lhb200_bls_batch::N_PK_STREAMS; j++) LHB_CUDA(cudaStreamWaitEvent(b->s_pk[j], b->e_fork, 0));
        for (int c = 0; c < b->n_chunks; c++) {
            const uint32_t lo = b->chunk_lo[c], cnt = b->chunk_lo[c + 1] - lo;
            const uint64_t k0 = b->chunk_key[c], k1 = b->chunk_key[c + 1];
            if (k1 > k0) {
                if (stage_keys) {
                    LHB_CUDA(g_stager.copy(b->d_pks + k0 * 96, b->h_pks + k0 * 96, (k1 - k0) * 96,
                                           b->s_pk[c % lhb200_bls_batch::N_PK_STREAMS]));
                } else {
                    LHB_CUDA(cudaMemcpyAsync(b->d_pks + k0 * 96, b->h_pks + k0 * 96, (k1 - k0) * 96, cudaMemcpyHostToDevice,
                                             b->s_pk[c % lhb200_bls_batch::N_PK_STREAMS]));
                }
            }
            if (cnt == 0) continue;
            launch_pk(lo, cnt, b->s_pk[c % lhb200_bls_batch::N_PK_STREAMS]);
        }
        for (int j = 0; j < lhb200_bls_batch::N_PK_STREAMS; j++) {
            LHB_CUDA(cudaEventRecord(b->e_pk[j], b->s_pk[j]));
            LHB_CUDA(cudaStreamWaitEvent(s, b->e_pk[j], 0));
        }
    } else
        launch_pk(0, n, s);
    LHB_CUDA(cudaStreamWaitEvent(s, b->e_h2c, 0));
    LHB_CUDA(cudaStreamWaitEvent(s, b->e_sig, 0));    // the Miller kernel reads the status bytes k_sig_prepare may set
    if (b->grp) return enqueue_group_tail(b, s, n, launches);
    static const int miller_coop = [] { const char* e = getenv("LHB_MILLER_COOP"); return e ? atoi(e) : 1; }();
    const Fp12* cur = b->d_f;
    uint32_t n_tail = 0;
    const Fp12* f_last = b->d_flast;
    if (miller_coop) {
        // Cooperative shared-memory Miller loop over the n sets AND the (-g1, sum r sig) pair (bls/miller_coop.cuh):
        // one block of 8 independent warps per SM, 30 working lanes per warp, every lane runs `rounds` sets, six lanes
        // share one accumulator.  Small batches spread over more, emptier warps (latency), large ones fill 8 x n_sm.
        static const bool attr_ok = [] {
            return cudaFuncSetAttribute(mc::k_miller_coop, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)mc::mc_smem_bytes()) == cudaSuccess;
        }();
        if (!attr_ok) { set_error("k_miller_coop: cannot reserve %zu B of shared memory", mc::mc_smem_bytes()); return LHB200_ECUDA; }
        constexpr uint32_t LU = 30;
        const uint32_t n_total = n + 1;
        const uint32_t max_warps = (uint32_t)n_sm * mc::MC_WARPS;
        // Latency mode (bls/miller_warp.cuh): while every pair can have a warp of its own in one wave, a whole warp runs
        // one Miller loop at Fp granularity — 0.x ms instead of the 3.7 ms of a lane-per-set loop.  Four warps per block
        // (one per scheduler) up to 256 pairs, eight above; <= 64 block products go straight to k_final_coop.
        static const int miller_warp_env = [] { const char* e = getenv("LHB_MILLER_WARP"); return e ? atoi(e) : 1; }();
        if (miller_warp_env && n_total <= max_warps) {
            static const bool mw_attr_ok = [] {
                return cudaFuncSetAttribute(mw::k_miller_warp, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)mw::smem_bytes(mc::MC_WARPS)) == cudaSuccess;
            }();
            if (!mw_attr_ok) { set_error("k_miller_warp: cannot reserve shared memory"); return LHB200_ECUDA; }
            const uint32_t wpb = n_total <= 4 * COOP_TAIL ? 4 : mc::MC_WARPS;
            const uint32_t mgrid = cdiv(n_total, wpb);
            LHB_CUDA(cudaStreamWaitEvent(s, b->e_join, 0));   // sum r sig (and -g1) ready
            LHB_CUDA(cudaEventRecord(b->e_k0, s));
            mw::k_miller_warp<<<mgrid, 32 * wpb, mw::smem_bytes((int)wpb), s>>>(b->d_p, b->d_h, b->d_status, n,
                                                                                         b->d_sig_sum, b->d_neg_g1, b->d_f);
            LHB_CUDA(cudaEventRecord(b->e_k1, s));
            launches += 1;
            uint32_t m = mgrid;
            int flip = 0;
            while (m > COOP_TAIL) {
                const uint32_t mo = cdiv(m, REDUCE_CHUNK);
                k_fp12_reduce<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, s>>>(cur, m, REDUCE_CHUNK, b->d_f_tmp[flip]);
                launches++;
                cur = b->d_f_tmp[flip];
                flip ^= 1;
                m = mo;
            }
            n_tail = m;
            f_last = nullptr;
        } else {
        uint32_t spw = cdiv(n_total, max_warps);             // sets per warp
        spw = cdiv(spw, LU) * LU;                            // whole rounds
        uint32_t n_warps, mgrid;
        // Batches below one full round per warp.  A warp's five groups take one set each at no extra latency (SIMT), and
        // every further set of a group adds one serial sparse product per iteration (81 multiply units for a 1-set
        // group, 141 for a full one).  Small batches therefore use at least five sets per warp, at most 256 warps, four
        // per block (one per scheduler): <= 64 block products, which k_final_coop folds itself (no k_fp12_reduce level,
        // 0.55 ms of single-thread latency).  Above that: as few sets per warp as the 8 x n_sm warp budget allows.
        constexpr uint32_t FEW_WARPS = 4 * COOP_TAIL;
        if (n_total <= FEW_WARPS * LU) {
            spw = std::min<uint32_t>(LU, std::max<uint32_t>(5, cdiv(cdiv(n_total, FEW_WARPS), 5) * 5));
            n_warps = cdiv(n_total, spw);
            mgrid = cdiv(n_warps, 4);
        } else {
            if (n_total <= max_warps * LU) spw = std::max<uint32_t>(1, cdiv(n_total, max_warps));
            n_warps = cdiv(n_total, spw);
            // warps are dealt round-robin to blocks (gw = warp_in_block * grid + block): few warps spread over all SMs
            mgrid = std::max<uint32_t>(std::min<uint32_t>((uint32_t)n_sm, n_warps), cdiv(n_warps, mc::MC_WARPS));
        }
        const uint32_t rounds_cap = cdiv(spw, LU);
        const size_t need = (size_t)mgrid * mc::MC_WARPS * rounds_cap * 2 * mc::TWORDS * 32;
        if (need > b->mc_scratch_words) {
            LHB_CUDA(cudaStreamSynchronize(s));
            if (b->d_mc_scratch) cudaFree(b->d_mc_scratch);
            b->d_mc_scratch = nullptr;
            LHB_CUDA(cudaMalloc(reinterpret_cast<void**>(&b->d_mc_scratch), need * 4));
            b->mc_scratch_words = need;
        }
        LHB_CUDA(cudaStreamWaitEvent(s, b->e_join, 0));   // sum r sig (and -g1) ready
        LHB_CUDA(cudaEventRecord(b->e_k0, s));
        mc::k_miller_coop<<<mgrid, 32 * mc::MC_WARPS, mc::mc_smem_bytes(), s>>>(b->d_p, b->d_h, b->d_status, n, b->d_sig_sum,
                                                                                b->d_neg_g1, spw, b->d_mc_scratch, b->d_f);
        LHB_CUDA(cudaEventRecord(b->e_k1, s));
        launches += 1;
        uint32_t m = mgrid;   // the kernel multiplies groups and warps together: one value per block
        int flip = 0;
        // k_final_warp folds the block products itself (8 warps x ~19 products of 7 us): no single-thread product level
        static const int fw_env = [] { const char* e = getenv("LHB_FINAL_WARP"); return e ? atoi(e) : 1; }();
        const uint32_t tail_max = fw_env ? FINAL_WARP_TAIL : COOP_TAIL;
        while (m > tail_max) {
            const uint32_t mo = cdiv(m, REDUCE_CHUNK);
            k_fp12_reduce<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, s>>>(cur, m, REDUCE_CHUNK, b->d_f_tmp[flip]);
            launches++;
            cur = b->d_f_tmp[flip];
            flip ^= 1;
            m = mo;
        }
        n_tail = m;
        f_last = nullptr;
        }
    } else {
    LHB_CUDA(cudaEventRecord(b->e_k0, s));
    // Sets per thread: k = ceil(n / resident threads) (<= MILLER_KMAX) share their Fp12 squarings in one thread, so a
    // 100 k batch is ONE wave of 3-set groups instead of three waves of single Miller loops.  LHB_MILLER_K overrides.
    static const int miller_occ = [] {
        int v = 4;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_miller_multi, MILLER_BLOCK, 0);
        return std::max(v, 1);
    }();
    static const int miller_k_env = [] { const char* e = getenv("LHB_MILLER_K"); return e ? atoi(e) : 0; }();
    const uint32_t resident = (uint32_t)(n_sm * miller_occ) * MILLER_BLOCK;
    uint32_t mk = miller_k_env > 0 ? (uint32_t)miller_k_env : cdiv(n, resident);
    mk = std::min<uint32_t>(std::max<uint32_t>(mk, 1), MILLER_KMAX);
    const uint32_t n_groups = cdiv(n, mk);
    k_miller_multi<<<std::min<uint32_t>(cdiv(n_groups, MILLER_BLOCK), (uint32_t)(n_sm * miller_occ)), MILLER_BLOCK, 0, s>>>(
        b->d_p, b->d_h, b->d_status, n, mk, n_groups, b->d_f);
    LHB_CUDA(cudaEventRecord(b->e_k1, s));
    launches += 1;
    {
        uint32_t m = n_groups;
        int flip = 0;
        while (m > COOP_TAIL) {   // the last <= 16 values are folded cooperatively inside k_final_coop
            const uint32_t mo = cdiv(m, REDUCE_CHUNK);
            k_fp12_reduce<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, s>>>(cur, m, REDUCE_CHUNK, b->d_f_tmp[flip]);
            launches++;
            cur = b->d_f_tmp[flip];
            flip ^= 1;
            m = mo;
        }
        n_tail = m;
    }
    LHB_CUDA(cudaStreamWaitEvent(s, b->e_join, 0));
    }
    static const int final_warp_env = [] { const char* e = getenv("LHB_FINAL_WARP"); return e ? atoi(e) : 1; }();
    if (final_warp_env && !f_last) {   // phase-interpreter tail (bls/fe_warp.cuh)
        static const bool fe_attr_ok = [] {
            return cudaFuncSetAttribute(fe::k_final_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fe::smem_bytes()) == cudaSuccess;
        }();
        if (!fe_attr_ok) { set_error("k_final_warp: cannot reserve shared memory"); return LHB200_ECUDA; }
        fe::k_final_warp<<<1, 32 * fe::FE_WARPS, fe::smem_bytes(), s>>>(cur, n_tail, b->d_fail, b->d_ok, b->d_gt);
    } else
        k_final_coop<<<1, COOP_THREADS, sizeof(CoopFinalSmem), s>>>(cur, n_tail, f_last, b->d_fail, b->d_ok, b->d_gt);
    launches++;
    LHB_CUDA(cudaGetLastError());
    count_launch(launches);
    b->launches_last = launches;
    return LHB200_OK;
}

// ncclAllReduce(min) of the batch's device verdict over the library's communicator (lhb200_comm_init), enqueued on
// `stream` right behind lhb200_bls_batch_verify_enqueue: the one collective of the sharded BLS path (SURVEY.md §8e),
// on the device buffer, no host hop.  A no-op without a communicator.
int32_t lhb200_bls_batch_allreduce_verdict(lhb200_bls_batch* b, void* stream) {
    LHB_REQUIRE_READY();
    if (!b) return LHB200_EINVAL;
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx().stream;
    return comm_allreduce_min_u8(b->d_ok, 1, s);
}

int32_t lhb200_bls_batch_result(lhb200_bls_batch* b, void* stream, uint8_t* ok, uint8_t* set_status) {
    LHB_REQUIRE_READY();
    if (!b || !ok) return LHB200_EINVAL;
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx().stream;
    LHB_CUDA(cudaMemcpyAsync(b->h_res, b->d_ok, 1, cudaMemcpyDeviceToHost, s));
    if (set_status) LHB_CUDA(cudaMemcpyAsync(b->h_res + 64, b->d_status, b->n, cudaMemcpyDeviceToHost, s));
    if (b->n >= BLOCKING_WAIT_MIN_SETS && b->e_done) {
        // a long step: sleep on a blocking event instead of spinning in cudaStreamSynchronize — with one process per GPU
        // on a shared host (8 ranks + NCCL proxies under one cgroup CPU quota) eight spinning threads get throttled and
        // the next step's launches start late; the ~30 us wake-up is noise against tens of milliseconds
        LHB_CUDA(cudaEventRecord(b->e_done, s));
        LHB_CUDA(cudaEventSynchronize(b->e_done));
    } else {
        LHB_CUDA(cudaStreamSynchronize(s));
    }
    *ok = b->h_res[0];
    if (set_status) memcpy(set_status, b->h_res + 64, b->n);
    return LHB200_OK;
}

// Test hook: the value final_exp(product)^... of the last verify as 12 x 48-byte big-endian canonical Fp
// (order c0.c0.c0, c0.c0.c1, c0.c1.c0, ... c1.c2.c1).  It is the CUBE of the canonical GT element (pairing.cuh).
int32_t lhb200_bls_batch_gt(lhb200_bls_batch* b, uint8_t out576[576]) {
    LHB_REQUIRE_READY();
    if (!b || !out576) return LHB200_EINVAL;
    Fp12 f;
    LHB_CUDA(cudaDeviceSynchronize());
    LHB_CUDA(cudaMemcpy(&f, b->d_gt, sizeof f, cudaMemcpyDeviceToHost));
    const Fp* c = reinterpret_cast<const Fp*>(&f);
    // host-side conversion out of Montgomery form (plain integer arithmetic on 12 limbs, test hook only)
    for (int k = 0; k < 12; k++) {
        // t = c[k] * R^-1 mod p via 12 rounds of word-wise Montgomery reduction
        uint64_t t[13] = {0};
        for (int i = 0; i < 12; i++) t[i] = c[k].v[i];
        static const uint32_t P32[12] = {0xffffaaabu, 0xb9feffffu, 0xb153ffffu, 0x1eabfffeu, 0xf6b0f624u, 0x6730d2a0u,
                                         0xf38512bfu, 0x64774b84u, 0x434bacd7u, 0x4b1ba7b6u, 0x397fe69au, 0x1a0111eau};
        for (int i = 0; i < 12; i++) {
            const uint32_t m = (uint32_t)t[0] * 0xfffcfffdu;
            uint64_t carry = 0;
            for (int j = 0; j < 12; j++) {
                uint64_t v = t[j] + (uint64_t)m * P32[j] + carry;
                t[j] = v & 0xffffffffu;
                carry = v >> 32;
            }
            uint64_t top = t[12] + carry;
            for (int j = 0; j < 12; j++) t[j] = t[j + 1];
            t[11] = top & 0xffffffffu;
            t[12] = top >> 32;
        }
        // conditional subtract
        bool ge = t[12] != 0;
        if (!ge) {
            ge = true;
            for (int j = 11; j >= 0; j--) {
                if (t[j] != P32[j]) { ge = t[j] > P32[j]; break; }
            }
        }
        if (ge) {
            int64_t brw = 0;
            for (int j = 0; j < 12; j++) {
                int64_t v = (int64_t)t[j] - P32[j] - brw;
                brw = v < 0;
                t[j] = (uint64_t)(v & 0xffffffff);
            }
        }
        for (int j = 0; j < 12; j++) {
            uint8_t* q = out576 + 48 * k + 4 * (11 - j);
            q[0] = t[j] >> 24; q[1] = t[j] >> 16; q[2] = t[j] >> 8; q[3] = t[j];
        }
    }
    return LHB200_OK;
}

uint64_t lhb200_bls_batch_launches(const lhb200_bls_batch* b) { return b ? b->launches_last : 0; }

// Device time (ms, CUDA events on the launching stream) of the dominant kernel k_miller_multi in the last completed
// enqueue; negative if unavailable.  Call after the stream has been synchronised.
float lhb200_bls_batch_dominant_kernel_ms(const lhb200_bls_batch* b) {
    float ms = -1.f;
    if (!b || cudaEventElapsedTime(&ms, b->e_k0, b->e_k1) != cudaSuccess) { cudaGetLastError(); return -1.f; }
    return ms;
}

// bls::verify_signature_sets (crypto/bls/src/impls/blst.rs:37-119).  *ok = 1 iff every set verifies.
// n_sets == 0 -> *ok = 0 (blst.rs:42-44).  rands may be NULL (drawn internally, 64 nonzero bits each).
// set_status (optional, n bytes): per-set preparation status (0 = fine; see SetStatus in kernels.cuh).
int32_t lhb200_verify_signature_sets(const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                     const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets, uint8_t* ok,
                                     uint8_t* set_status) {
    LHB_REQUIRE_READY();
    if (!ok) return LHB200_EINVAL;
    *ok = 0;
    if (n_sets == 0) return LHB200_OK;
    if (!pk_offsets) { set_error("verify_signature_sets: null offsets"); return LHB200_EINVAL; }
    // Re-entrant: Lighthouse calls this from up to num_cpus blocking workers with <= 64-set gossip batches
    // (beacon_processor/src/lib.rs:202-203,256).  Every call borrows a batch handle (device buffers, streams, events —
    // no cudaMalloc on the steady path) from a pool and drives it on the handle's own stream, so concurrent calls
    // overlap on the device instead of queueing behind one mutex.
    const uint64_t n_keys = pk_offsets[n_sets];
    lhb200_bls_batch* b = pool_acquire(n_sets, n_keys);
    if (!b) return LHB200_ENOMEM;
    int32_t rc = lhb200_bls_batch_upload_async(b, sigs, msgs, pks, pk_offsets, rands, n_sets, b->s_main);
    if (!rc) rc = lhb200_bls_batch_verify_enqueue(b, b->s_main);
    if (!rc) rc = lhb200_bls_batch_result(b, b->s_main, ok, set_status);
    cudaStreamSynchronize(b->s2);
    cudaStreamSynchronize(b->s3);
    pool_release(b);
    return rc;
}

// Many independent verify_signature_sets calls in one pass: group g owns sets [group_offsets[g], group_offsets[g+1])
// and ok[g] is what lhb200_verify_signature_sets would return for those sets alone (an empty group: 0).  What
// Lighthouse's batch fallbacks need (attestation_verification/batch.rs): one call that names the bad items instead of one
// call per item.  The per-set stages are shared; sums, Miller products and final exponentiations are per group.
int32_t lhb200_verify_signature_set_groups(const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                           const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets,
                                           const uint32_t* group_offsets, uint32_t n_groups, uint8_t* ok,
                                           uint8_t* set_status) {
    LHB_REQUIRE_READY();
    if (!group_offsets || (n_groups && !ok)) { set_error("verify_signature_set_groups: null argument"); return LHB200_EINVAL; }
    if (n_groups) memset(ok, 0, n_groups);
    if (group_offsets[0] != 0 || group_offsets[n_groups] != n_sets) {
        set_error("verify_signature_set_groups: group offsets must run from 0 to n_sets");
        return LHB200_EINVAL;
    }
    for (uint32_t g = 0; g < n_groups; g++)
        if (group_offsets[g] > group_offsets[g + 1]) { set_error("verify_signature_set_groups: group offsets not monotone"); return LHB200_EINVAL; }
    if (n_sets == 0) return LHB200_OK;   // every group is empty
    // one group: the plain single-verdict path
    if (n_groups == 1) return lhb200_verify_signature_sets(sigs, msgs, pks, pk_offsets, rands, n_sets, ok, set_status);
    if (!pk_offsets) { set_error("verify_signature_set_groups: null offsets"); return LHB200_EINVAL; }
    groups::Plan plan;
    groups::build_plan(plan, group_offsets, n_groups);
    lhb200_bls_batch* b = pool_acquire(n_sets, pk_offsets[n_sets]);
    if (!b) return LHB200_ENOMEM;
    int32_t rc = group_reserve(b, plan, n_sets);
    if (!rc) rc = lhb200_bls_batch_upload_async(b, sigs, msgs, pks, pk_offsets, rands, n_sets, b->s_main);
    if (!rc) {
        const cudaError_t e = cudaMemcpyAsync(b->d_gwords, plan.words.data(), plan.words.size() * 4, cudaMemcpyHostToDevice, b->s_main);
        if (e != cudaSuccess) rc = cuda_fail(e, "group plan upload");
    }
    if (!rc) {
        b->grp = &plan;
        rc = lhb200_bls_batch_verify_enqueue(b, b->s_main);
        b->grp = nullptr;
    }
    if (!rc) {   // (there may be more groups than the handle's pinned result buffer holds: straight to the caller)
        cudaError_t e = cudaMemcpyAsync(ok, b->d_gok, n_groups, cudaMemcpyDeviceToHost, b->s_main);
        if (e == cudaSuccess && set_status)
            e = cudaMemcpyAsync(set_status, b->d_status, n_sets, cudaMemcpyDeviceToHost, b->s_main);
        if (e == cudaSuccess) e = cudaStreamSynchronize(b->s_main);
        if (e != cudaSuccess) rc = cuda_fail(e, "grouped verdicts");
    }
    cudaStreamSynchronize(b->s_main);   // `plan` must outlive its upload
    cudaStreamSynchronize(b->s2);
    cudaStreamSynchronize(b->s3);
    pool_release(b);
    if (rc && n_groups) memset(ok, 0, n_groups);
    return rc;
}

// verify_signature_sets over the ranks of the library's communicator: every rank passes ITS shard of the sets (possibly
// empty: an empty shard contributes `true`), runs the batch check on it with its own blinding scalars and final
// exponentiation, and the verdicts are combined by one ncclAllReduce(min) on the device (SURVEY.md §8e option (a)).
// *ok is the verdict of the WHOLE batch on every rank.  Without a communicator this is lhb200_verify_signature_sets
// (except that n_sets == 0 yields *ok = 1: "this shard has nothing to object to").
int32_t lhb200_verify_signature_sets_collective(const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                                const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets,
                                                uint8_t* ok) {
    LHB_REQUIRE_READY();
    if (!ok) return LHB200_EINVAL;
    *ok = 0;
    if (n_sets && !pk_offsets) return LHB200_EINVAL;
    const uint64_t n_keys = n_sets ? pk_offsets[n_sets] : 0;
    lhb200_bls_batch* b = pool_acquire(std::max<uint32_t>(n_sets, 1), n_keys);
    if (!b) return LHB200_ENOMEM;
    int32_t rc = LHB200_OK;
    if (n_sets) {
        rc = lhb200_bls_batch_upload_async(b, sigs, msgs, pks, pk_offsets, rands, n_sets, b->s_main);
        if (!rc) rc = lhb200_bls_batch_verify_enqueue(b, b->s_main);
    } else {
        const uint8_t one = 1;
        cudaError_t e = cudaMemcpyAsync(b->d_ok, &one, 1, cudaMemcpyHostToDevice, b->s_main);
        if (e == cudaSuccess) e = cudaStreamSynchronize(b->s_main);   // `one` is a stack variable
        if (e != cudaSuccess) rc = cuda_fail(e, "empty shard verdict");
        b->n = 0;
    }
    if (!rc) rc = comm_allreduce_min_u8(b->d_ok, 1, b->s_main);
    if (!rc) rc = lhb200_bls_batch_result(b, b->s_main, ok, nullptr);
    cudaStreamSynchronize(b->s2);
    cudaStreamSynchronize(b->s3);
    pool_release(b);
    return rc;
}

// TSecretKey::public_key (blst.rs:282-298): n big-endian 32-byte scalars -> compressed (48 B) and/or
// uncompressed (96 B) public keys.  Either output may be NULL.
int32_t lhb200_sk_to_pk(const uint8_t* sk32, uint32_t n, uint8_t* pk48, uint8_t* pk96) {
    LHB_REQUIRE_READY();
    if (n == 0) return LHB200_OK;
    if (!sk32 || (!pk48 && !pk96)) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch((size_t)n * (32 + 48 + 96) + 1024));
    if (!d) return LHB200_ENOMEM;
    uint8_t *d48 = d + (size_t)n * 32, *d96 = d48 + (size_t)n * 48;
    LHB_CUDA(cudaMemcpyAsync(d, sk32, (size_t)n * 32, cudaMemcpyHostToDevice, c.stream));
    k_sk_to_pk<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, n, pk48 ? d48 : nullptr, pk96 ? d96 : nullptr);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    if (pk48) LHB_CUDA(cudaMemcpyAsync(pk48, d48, (size_t)n * 48, cudaMemcpyDeviceToHost, c.stream));
    if (pk96) LHB_CUDA(cudaMemcpyAsync(pk96, d96, (size_t)n * 96, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    return LHB200_OK;
}

// TSecretKey::sign (blst.rs:282-298 / generic_secret_key.rs): sig_i = sk_i * H(msg_i), compressed 96 B.
int32_t lhb200_sign(const uint8_t* sk32, const uint8_t* msg32, uint32_t n, uint8_t* sig96) {
    LHB_REQUIRE_READY();
    if (n == 0) return LHB200_OK;
    if (!sk32 || !msg32 || !sig96) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch((size_t)n * (32 + 32 + 96) + 1024));
    if (!d) return LHB200_ENOMEM;
    uint8_t *dm = d + (size_t)n * 32, *ds = dm + (size_t)n * 32;
    LHB_CUDA(cudaMemcpyAsync(d, sk32, (size_t)n * 32, cudaMemcpyHostToDevice, c.stream));
    LHB_CUDA(cudaMemcpyAsync(dm, msg32, (size_t)n * 32, cudaMemcpyHostToDevice, c.stream));
    k_sign<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, dm, n, ds);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    LHB_CUDA(cudaMemcpyAsync(sig96, ds, (size_t)n * 96, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    return LHB200_OK;
}

// PublicKey::deserialize + key_validate for n compressed keys (blst.rs:130-140; the batch form of
// validator_pubkey_cache.rs:116-118).  status[i]: 0 ok, 1 infinity (rejected, generic_public_key.rs:87-88),
// 2 bad encoding / not on curve, 3 not in the r-order subgroup.  pk96[i] is zeroed unless status is 0.
int32_t lhb200_g1_decompress_validate(const uint8_t* pk48, uint32_t n, uint8_t* pk96, uint8_t* status) {
    LHB_REQUIRE_READY();
    if (n == 0) return LHB200_OK;
    if (!pk48 || !pk96 || !status) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch((size_t)n * (48 + 96 + 1) + 1024));
    if (!d) return LHB200_ENOMEM;
    uint8_t *d96 = d + (size_t)n * 48, *dst = d96 + (size_t)n * 96;
    LHB_CUDA(cudaMemcpyAsync(d, pk48, (size_t)n * 48, cudaMemcpyHostToDevice, c.stream));
    k_g1_decompress_validate<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, n, d96, dst);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    LHB_CUDA(cudaMemcpyAsync(pk96, d96, (size_t)n * 96, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaMemcpyAsync(status, dst, n, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    return LHB200_OK;
}

// Signature::deserialize for n compressed signatures (blst.rs:192-194): 192-byte affine out
// (x.c1 | x.c0 | y.c1 | y.c0), status[i]: 0 ok, 1 infinity, 2 bad encoding / not on curve.  No subgroup check.
int32_t lhb200_g2_decompress(const uint8_t* sig96, uint32_t n, uint8_t* out192, uint8_t* status) {
    LHB_REQUIRE_READY();
    if (n == 0) return LHB200_OK;
    if (!sig96 || !out192 || !status) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch((size_t)n * (96 + 192 + 1) + 1024));
    if (!d) return LHB200_ENOMEM;
    uint8_t *do_ = d + (size_t)n * 96, *dst = do_ + (size_t)n * 192;
    LHB_CUDA(cudaMemcpyAsync(d, sig96, (size_t)n * 96, cudaMemcpyHostToDevice, c.stream));
    k_g2_decompress<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, n, do_, dst);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    LHB_CUDA(cudaMemcpyAsync(out192, do_, (size_t)n * 192, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaMemcpyAsync(status, dst, n, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    return LHB200_OK;
}


// ---- aggregation surface of a crypto/bls backend --------------------------------------------------------------
// TAggregateSignature::add_assign / add_assign_aggregate (blst.rs:230-237) and AggregateSignature aggregation in
// general: out = sum of n compressed signatures.  No subgroup check (blst.rs:231: "signature has already been subgroup
// checked"); infinity encodings are the identity; n == 0 gives the infinity signature.  LHB200_EDECODE if any encoding
// is malformed.
int32_t lhb200_g2_aggregate(const uint8_t* sigs96, uint32_t n, uint8_t out96[96]) {
    LHB_REQUIRE_READY();
    if (!out96 || (n && !sigs96)) return LHB200_EINVAL;
    if (n == 0) { memset(out96, 0, 96); out96[0] = 0xc0; return LHB200_OK; }
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    const uint64_t n1 = cdiv(n, REDUCE_CHUNK) + 1;
    const size_t b_in = ((size_t)n * 96 + 255) / 256 * 256, b_pts = (size_t)n * sizeof(G2Jac), b_t = (size_t)n1 * sizeof(G2Jac);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch(b_in + b_pts + 2 * b_t + 512));
    if (!d) return LHB200_ENOMEM;
    G2Jac* pts = reinterpret_cast<G2Jac*>(d + b_in);
    G2Jac* tmp[2] = {reinterpret_cast<G2Jac*>(d + b_in + b_pts), reinterpret_cast<G2Jac*>(d + b_in + b_pts + b_t)};
    uint8_t* d_out = d + b_in + b_pts + 2 * b_t;
    uint32_t* d_bad = reinterpret_cast<uint32_t*>(d_out + 128);
    LHB_CUDA(cudaMemcpyAsync(d, sigs96, (size_t)n * 96, cudaMemcpyHostToDevice, c.stream));
    LHB_CUDA(cudaMemsetAsync(d_bad, 0, 4, c.stream));
    k_g2_load_points<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, n, pts, d_bad);
    uint64_t launches = 2;
    const G2Jac* cur = pts;
    uint32_t m = n;
    int flip = 0;
    while (m > 1) {
        const uint32_t mo = cdiv(m, REDUCE_CHUNK);
        k_g2_reduce<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(cur, m, REDUCE_CHUNK, tmp[flip]);
        launches++;
        cur = tmp[flip];
        flip ^= 1;
        m = mo;
    }
    k_g2_store_point<<<1, 32, 0, c.stream>>>(cur, d_out);
    count_launch(launches);
    LHB_CUDA(cudaGetLastError());
    uint8_t h[96];
    uint32_t bad = 0;
    LHB_CUDA(cudaMemcpyAsync(h, d_out, 96, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    if (bad) { set_error("g2_aggregate: %u malformed signature encodings", bad); return LHB200_EDECODE; }
    memcpy(out96, h, 96);
    return LHB200_OK;
}

// TAggregatePublicKey::aggregate (blst.rs:178-184): sum of n uncompressed keys ("already checked for subgroup and
// infinity"), both serialisations out (either may be NULL).  n == 0 -> LHB200_EINVAL (blst: AGGR_TYPE_MISMATCH).
// Malformed / off-curve key -> LHB200_EDECODE.
int32_t lhb200_g1_aggregate(const uint8_t* pks96, uint32_t n, uint8_t* out48, uint8_t* out96) {
    LHB_REQUIRE_READY();
    if (!pks96 || n == 0 || (!out48 && !out96)) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    const uint64_t n1 = cdiv(n, REDUCE_CHUNK) + 1;
    const size_t b_in = ((size_t)n * 96 + 255) / 256 * 256, b_pts = (size_t)n * sizeof(G1Jac), b_t = (size_t)n1 * sizeof(G1Jac);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch(b_in + b_pts + 2 * b_t + 512));
    if (!d) return LHB200_ENOMEM;
    G1Jac* pts = reinterpret_cast<G1Jac*>(d + b_in);
    G1Jac* tmp[2] = {reinterpret_cast<G1Jac*>(d + b_in + b_pts), reinterpret_cast<G1Jac*>(d + b_in + b_pts + b_t)};
    uint8_t* d_out = d + b_in + b_pts + 2 * b_t;
    uint32_t* d_bad = reinterpret_cast<uint32_t*>(d_out + 256);
    LHB_CUDA(cudaMemcpyAsync(d, pks96, (size_t)n * 96, cudaMemcpyHostToDevice, c.stream));
    LHB_CUDA(cudaMemsetAsync(d_bad, 0, 4, c.stream));
    k_g1_load_points<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, n, pts, nullptr, nullptr, d_bad);
    uint64_t launches = 2;
    const G1Jac* cur = pts;
    uint32_t m = n;
    int flip = 0;
    while (m > 1) {
        const uint32_t mo = cdiv(m, REDUCE_CHUNK);
        k_g1_reduce<<<cdiv(mo, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(cur, m, REDUCE_CHUNK, tmp[flip]);
        launches++;
        cur = tmp[flip];
        flip ^= 1;
        m = mo;
    }
    k_g1_store_point<<<1, 32, 0, c.stream>>>(cur, d_out, d_out + 64);
    count_launch(launches);
    LHB_CUDA(cudaGetLastError());
    uint8_t h[160];
    uint32_t bad = 0;
    LHB_CUDA(cudaMemcpyAsync(h, d_out, 160, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    if (bad) { set_error("g1_aggregate: %u malformed or off-curve keys", bad); return LHB200_EDECODE; }
    if (out48) memcpy(out48, h, 48);
    if (out96) memcpy(out96, h + 64, 96);
    return LHB200_OK;
}

// TPublicKey::deserialize_uncompressed (blst.rs:142-150), batch form: encoding and on-curve checks, NO subgroup check
// (blst's P1 deserialize does none).  status[i]: 0 ok, 1 infinity, 2 bad encoding / not on the curve.  pk48 (optional):
// the compressed form of every accepted key (zeros otherwise).
int32_t lhb200_g1_deserialize_uncompressed(const uint8_t* pks96, uint32_t n, uint8_t* pk48, uint8_t* status) {
    LHB_REQUIRE_READY();
    if (n == 0) return LHB200_OK;
    if (!pks96 || !status) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    const size_t b_in = ((size_t)n * 96 + 255) / 256 * 256, b_48 = ((size_t)n * 48 + 255) / 256 * 256;
    uint8_t* d = static_cast<uint8_t*>(dev_scratch(b_in + b_48 + n + 512));
    if (!d) return LHB200_ENOMEM;
    uint8_t *d48 = d + b_in, *dst = d48 + b_48;
    uint32_t* d_bad = reinterpret_cast<uint32_t*>(dst + (n + 255) / 256 * 256);
    LHB_CUDA(cudaMemcpyAsync(d, pks96, (size_t)n * 96, cudaMemcpyHostToDevice, c.stream));
    LHB_CUDA(cudaMemsetAsync(d_bad, 0, 4, c.stream));
    k_g1_load_points<<<cdiv(n, BLS_BLOCK), BLS_BLOCK, 0, c.stream>>>(d, n, nullptr, pk48 ? d48 : nullptr, dst, d_bad);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    if (pk48) LHB_CUDA(cudaMemcpyAsync(pk48, d48, (size_t)n * 48, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaMemcpyAsync(status, dst, n, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    return LHB200_OK;
}

// TAggregateSignature::aggregate_verify (blst.rs:263-273; generic_aggregate_signature.rs:213-222):
// e(g1, sig) == prod_i e(pk_i, H(m_i)) with the signature subgroup-checked.  n == 0 -> *ok = 0.
// Runs on the batch pipeline: set 0 carries `sig`, the other sets the infinity signature, all blinding scalars are 1,
// so prod_i e(pk_i, H(m_i)) * e(-g1, sig) == 1 is exactly the check.
int32_t lhb200_aggregate_verify(const uint8_t sig96[96], const uint8_t* msgs, const uint8_t* pks96, uint32_t n, uint8_t* ok) {
    LHB_REQUIRE_READY();
    if (!ok) return LHB200_EINVAL;
    *ok = 0;
    if (n == 0) return LHB200_OK;
    if (!sig96 || !msgs || !pks96) return LHB200_EINVAL;
    std::vector<uint8_t> sigs((size_t)n * 96, 0);
    std::vector<uint32_t> offs(n + 1);
    std::vector<uint64_t> ones(n, 1);
    memcpy(sigs.data(), sig96, 96);
    for (uint32_t i = 1; i < n; i++) sigs[(size_t)i * 96] = 0xc0;
    for (uint32_t i = 0; i <= n; i++) offs[i] = i;
    return lhb200_verify_signature_sets(sigs.data(), msgs, pks96, offs.data(), ones.data(), n, ok, nullptr);
}

// Test hook: run one pipeline stage on a single device thread (op codes in bls/debug.cuh).
int32_t lhb200_debug_bls(int32_t op, const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len, int32_t* rc) {
    LHB_REQUIRE_READY();
    if (!in || !out || !rc) return LHB200_EINVAL;
    Ctx& c = ctx();
    std::lock_guard<std::recursive_mutex> g(c.mu);
    uint8_t* d = static_cast<uint8_t*>(dev_scratch((size_t)in_len + out_len + 1024));
    if (!d) return LHB200_ENOMEM;
    uint8_t* d_out = d + ((in_len + 255) / 256) * 256;
    int32_t* d_rc = reinterpret_cast<int32_t*>(d_out + ((out_len + 255) / 256) * 256);
    LHB_CUDA(cudaMemcpyAsync(d, in, in_len, cudaMemcpyHostToDevice, c.stream));
    LHB_CUDA(cudaMemsetAsync(d_out, 0, out_len, c.stream));
    k_debug_bls<<<1, 32, 0, c.stream>>>(op, d, d_out, d_rc);
    count_launch();
    LHB_CUDA(cudaGetLastError());
    LHB_CUDA(cudaMemcpyAsync(out, d_out, out_len, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaMemcpyAsync(rc, d_rc, 4, cudaMemcpyDeviceToHost, c.stream));
    LHB_CUDA(cudaStreamSynchronize(c.stream));
    return LHB200_OK;
}

}  // extern "C"
