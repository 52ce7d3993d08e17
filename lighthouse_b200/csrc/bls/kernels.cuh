// kernels.cuh — CUDA kernels of the batch BLS verification path (sm_100a).  One thread owns one SignatureSet
// through each stage (the work is long, branch-light and identical across sets; parallelism comes from the
// batch).  Stage outputs go through HBM in AoS form: they are tiny next to the arithmetic
// (1.2 KB per set against ~20k Montgomery multiplications).
//
// Stage map (SURVEY.md §2d):
//   k_sig_prepare ...... K10 g2_decompress + K4 subgroup check + K7 r*sig        (blst.rs:73-83, :114)
//   k_pk_aggregate ..... K5 segmented G1 sum over CSR offsets + K7 r*apk          (blst.rs:86-106, :114)
//   k_hash_to_g2 ....... K6 hash_to_curve                                         (blst.rs:114, DST :15)
//   k_miller_multi ..... K8 Miller loops, k sets per thread sharing the Fp12 squarings
//   k_fp12_reduce / k_g2_reduce ... product / sum trees
//   k_final ............ K8 Miller loop for (-g1, sum r*sig) + K9 final exponentiation and == 1
#pragma once
#include "pairing.cuh"
#include "miller_coop.cuh"
#include "miller_warp.cuh"
#include "h2c.cuh"

namespace lhb200 {
namespace bls {

enum SetStatus : uint8_t {
    SET_OK = 0,
    SET_EMPTY_SIG = 1,      // all-zero "empty" signature (generic_signature.rs:26) -> batch false (blst.rs:79-82)
    SET_SIG_DECODE = 2,     // malformed compressed G2
    SET_SIG_SUBGROUP = 3,   // blst.rs:75-77
    SET_NO_KEYS = 4,        // blst.rs:86-89
    SET_APK_INFINITY = 5,   // aggregate key at infinity (Appendix C item 5)
    SET_PK_DECODE = 6,      // malformed uncompressed G1 key
};

constexpr int BLS_BLOCK = 64;
#ifndef LHB_MILLER_BLOCK
#define LHB_MILLER_BLOCK 64
#endif
constexpr int MILLER_BLOCK = LHB_MILLER_BLOCK;  // k_miller_multi's block size (its 4.5 KB/thread stack vs the 126 MB L2)

__device__ __forceinline__ void load_bytes16(uint8_t* dst, const uint8_t* src, int nbytes) {
    // src is 16-byte aligned; nbytes multiple of 16
    for (int i = 0; i < nbytes; i += 16) {
        uint4 v = __ldg(reinterpret_cast<const uint4*>(src + i));
        *reinterpret_cast<uint4*>(dst + i) = v;
    }
}

}  // namespace bls
}  // namespace lhb200
#include "g2_warp.cuh"   // latency-mode twins of the two kernels below (one warp per signature / message)
#include "fe_warp.cuh"   // product of the Miller values + final exponentiation by one warp
namespace lhb200 {
namespace bls {

__global__ void __launch_bounds__(BLS_BLOCK) k_sig_prepare(const uint8_t* __restrict__ sigs,
                                                            const uint64_t* __restrict__ rands, uint32_t n,
                                                            G2Jac* __restrict__ sig_r, uint8_t* __restrict__ status,
                                                            uint32_t* __restrict__ fail) {
    // grid-stride: the host caps resident CTAs per SM so the per-thread stacks stay cache-resident
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        __align__(16) uint8_t b[96];
        load_bytes16(b, sigs + 96ull * i, 96);
        uint32_t nz = 0;
        for (int k = 0; k < 96; k++) nz |= b[k];
        G2Jac out;
        jac_set_inf(out);
        uint8_t st = SET_OK;
        if (nz == 0) {
            st = SET_EMPTY_SIG;
        } else {
            G2Affine a;
            const int32_t rc = g2_decompress(a, b);
            if (rc == DEC_BAD) st = SET_SIG_DECODE;
            else if (rc == DEC_OK) {
                // [r]sig and [|x|]sig in one pass; in G2  <=>  psi(sig) == -[|x|]sig   (blst.rs:75)
                G2Jac xs, ps, aj;
                g2_mul_r_and_x(out, xs, a, rands[i]);
                jac_neg(xs, xs);
                jac_from_affine(aj, a);
                g2_psi(ps, aj);
                if (!jac_eq(ps, xs)) { st = SET_SIG_SUBGROUP; jac_set_inf(out); }
            }
            // DEC_INFINITY: the infinity signature passes the subgroup check and contributes nothing to the sum
        }
        sig_r[i] = out;
        if (st != SET_OK) { status[i] = st; atomicOr(fail, 1u); }
    }
}

__global__ void __launch_bounds__(BLS_BLOCK) k_pk_aggregate(const uint8_t* __restrict__ pks,
                                                             const uint32_t* __restrict__ offsets,
                                                             const uint64_t* __restrict__ rands, uint32_t n,
                                                             G1Proj3* __restrict__ out_p, uint8_t* __restrict__ status,
                                                             uint32_t* __restrict__ fail) {
    // grid-stride: the host caps resident CTAs per SM so the per-thread stacks stay cache-resident
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t lo = offsets[i], hi = offsets[i + 1];
        uint8_t st = SET_OK;
        G1Jac acc;
        jac_set_inf(acc);
        if (hi <= lo) st = SET_NO_KEYS;
        for (uint32_t j = lo; j < hi && st == SET_OK; j++) {
            __align__(16) uint8_t b[96];
            load_bytes16(b, pks + 96ull * j, 96);
            G1Affine a;
            if (g1_from_uncompressed(a, b) == DEC_BAD) { st = SET_PK_DECODE; break; }
            jac_add_affine(acc, acc, a);
        }
        if (st == SET_OK && jac_is_inf(acc)) st = SET_APK_INFINITY;
        G1Proj3 P;
        if (st == SET_OK) {
            G1Jac ra;
            jac_mul_u64(ra, acc, rands[i]);
            g1proj3_from_jac(P, ra);
        } else {
            P.px = FP_ONE; P.py = FP_ONE; P.pz = FP_ONE;
        }
        out_p[i] = P;
        if (st != SET_OK) { status[i] = st; atomicOr(fail, 1u); }
    }
}


// ---------------------------------------------------------------------------------------------------------
// Small and medium batches (the reference's steady state: gossip batches of <= 64 sets, block import with 1 ... 512-key
// sets): one thread per set leaves the GPU idle behind a serial chain of up to 512 additions (7 ms).  Here a set's
// key list is cut into PK_SLICES contiguous slices, one thread each (k_pk_partial); k_pk_combine adds the slice sums
// and multiplies by r.  512 keys: 64 + 8 additions deep instead of 512.  Same statuses as k_pk_aggregate.
constexpr int PK_SLICES = 8;
__global__ void __launch_bounds__(BLS_BLOCK) k_pk_partial(const uint8_t* __restrict__ pks,
                                                           const uint32_t* __restrict__ offsets, uint32_t n,
                                                           G1Jac* __restrict__ part, uint8_t* __restrict__ part_bad) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t i = idx / PK_SLICES, sl = idx % PK_SLICES;
    if (i >= n) return;
    const uint32_t lo = offsets[i], hi = offsets[i + 1];
    const uint32_t nk = hi > lo ? hi - lo : 0, per = (nk + PK_SLICES - 1) / PK_SLICES;
    const uint32_t a0 = min(hi, lo + sl * per), a1 = min(hi, a0 + per);
    G1Jac acc;
    jac_set_inf(acc);
    uint8_t bad = 0;
    for (uint32_t j = a0; j < a1; j++) {
        __align__(16) uint8_t b[96];
        load_bytes16(b, pks + 96ull * j, 96);
        G1Affine a;
        if (g1_from_uncompressed(a, b) == DEC_BAD) { bad = 1; break; }
        jac_add_affine(acc, acc, a);
    }
    part[idx] = acc;
    part_bad[idx] = bad;
}
__global__ void __launch_bounds__(BLS_BLOCK) k_pk_combine(const G1Jac* __restrict__ part,
                                                           const uint8_t* __restrict__ part_bad,
                                                           const uint32_t* __restrict__ offsets,
                                                           const uint64_t* __restrict__ rands, uint32_t n,
                                                           G1Proj3* __restrict__ out_p, uint8_t* __restrict__ status,
                                                           uint32_t* __restrict__ fail) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t st = SET_OK;
    if (offsets[i + 1] <= offsets[i]) st = SET_NO_KEYS;
    G1Jac acc = part[(size_t)i * PK_SLICES];
    uint8_t bad = part_bad[(size_t)i * PK_SLICES];
    for (int sl = 1; sl < PK_SLICES; sl++) {
        G1Jac x = part[(size_t)i * PK_SLICES + sl];
        bad |= part_bad[(size_t)i * PK_SLICES + sl];
        jac_add(acc, acc, x);
    }
    if (st == SET_OK && bad) st = SET_PK_DECODE;
    if (st == SET_OK && jac_is_inf(acc)) st = SET_APK_INFINITY;
    G1Proj3 P;
    if (st == SET_OK) {
        G1Jac ra;
        jac_mul_u64(ra, acc, rands[i]);
        g1proj3_from_jac(P, ra);
    } else {
        P.px = FP_ONE; P.py = FP_ONE; P.pz = FP_ONE;
    }
    out_p[i] = P;
    if (st != SET_OK) { status[i] = st; atomicOr(fail, 1u); }
}

// ---------------------------------------------------------------------------------------------------------
// k_pk_aggregate_tma — the same per-set aggregation with the key ingest STAGED THROUGH SHARED MEMORY BY THE TMA UNIT
// (north_star: "pubkey batches staged through shared memory via TMA with coalesced HBM loads"; replaces the loop at
// blst.rs:86-106).  One thread still owns one set (the additions of a set are a serial chain), but it never touches
// global memory for keys: every thread issues bulk async copies (cp.async.bulk, SASS UBLKCP) of PK_TMA_KEYS consecutive
// keys of ITS set — whole 32-byte sectors, 192 B per request — into its slot of a PK_TMA_STAGES-deep ring, tracked by
// one mbarrier per stage (64 arrivals + the stage's byte count), and adds keys from shared memory while the next
// stages are in flight.  Ragged sets are natural: a thread copies min(PK_TMA_KEYS, keys left) and, once its set is
// exhausted, keeps arriving with zero bytes until the block's longest set is done.
constexpr int PK_TMA_KEYS = 2;
constexpr int PK_TMA_STAGES = 2;   // 24.6 KB of ring per block: 8 resident blocks per SM, the register limit (3 stages: 6)
constexpr int PK_TMA_SLOT = PK_TMA_KEYS * 96;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// 96-byte uncompressed key held as 24 aligned little-endian words (shared memory): same checks as g1_from_uncompressed
__device__ __forceinline__ int32_t g1_from_uncompressed_words(G1Affine& r, const uint32_t* w) {
    uint32_t v[24];
#pragma unroll
    for (int i = 0; i < 24; i++) v[i] = w[i];
    const uint32_t b0 = v[0] & 0xffu;
    if (b0 & 0xa0) return DEC_BAD;
    if (b0 & 0x40) {
        uint32_t nz = v[0] & 0xffffff3fu;
#pragma unroll
        for (int i = 1; i < 24; i++) nz |= v[i];
        if (nz) return DEC_BAD;
        f_set_zero(r.x); f_set_zero(r.y); r.inf = 1;
        return DEC_INFINITY;
    }
    Fp cx, cy;
#pragma unroll
    for (int i = 0; i < NL; i++) {   // limb i = big-endian bytes 4 (11 - i) .. +3
        cx.v[i] = __byte_perm(v[NL - 1 - i], 0, 0x0123);
        cy.v[i] = __byte_perm(v[2 * NL - 1 - i], 0, 0x0123);
    }
    if (!fp_canon_lt_p(cx) || !fp_canon_lt_p(cy)) return DEC_BAD;
    fp_to_mont(r.x, cx);
    fp_to_mont(r.y, cy);
    r.inf = 0;
    return DEC_OK;
}

__global__ void __launch_bounds__(BLS_BLOCK) k_pk_aggregate_tma(const uint8_t* __restrict__ pks,
                                                                 const uint32_t* __restrict__ offsets,
                                                                 const uint64_t* __restrict__ rands, uint32_t n,
                                                                 G1Proj3* __restrict__ out_p, uint8_t* __restrict__ status,
                                                                 uint32_t* __restrict__ fail) {
    __shared__ __align__(128) uint8_t ring[PK_TMA_STAGES][BLS_BLOCK][PK_TMA_SLOT];
    __shared__ __align__(8) uint64_t bars[PK_TMA_STAGES];
    __shared__ uint32_t max_chunks;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool have = i < n;
    const uint32_t lo = have ? offsets[i] : 0, hi = have ? offsets[i + 1] : 0;
    const uint32_t nk = hi > lo ? hi - lo : 0;
    const uint32_t my_chunks = (nk + PK_TMA_KEYS - 1) / PK_TMA_KEYS;
    if (threadIdx.x == 0) {
        max_chunks = 0;
        for (int s = 0; s < PK_TMA_STAGES; s++) mbar_init(&bars[s], BLS_BLOCK);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    atomicMax(&max_chunks, my_chunks);
    __syncthreads();
    const uint32_t n_chunks = max_chunks;
    auto issue = [&](uint32_t c) {   // chunk c of my set -> my slot of stage c % STAGES
        const int s = c % PK_TMA_STAGES;
        if (c < my_chunks) {
            const uint32_t k0 = lo + c * PK_TMA_KEYS, cnt = min((uint32_t)PK_TMA_KEYS, hi - k0);
            mbar_arrive_expect_tx(&bars[s], cnt * 96);
            bulk_g2s(ring[s][threadIdx.x], pks + 96ull * k0, cnt * 96, &bars[s]);
        } else {
            mbar_arrive(&bars[s]);
        }
    };
    for (uint32_t c = 0; c < (uint32_t)PK_TMA_STAGES && c < n_chunks; c++) issue(c);
    uint8_t st = SET_OK;
    G1Jac acc;
    jac_set_inf(acc);
    if (have && nk == 0) st = SET_NO_KEYS;
    for (uint32_t c = 0; c < n_chunks; c++) {
        const int s = c % PK_TMA_STAGES;
        mbar_wait(&bars[s], (c / PK_TMA_STAGES) & 1);
        if (c < my_chunks && st == SET_OK) {
            const uint32_t cnt = min((uint32_t)PK_TMA_KEYS, nk - c * PK_TMA_KEYS);
            for (uint32_t k = 0; k < cnt; k++) {
                G1Affine a;
                if (g1_from_uncompressed_words(a, reinterpret_cast<const uint32_t*>(ring[s][threadIdx.x] + 96 * k)) == DEC_BAD) {
                    st = SET_PK_DECODE;
                    break;
                }
                jac_add_affine(acc, acc, a);
            }
        }
        if (c + PK_TMA_STAGES < n_chunks) {   // my slot of this stage is free again: order my reads before the refill
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(c + PK_TMA_STAGES);
        }
    }
    if (!have) return;
    if (st == SET_OK && jac_is_inf(acc)) st = SET_APK_INFINITY;
    G1Proj3 P;
    if (st == SET_OK) {
        G1Jac ra;
        jac_mul_u64(ra, acc, rands[i]);
        g1proj3_from_jac(P, ra);
    } else {
        P.px = FP_ONE; P.py = FP_ONE; P.pz = FP_ONE;
    }
    out_p[i] = P;
    if (st != SET_OK) { status[i] = st; atomicOr(fail, 1u); }
}

// Device-resident pubkey table (mirror of ValidatorPubkeyCache, beacon_chain/src/validator_pubkey_cache.rs:20-25):
// entries are affine G1 in Montgomery form, converted once at import, so per-set aggregation needs no decoding.
struct G1Mont {
    Fp x, y;
};
__global__ void __launch_bounds__(BLS_BLOCK) k_table_import(const uint8_t* __restrict__ pks96, uint32_t n,
                                                             G1Mont* __restrict__ out, uint32_t* __restrict__ n_bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    __align__(16) uint8_t b[96];
    load_bytes16(b, pks96 + 96ull * i, 96);
    G1Affine a;
    const int32_t rc = g1_from_uncompressed(a, b);
    G1Mont m;
    m.x = a.x; m.y = a.y;
    if (rc != DEC_OK || !g1_on_curve(a)) {  // infinity is rejected at import like generic_public_key.rs:87-88
        atomicAdd(n_bad, 1u);
        fp_set_zero(m.x); fp_set_zero(m.y);
    }
    out[i] = m;
}

__global__ void __launch_bounds__(BLS_BLOCK) k_pk_aggregate_indexed(const G1Mont* __restrict__ table, uint32_t table_len,
                                                                     const uint32_t* __restrict__ indices,
                                                                     const uint32_t* __restrict__ offsets,
                                                                     const uint64_t* __restrict__ rands, uint32_t n,
                                                                     G1Proj3* __restrict__ out_p,
                                                                     uint8_t* __restrict__ status,
                                                                     uint32_t* __restrict__ fail) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t lo = offsets[i], hi = offsets[i + 1];
        uint8_t st = SET_OK;
        G1Jac acc;
        jac_set_inf(acc);
        if (hi <= lo) st = SET_NO_KEYS;
        for (uint32_t j = lo; j < hi && st == SET_OK; j++) {
            const uint32_t idx = __ldg(indices + j);
            if (idx >= table_len) { st = SET_PK_DECODE; break; }
            G1Affine a;
            const G1Mont& m = table[idx];
            a.x = m.x; a.y = m.y; a.inf = 0;
            jac_add_affine(acc, acc, a);
        }
        if (st == SET_OK && jac_is_inf(acc)) st = SET_APK_INFINITY;
        G1Proj3 P;
        if (st == SET_OK) {
            G1Jac ra;
            jac_mul_u64(ra, acc, rands[i]);
            g1proj3_from_jac(P, ra);
        } else {
            P.px = FP_ONE; P.py = FP_ONE; P.pz = FP_ONE;
        }
        out_p[i] = P;
        if (st != SET_OK) { status[i] = st; atomicOr(fail, 1u); }
    }
}

__global__ void __launch_bounds__(BLS_BLOCK) k_hash_to_g2(const uint8_t* __restrict__ msgs, uint32_t n,
                                                           G2Jac* __restrict__ out_h) {
    // grid-stride: the host caps resident CTAs per SM so the per-thread stacks stay cache-resident
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        __align__(16) uint8_t m[32];
        load_bytes16(m, msgs + 32ull * i, 32);
        G2Jac j;
        hash_to_g2_jac(j, m);
        out_h[i] = j;   // stays Jacobian: the Miller loop's addition steps take a projective Q (no inversion here)
    }
}

// Small batches: two threads per message, one per field element u0 / u1 (hash_to_field is recomputed by both: two SHA
// blocks against ~1 000 field multiplications of a map); the even thread adds the two isogeny images and clears the
// cofactor.  Cuts the serial chain of a hash from two maps + clearing (6.0 ms) to one map + clearing (4.7 ms).
__global__ void __launch_bounds__(BLS_BLOCK) k_hash_to_g2_pair(const uint8_t* __restrict__ msgs, uint32_t n,
                                                                G2Jac* __restrict__ out_h) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t i = idx >> 1, half = idx & 1;
    G2Jac q;
    jac_set_inf(q);
    if (i < n) {
        __align__(16) uint8_t m[32];
        load_bytes16(m, msgs + 32ull * i, 32);
        Fp2 u0, u1, x, y;
        hash_to_field_fp2(u0, u1, m);
        map_to_curve_sswu(x, y, half ? u1 : u0);
        iso_map_g2(q, x, y);
    }
    // the odd lane's point travels to its even neighbour through registers (no shared memory: a carve-out would keep
    // these blocks off the SMs that run the other per-set kernels, see k_pk_aggregate_tma)
    G2Jac o;
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&q);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&o);
#pragma unroll 8
        for (int w = 0; w < (int)(sizeof(G2Jac) / 4); w++) dst[w] = __shfl_down_sync(0xffffffffu, src[w], 1);
    }
    if (i < n && !half) {
        G2Jac r;
        jac_add(q, q, o);
        g2_clear_cofactor(r, q);
        out_h[i] = r;
    }
}

// Group g = sets [g*k, (g+1)*k): one thread runs their Miller loops with shared squarings; out_f[g] = the product.
// The host picks k = ceil(n / resident threads) so that every resident thread gets one group (no partial last wave).
__global__ void __launch_bounds__(MILLER_BLOCK) k_miller_multi(const G1Proj3* __restrict__ P, const G2Jac* __restrict__ H,
                                                             const uint8_t* __restrict__ status, uint32_t n, uint32_t k,
                                                             uint32_t n_groups, Fp12* __restrict__ out_f) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += gridDim.x * blockDim.x) {
        uint32_t idx[MILLER_KMAX];
        int m = 0;
        for (uint32_t j = 0; j < k; j++) {
            const uint32_t i = g * k + j;
            if (i < n && status[i] == SET_OK && !jac_is_inf(H[i])) idx[m++] = i;
        }
        Fp12 f;
        if (m == 0) fp12_set_one(f);
        else miller_loop_multi(f, P, H, idx, m);
        out_f[g] = f;
    }
}

// out[t] = prod in[t*chunk .. min(n,(t+1)*chunk))
__global__ void __launch_bounds__(BLS_BLOCK) k_fp12_reduce(const Fp12* __restrict__ in, uint32_t n, uint32_t chunk,
                                                            Fp12* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t lo = (uint64_t)t * chunk;
    if (lo >= n) return;
    const uint32_t hi = (uint32_t)min((uint64_t)n, lo + chunk);
    Fp12 acc = in[lo];
    for (uint32_t j = (uint32_t)lo + 1; j < hi; j++) {
        Fp12 x = in[j];
        fp12_mul(acc, acc, x);
    }
    out[t] = acc;
}
// out[t] = prod in[seg[t] .. seg[t+1]) (1 if empty): a product level whose chunks never cross a group boundary, so
// that k_final_groups_warp folds a bounded number of values per group (bls/groups.cuh builds the table)
__global__ void __launch_bounds__(BLS_BLOCK) k_fp12_reduce_seg(const Fp12* __restrict__ in, const uint32_t* __restrict__ seg,
                                                                uint32_t n_out, Fp12* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_out) return;
    const uint32_t lo = seg[t], hi = seg[t + 1];
    Fp12 acc;
    if (lo < hi) acc = in[lo];
    else fp12_set_one(acc);
    for (uint32_t j = lo + 1; j < hi; j++) {
        Fp12 x = in[j];
        fp12_mul(acc, acc, x);
    }
    out[t] = acc;
}
__global__ void __launch_bounds__(BLS_BLOCK) k_g2_reduce(const G2Jac* __restrict__ in, uint32_t n, uint32_t chunk,
                                                          G2Jac* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t lo = (uint64_t)t * chunk;
    if (lo >= n) return;
    const uint32_t hi = (uint32_t)min((uint64_t)n, lo + chunk);
    G2Jac acc = in[lo];
    for (uint32_t j = (uint32_t)lo + 1; j < hi; j++) {
        G2Jac x = in[j];
        jac_add(acc, acc, x);
    }
    out[t] = acc;
}

// The G1 argument of the aggregated-signature pair e(-g1, sum r sig), in the Miller kernels' projective form.
__global__ void k_init_neg_g1(G1Proj3* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    G1Proj3 p;
    p.px = G1_GEN_X;
    fp_neg(p.py, G1_GEN_Y);
    p.pz = FP_ONE;
    *out = p;
}

// f_last = Miller(-g1, S) for the aggregated signature term; runs concurrently with k_miller_multi.
__global__ void k_last_miller(const G2Jac* __restrict__ sig_sum, Fp12* __restrict__ out_f) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    G2Jac s = *sig_sum;
    Fp12 f;
    if (jac_is_inf(s)) {
        fp12_set_one(f);
    } else {
        G2Affine q;
        jac_to_affine(q, s);
        G1Proj3 p;
        p.px = G1_GEN_X;
        fp_neg(p.py, G1_GEN_Y);
        p.pz = FP_ONE;
        miller_loop(f, p, q);
    }
    *out_f = f;
}

// verdict = !fail && final_exp(prod * f_last) == 1 ; also exposes the GT value for tests
__global__ void k_final(const Fp12* __restrict__ prod, const Fp12* __restrict__ f_last, const uint32_t* __restrict__ fail,
                        uint8_t* __restrict__ ok, Fp12* __restrict__ gt_out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (*fail) { *ok = 0; return; }
    Fp12 a = *prod, b = *f_last;
    fp12_mul(a, a, b);
    final_exp(a, a);
    if (gt_out) *gt_out = a;
    *ok = fp12_is_one(a) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------------------
// Key-side kernels (SecretKey surface of crypto/bls: sk -> pk, sign) — also the synthetic-workload generators.
// sk: 32-byte big-endian scalars (already reduced mod r).
__global__ void __launch_bounds__(BLS_BLOCK) k_sk_to_pk(const uint8_t* __restrict__ sks, uint32_t n,
                                                         uint8_t* __restrict__ pk48, uint8_t* __restrict__ pk96) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k[8];
    const uint8_t* s = sks + 32ull * i;
    for (int w = 0; w < 8; w++) {
        const uint8_t* q = s + 4 * (7 - w);
        k[w] = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
    }
    G1Affine g;
    g.x = G1_GEN_X; g.y = G1_GEN_Y; g.inf = 0;
    G1Jac j;
    jac_mul_affine(j, g, k, 255);
    G1Affine a;
    jac_to_affine(a, j);
    uint8_t b[96];
    if (pk48) { g1_compress(b, a); for (int t = 0; t < 48; t++) pk48[48ull * i + t] = b[t]; }
    if (pk96) { g1_to_uncompressed(b, a); for (int t = 0; t < 96; t++) pk96[96ull * i + t] = b[t]; }
}

__global__ void __launch_bounds__(BLS_BLOCK) k_sign(const uint8_t* __restrict__ sks, const uint8_t* __restrict__ msgs,
                                                     uint32_t n, uint8_t* __restrict__ sig96) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k[8];
    const uint8_t* s = sks + 32ull * i;
    for (int w = 0; w < 8; w++) {
        const uint8_t* q = s + 4 * (7 - w);
        k[w] = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
    }
    __align__(16) uint8_t m[32];
    for (int t = 0; t < 32; t++) m[t] = msgs[32ull * i + t];
    G2Jac h, r;
    hash_to_g2_jac(h, m);
    jac_mul(r, h, k, 255);
    G2Affine a;
    jac_to_affine(a, r);
    uint8_t b[96];
    g2_compress(b, a);
    for (int t = 0; t < 96; t++) sig96[96ull * i + t] = b[t];
}


// ---------------------------------------------------------------------------------------------------------
// Aggregation surface of a crypto/bls backend (TAggregateSignature::add_assign / add_assign_aggregate
// blst.rs:230-237, TAggregatePublicKey::aggregate blst.rs:178-184, deserialize_uncompressed blst.rs:142-150).
// sum tree over G1 points (k_g2_reduce's twin)
__global__ void __launch_bounds__(BLS_BLOCK) k_g1_reduce(const G1Jac* __restrict__ in, uint32_t n, uint32_t chunk,
                                                          G1Jac* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t lo = (uint64_t)t * chunk;
    if (lo >= n) return;
    const uint32_t hi = (uint32_t)min((uint64_t)n, lo + chunk);
    G1Jac acc = in[lo];
    for (uint32_t j = (uint32_t)lo + 1; j < hi; j++) {
        G1Jac x = in[j];
        jac_add(acc, acc, x);
    }
    out[t] = acc;
}
// compressed signatures -> Jacobian points (infinity = identity); any malformed encoding raises *n_bad
__global__ void __launch_bounds__(BLS_BLOCK) k_g2_load_points(const uint8_t* __restrict__ sig96, uint32_t n,
                                                               G2Jac* __restrict__ out, uint32_t* __restrict__ n_bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t b[96];
    for (int t = 0; t < 96; t++) b[t] = sig96[96ull * i + t];
    G2Affine a;
    G2Jac j;
    jac_set_inf(j);
    const int32_t rc = g2_decompress(a, b);
    if (rc == DEC_BAD) atomicAdd(n_bad, 1u);
    else if (rc == DEC_OK) jac_from_affine(j, a);
    out[i] = j;
}
__global__ void k_g2_store_point(const G2Jac* __restrict__ in, uint8_t* __restrict__ out96) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    G2Jac j = *in;
    G2Affine a;
    jac_to_affine(a, j);
    uint8_t b[96];
    g2_compress(b, a);
    for (int t = 0; t < 96; t++) out96[t] = b[t];
}
// uncompressed keys -> Jacobian points; status as lhb200_g1_deserialize_uncompressed (0 ok, 1 infinity, 2 bad)
__global__ void __launch_bounds__(BLS_BLOCK) k_g1_load_points(const uint8_t* __restrict__ pk96, uint32_t n,
                                                               G1Jac* __restrict__ out, uint8_t* __restrict__ pk48,
                                                               uint8_t* __restrict__ st, uint32_t* __restrict__ n_bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    __align__(16) uint8_t b[96];
    for (int t = 0; t < 96; t++) b[t] = pk96[96ull * i + t];
    G1Affine a;
    int32_t rc = g1_from_uncompressed(a, b);
    if (rc == DEC_OK && !g1_on_curve(a)) rc = DEC_BAD;
    if (rc == DEC_BAD) { atomicAdd(n_bad, 1u); a.inf = 1; }
    if (out) { G1Jac j; jac_from_affine(j, a); out[i] = j; }
    if (st) st[i] = (uint8_t)rc;
    if (pk48) {
        uint8_t c[48];
        if (rc == DEC_OK) g1_compress(c, a);
        else for (int t = 0; t < 48; t++) c[t] = 0;
        for (int t = 0; t < 48; t++) pk48[48ull * i + t] = c[t];
    }
}
__global__ void k_g1_store_point(const G1Jac* __restrict__ in, uint8_t* __restrict__ out48, uint8_t* __restrict__ out96) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    G1Jac j = *in;
    G1Affine a;
    jac_to_affine(a, j);
    uint8_t b[96];
    if (out48) { g1_compress(b, a); for (int t = 0; t < 48; t++) out48[t] = b[t]; }
    if (out96) { g1_to_uncompressed(b, a); for (int t = 0; t < 96; t++) out96[t] = b[t]; }
}

// PublicKey::deserialize + key_validate (blst.rs:130-140): decompress, reject infinity, subgroup check.
// status: 0 ok, 1 infinity, 2 bad encoding / not on curve, 3 not in subgroup.
__global__ void __launch_bounds__(BLS_BLOCK) k_g1_decompress_validate(const uint8_t* __restrict__ pk48, uint32_t n,
                                                                       uint8_t* __restrict__ pk96,
                                                                       uint8_t* __restrict__ st) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t b[96];
    for (int t = 0; t < 48; t++) b[t] = pk48[48ull * i + t];
    G1Affine a;
    const int32_t rc = g1_decompress(a, b);
    uint8_t s = 0;
    if (rc == DEC_BAD) s = 2;
    else if (rc == DEC_INFINITY) s = 1;
    else {
        if (!g1_in_subgroup(a)) s = 3;
    }
    g1_to_uncompressed(b, a);
    for (int t = 0; t < 96; t++) pk96[96ull * i + t] = (s == 0) ? b[t] : 0;
    st[i] = s;
}

// Signature::deserialize (blst.rs:192-194): decompress only (no subgroup check); out 192-byte affine x.c1|x.c0|y.c1|y.c0
__global__ void __launch_bounds__(BLS_BLOCK) k_g2_decompress(const uint8_t* __restrict__ sig96, uint32_t n,
                                                              uint8_t* __restrict__ out192, uint8_t* __restrict__ st) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t b[96];
    for (int t = 0; t < 96; t++) b[t] = sig96[96ull * i + t];
    G2Affine a;
    const int32_t rc = g2_decompress(a, b);
    uint8_t o[192];
    for (int t = 0; t < 192; t++) o[t] = 0;
    if (rc == DEC_OK) {
        Fp c;
        fp_from_mont(c, a.x.c1); fp_to_be48(o, c);
        fp_from_mont(c, a.x.c0); fp_to_be48(o + 48, c);
        fp_from_mont(c, a.y.c1); fp_to_be48(o + 96, c);
        fp_from_mont(c, a.y.c0); fp_to_be48(o + 144, c);
    } else if (rc == DEC_INFINITY) {
        o[0] = 0x40;
    }
    for (int t = 0; t < 192; t++) out192[192ull * i + t] = o[t];
    st[i] = (uint8_t)rc;
}

}  // namespace bls
}  // namespace lhb200
