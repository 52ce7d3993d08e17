// miller_warp.cuh — ONE WARP PER PAIRING: the Miller loop of small batches at Fp granularity.
//
// verify_signature_sets on 64 ... a few hundred sets (the reference's gossip batches, beacon_processor/src/lib.rs:202-203;
// blst.rs:114-118 is the multi-pairing behind them) is latency bound: bls/miller_coop.cuh gives a set one lane for its point
// arithmetic and six for f, which leaves a chain of ~33 dependent Fp2 operations per iteration (3.7 ms per loop).  Here a
// whole warp serves one (P, Q) pair and every lane computes ONE Fp value per phase:
//     MUL phase:  slot[d] = (sum_{q<K} X_q * slot[y_q]) / R mod p     X_q = +-slot[x_q] or +-2 slot[x_q]   (fp_sop1<K>)
//     LIN phase:  slot[d] = (sum_q c_q slot[s_q]) / 2^h mod p          c_q in {+-1, +-2, +-3, +-12}
// with a warp barrier between phases.  A doubling step is 2 MUL phases (K = 2) instead of 12 serial Fp2 operations, f^2 and
// f * line one MUL phase (K = 4) each.  The phase tables (which lane computes what, from which slots) are generated and
// CHECKED AGAINST THE ORACLE'S PAIRING on Python integers by scripts/gen_miller_warp.py (formulas as in miller_coop.cuh);
// this file is only the interpreter, and tests/hostsim runs it lane by lane on the CPU.
#pragma once
#include "pairing.cuh"
#include "sop.cuh"

namespace lhb200 {
namespace bls {
namespace mw {

#ifdef LHB_HOSTSIM
#define MW_TABLE static const
#else
#define MW_TABLE static __device__ const   // global memory (L1): the lanes of a warp read 32 different rows
#endif
#include "miller_warp_tables.inc"

constexpr int SL = 13;                          // words per slot: odd, so lanes on distinct slots hit distinct banks
constexpr int REGION_WORDS = MW_NSLOTS * SL;    // one warp's working set (9.8 KB)
constexpr uint32_t X_ZERO = 0, X_NEG = 2, X_DBL = 3, X_NEGDBL = 4;

// Warp bodies shared with tests/hostsim (LHB_HD): a copy loop `for (w = lane; w < n; w += LANES)` is split over the 32
// lanes on the device and run whole by the one CPU "lane" 0; warp_any is the vote over the lanes.
#ifdef LHB_HOSTSIM
constexpr int LANES = 1;
#define MW_SYNCWARP() ((void)0)
LHB_HD LHB_INLINE bool warp_any(bool v) { return v; }
#else
constexpr int LANES = 32;
#define MW_SYNCWARP() __syncwarp()
__device__ __forceinline__ bool warp_any(bool v) { return __any_sync(0xffffffffu, v); }
#endif

LHB_HD LHB_INLINE void ld(Fp& r, const uint32_t* R, int s) {
#pragma unroll
    for (int i = 0; i < NL; i++) r.v[i] = R[s * SL + i];
}
LHB_HD LHB_INLINE void st(uint32_t* R, int s, const Fp& a) {
#pragma unroll
    for (int i = 0; i < NL; i++) R[s * SL + i] = a.v[i];
}

// x operand of a MUL term, branch-free (the 32 lanes of a phase mix all modes): 0, a, p - a, 2 a, 2 p - 2 a  (< 2 p)
LHB_HD LHB_INLINE void xop(Fp& x, const uint32_t* R, int slot, uint32_t mode) {
    Fp a, n, d;
    ld(a, R, slot);
    const uint32_t nz = mode != X_ZERO ? ~0u : 0u;
    const uint32_t neg = (mode == X_NEG || mode == X_NEGDBL) ? ~0u : 0u;
    const uint32_t dbl = mode >= X_DBL ? ~0u : 0u;
#pragma unroll
    for (int i = 0; i < NL; i++) a.v[i] &= nz;
    fp_neg_nr(n, a);
#pragma unroll
    for (int i = 0; i < NL; i++) a.v[i] = (n.v[i] & neg) | (a.v[i] & ~neg);
#pragma unroll
    for (int i = 0; i < NL; i++) d.v[i] = a.v[i] & dbl;
    fp_add_nr(x, a, d);
}

// K * X <= 8 (X = 2: every x operand < 2 p), Y = 1 (stored values are canonical): the bound of fp_sop1
template <int K>
LHB_HD LHB_INLINE void mul_lane(Fp& r, const uint32_t* R, const MwMulOp& op) {
    SopX<K> x;
    SopY<K> y;
#pragma unroll
    for (int q = 0; q < K; q++) {
        xop(x.x[q], R, op.xs[q], op.xm[q]);
        y.base[q] = R + op.ys[q] * SL;
    }
    y.stride = 1;
    fp_sop1<K>(r, x, y);
}

LHB_HD LHB_INLINE void lin_lane(Fp& r, const uint32_t* R, const MwLinOp& op) {
    Fp acc;
    fp_set_zero(acc);
    for (int q = 0; q < (int)op.n; q++) {
        Fp t, m;
        ld(t, R, op.s[q]);
        const int c = op.c[q], ac = c < 0 ? -c : c;
        m = t;
        if (ac >= 2) fp_add_inl(m, t, t);                     // 2 t
        if (ac == 3) fp_add_inl(m, m, t);                     // 3 t
        if (ac == 12) {                                       // 4 t, 8 t, 12 t
            Fp m8;
            fp_add_inl(m, m, m);
            fp_add_inl(m8, m, m);
            fp_add_inl(m, m8, m);
        }
        if (c > 0) fp_add_inl(acc, acc, m);
        else fp_sub_inl(acc, acc, m);
    }
    for (int h = 0; h < (int)op.h; h++) fp_half(acc, acc);
    r = acc;
}

// the three tables of a program (this file: the Miller program; g2_warp.cuh: the G2 ladders)
struct Tables {
    const MwPhase* ph;
    const MwMulOp* mul;
    const MwLinOp* lin;
};

// one lane's value of phase ph (reads only)
LHB_HD LHB_INLINE int phase_compute(Fp& r, const uint32_t* R, int lane, int ph, const Tables& T) {
    const MwPhase P = T.ph[ph];
    if (P.is_mul) {
        const MwMulOp& op = T.mul[(int)P.table * 32 + lane];
        if (P.k == 2) mul_lane<2>(r, R, op);                  // the tables use K = 2 (point steps) and K = 4 (products)
        else mul_lane<4>(r, R, op);
        return op.d;
    }
    const MwLinOp& op = T.lin[(int)P.table * 32 + lane];
    lin_lane(r, R, op);
    return op.d;
}

#ifdef LHB_HOSTSIM
// the CPU runs the 32 lanes of a phase one after the other: all reads first, then all writes
inline void run_section(uint32_t* R, int first, int count, const Tables& T) {
    for (int ph = first; ph < first + count; ph++) {
        Fp r[32];
        int d[32];
        for (int lane = 0; lane < 32; lane++) d[lane] = phase_compute(r[lane], R, lane, ph, T);
        for (int lane = 0; lane < 32; lane++) st(R, d[lane], r[lane]);
    }
}
#else
__device__ __noinline__ void run_section(uint32_t* R, int lane, int first, int count, Tables T) {   // ONE copy of the interpreter
#pragma unroll 1
    for (int ph = first; ph < first + count; ph++) {
        Fp r;
        const int d = phase_compute(r, R, lane, ph, T);
        __syncwarp();
        st(R, d, r);
        __syncwarp();
    }
}
#endif

LHB_HD LHB_INLINE Tables miller_tables() { return Tables{MW_PHASES, MW_MUL, MW_LIN}; }
// words of shared memory a block needs for a copy of a program's tables (stage_tables)
constexpr int table_words(int n_mul, int n_lin, int n_phases) { return n_mul * 4 + n_lin * 3 + n_phases; }
#if !defined(LHB_HOSTSIM)
// Copy a program's tables next to the working sets: every phase starts with a dependent phase -> row fetch, ~0.4 us from
// global memory against ~2-4 us of arithmetic; from shared memory it is a few dozen cycles.  All threads of the block.
__device__ __forceinline__ Tables stage_tables(uint32_t* dst, const Tables& g, int n_mul, int n_lin, int n_phases) {
    static_assert(sizeof(MwMulOp) == 16 && sizeof(MwLinOp) == 12 && sizeof(MwPhase) == 4, "table row sizes");
    uint32_t* d_mul = dst;
    uint32_t* d_lin = d_mul + n_mul * 4;
    uint32_t* d_ph = d_lin + n_lin * 3;
    const uint32_t* s_mul = reinterpret_cast<const uint32_t*>(g.mul);
    const uint32_t* s_lin = reinterpret_cast<const uint32_t*>(g.lin);
    const uint32_t* s_ph = reinterpret_cast<const uint32_t*>(g.ph);
    for (int i = threadIdx.x; i < n_mul * 4; i += blockDim.x) d_mul[i] = s_mul[i];
    for (int i = threadIdx.x; i < n_lin * 3; i += blockDim.x) d_lin[i] = s_lin[i];
    for (int i = threadIdx.x; i < n_phases; i += blockDim.x) d_ph[i] = s_ph[i];
    __syncthreads();
    return Tables{reinterpret_cast<const MwPhase*>(d_ph), reinterpret_cast<const MwMulOp*>(d_mul),
                  reinterpret_cast<const MwLinOp*>(d_lin)};
}
#endif
#ifdef LHB_HOSTSIM
#define MW_RUN(R, lane, SEC) run_section(R, MW_SEC_##SEC##_FIRST, MW_SEC_##SEC##_COUNT, T)
#else
#define MW_RUN(R, lane, SEC) run_section(R, lane, MW_SEC_##SEC##_FIRST, MW_SEC_##SEC##_COUNT, T)
#endif

// f = 1 in the stored form (a0, a1, s, d) of every coefficient
LHB_HD LHB_INLINE void set_one_words(uint32_t* R, int word) {   // word < 24 * SL of the f block, one per call
    const int slot = word / SL, limb = word % SL;
    if (limb >= NL) return;
    const int form = slot & 3;                                  // a0, a1, s, d
    const bool one = slot < 4 && form != 1;                     // coefficient 0: a0 = s = d = 1
    R[(MW_S_F0_0 + slot) * SL + limb] = one ? FP_ONE.v[limb] : 0u;
}

constexpr size_t smem_bytes(int warps) { return ((size_t)warps * REGION_WORDS + table_words(MW_N_MUL, MW_N_LIN, MW_N_PHASES)) * 4; }
#if !defined(LHB_HOSTSIM)
// The Miller loop of one pair by the whole warp: f (stored form, MW_S_F0_0 ...) = f_{|x|,q}(p), conjugated; f = 1 when
// !active (warp-uniform).  Shared by k_miller_warp and k_miller_warp_pairs.
__device__ __forceinline__ void miller_pair(uint32_t* R, int lane, const Tables& T, const G1Proj3* p, const G2Jac* q,
                                            bool active) {
    for (int w = lane; w < 24 * SL; w += 32) set_one_words(R, w);
    if (active) {   // warp-uniform
        const uint32_t* qs = reinterpret_cast<const uint32_t*>(q);     // X.c0 X.c1 Y.c0 Y.c1 Z.c0 Z.c1, 12 words each
        for (int w = lane; w < 6 * NL; w += 32) R[(MW_S_HX_0 + w / NL) * SL + w % NL] = qs[w];
        const uint32_t* ps = reinterpret_cast<const uint32_t*>(p);     // px py pz
        for (int w = lane; w < 3 * NL; w += 32) R[(MW_S_PX + w / NL) * SL + w % NL] = ps[w];
        __syncwarp();
        MW_RUN(R, lane, INIT);
#pragma unroll 1
        for (int i = 62; i >= 0; i--) {
            MW_RUN(R, lane, SQR);
            MW_RUN(R, lane, DBL);
            MW_RUN(R, lane, SPARSE);
            if ((BLS_X_ABS >> i) & 1) {
                MW_RUN(R, lane, ADD);
                MW_RUN(R, lane, SPARSE);
            }
        }
        MW_RUN(R, lane, CONJ);
    }
}

// the warp's f (stored form) -> one Fp12 in tower order
__device__ __forceinline__ void store_f(const uint32_t* R, int lane, Fp12* out) {
    // w-basis coefficient k -> tower: 0 c0.c0, 1 c1.c0, 2 c0.c1, 3 c1.c1, 4 c0.c2, 5 c1.c2 (coop.cuh)
    uint32_t* o = reinterpret_cast<uint32_t*>(out);
    for (int w = lane; w < 12 * NL; w += 32) {
        const int fp2_idx = w / (2 * NL), comp = (w / NL) & 1, limb = w % NL;   // tower order: c0.c0 c0.c1 c0.c2 c1.c0 c1.c1 c1.c2
        const int k = fp2_idx < 3 ? 2 * fp2_idx : 2 * (fp2_idx - 3) + 1;
        o[w] = R[(MW_S_F0_0 + 4 * k + comp) * SL + limb];
    }
}

// One warp per pair (P_i, H_i), i < n, plus the pair (extra_p, extra_q) = (-g1, sum r sig) as pair n.  Invalid sets
// (status != 0, H at infinity) contribute f = 1, like k_miller_coop.  The warps of a block multiply their values
// (dense section) and the block writes ONE Fp12.  Dynamic shared memory: smem_bytes(warps_per_block).
__global__ void __launch_bounds__(256, 1) k_miller_warp(const G1Proj3* __restrict__ P, const G2Jac* __restrict__ H,
                                                        const uint8_t* __restrict__ status, uint32_t n,
                                                        const G2Jac* __restrict__ extra_q, const G1Proj3* __restrict__ extra_p,
                                                        Fp12* __restrict__ out_f) {
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    uint32_t* R = lhb_dyn_smem + (size_t)wib * REGION_WORDS;
    const Tables T = stage_tables(lhb_dyn_smem + (size_t)nw * REGION_WORDS, miller_tables(), MW_N_MUL, MW_N_LIN, MW_N_PHASES);
    const uint32_t n_total = n + (extra_q ? 1u : 0u);
    const uint32_t set = blockIdx.x * nw + wib;
    bool active = set < n_total;
    const G2Jac* q = nullptr;
    const G1Proj3* p = nullptr;
    if (active) {
        if (set >= n) { q = extra_q; p = extra_p; }
        else { q = H + set; p = P + set; active = status[set] == 0; }
        if (active) active = !jac_is_inf(*q);
    }
    miller_pair(R, lane, T, p, q, active);
    // product over the block's warps
    for (int stride = 1; stride < nw; stride *= 2) {
        __syncthreads();
        if (wib % (2 * stride) == 0 && wib + stride < nw) {
            const uint32_t* O = R + (size_t)stride * REGION_WORDS;
            for (int w = lane; w < 24 * SL; w += 32) R[MW_S_G0_0 * SL + w] = O[MW_S_F0_0 * SL + w];
            __syncwarp();
            MW_RUN(R, lane, DENSE);
        }
    }
    if (wib == 0) {
        __syncwarp();
        store_f(R, lane, out_f + blockIdx.x);
    }
}

// Grouped verification: one warp per pair and ONE Fp12 per pair — no product across the warps of a block, whose pairs
// may belong to different groups.  Pair i < n is (P_i, H_i), pair n + g is (extra_p, extra_q[g]) (-g1 and group g's
// sum r sig).  Invalid sets and points at infinity give f = 1, as in k_miller_warp.  Any pair count: the blocks beyond
// the resident ones run in later waves.  Dynamic shared memory: smem_bytes(warps_per_block).
__global__ void __launch_bounds__(256, 1) k_miller_warp_pairs(const G1Proj3* __restrict__ P, const G2Jac* __restrict__ H,
                                                              const uint8_t* __restrict__ status, uint32_t n,
                                                              const G2Jac* __restrict__ extra_q, uint32_t n_extra,
                                                              const G1Proj3* __restrict__ extra_p, Fp12* __restrict__ out_f) {
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    uint32_t* R = lhb_dyn_smem + (size_t)wib * REGION_WORDS;
    const Tables T = stage_tables(lhb_dyn_smem + (size_t)nw * REGION_WORDS, miller_tables(), MW_N_MUL, MW_N_LIN, MW_N_PHASES);
    const uint32_t k = blockIdx.x * nw + wib;
    if (k >= n + n_extra) return;   // no block barrier below
    const G2Jac* q;
    const G1Proj3* p;
    bool active = true;
    if (k >= n) { q = extra_q + (k - n); p = extra_p; }
    else { q = H + k; p = P + k; active = status[k] == 0; }
    if (active) active = !jac_is_inf(*q);
    miller_pair(R, lane, T, p, q, active);
    __syncwarp();
    store_f(R, lane, out_f + k);
}
#endif

}  // namespace mw
}  // namespace bls
}  // namespace lhb200
