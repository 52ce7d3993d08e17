// tests/hostsim/hostsim_groups.cpp — TEST INFRASTRUCTURE: the device pieces of the grouped verification
// (lhb200_verify_signature_set_groups) compiled for the host (LHB_HOSTSIM) and run lane by lane: the segmented sum
// r sig (gw::sum_points over the level tables of bls/groups.cuh) and the per-group fold + final exponentiation of
// k_final_groups_warp (fe::group_verdict).  Built by tests/test_hostsim_groups.py into a temporary directory; never
// linked into liblhb200.so.
#define LHB_HOSTSIM 1
#include <string.h>
#include "../../lighthouse_b200/csrc/bls/fp.cuh"
#include "../../lighthouse_b200/csrc/bls/fp2.cuh"
#include "../../lighthouse_b200/csrc/bls/ec.cuh"
#include "../../lighthouse_b200/csrc/bls/h2c.cuh"
#include "../../lighthouse_b200/csrc/bls/pairing.cuh"
#include "../../lighthouse_b200/csrc/bls/miller_warp.cuh"
#include "../../lighthouse_b200/csrc/bls/g2_warp.cuh"
#include "../../lighthouse_b200/csrc/bls/fe_warp.cuh"
#include "../../lighthouse_b200/csrc/bls/groups.cuh"
#include <vector>

using namespace lhb200::bls;
#define EXPORT extern "C" __attribute__((visibility("default")))

static void fp_in(Fp& r, const uint8_t* be48) { Fp c; fp_from_be48(c, be48); fp_to_mont(r, c); }
static void fp_out(uint8_t* be48, const Fp& a) { Fp c; fp_from_mont(c, a); fp_to_be48(be48, c); }
static void fp2_out(uint8_t* b, const Fp2& a) { fp_out(b, a.c0); fp_out(b + 48, a.c1); }
static void fp2_in(Fp2& r, const uint8_t* b) { fp_in(r.c0, b); fp_in(r.c1, b + 48); }
static void fp12_out(uint8_t* b, const Fp12& f) {
    const Fp2* c[6] = {&f.c0.c0, &f.c0.c1, &f.c0.c2, &f.c1.c0, &f.c1.c1, &f.c1.c2};
    for (int i = 0; i < 6; i++) fp2_out(b + 96 * i, *c[i]);
}
static void fp12_in(Fp12& f, const uint8_t* b) {
    Fp2* c[6] = {&f.c0.c0, &f.c0.c1, &f.c0.c2, &f.c1.c0, &f.c1.c1, &f.c1.c2};
    for (int i = 0; i < 6; i++) fp2_in(*c[i], b + 96 * i);
}
static void g2_jac_out(uint8_t* out96, const G2Jac& j) {
    G2Affine o;
    if (jac_is_inf(j)) { f_set_zero(o.x); f_set_zero(o.y); o.inf = 1; }
    else jac_to_affine(o, j);
    g2_compress(out96, o);
}

// The segmented sum r sig of groups (bls/groups.cuh plan, gw::sum_points per chunk, level after level): n compressed
// points (infinity encodings allowed), each fed as a Jacobian point with Z != 1; out96[g] = compressed sum of group g.
// Returns the number of levels run (0: every group has one point, which is its own sum), -1 on a bad encoding.
EXPORT int hs_g2_sum_seg(const uint8_t* pts96, int n, const uint32_t* group_off, int n_groups, uint8_t* out96) {
    using namespace gw;
    std::vector<G2Jac> cur(n);
    for (int j = 0; j < n; j++) {
        G2Affine a; const int rc = g2_decompress(a, pts96 + 96 * j);
        if (rc == DEC_BAD) return -1;
        if (rc == DEC_INFINITY) { jac_set_inf(cur[j]); continue; }
        G2Jac h; jac_from_affine(h, a); jac_dbl(h, h); G2Jac na; jac_from_affine(na, a); jac_neg(na, na); jac_add(h, h, na);
        cur[j] = h;
    }
    lhb200::groups::Plan plan;
    lhb200::groups::build_plan(plan, group_off, (uint32_t)n_groups);
    std::vector<uint32_t> Rv(REGION_WORDS, 0xdeadbeefu);
    uint32_t* R = Rv.data();
    const mw::Tables T = tables();
    put_consts(R);
    for (size_t l = 0; l < plan.sum.n_out.size(); l++) {
        const uint32_t* seg = plan.words.data() + plan.sum.at[l];
        std::vector<G2Jac> next(plan.sum.n_out[l]);
        for (uint32_t t = 0; t < plan.sum.n_out[l]; t++) sum_points(R, 0, T, cur.data(), seg[t], seg[t + 1], &next[t]);
        cur.swap(next);
    }
    if ((int)cur.size() != n_groups) return -2;
    for (int g = 0; g < n_groups; g++) g2_jac_out(out96 + 96 * g, cur[g]);
    return (int)plan.sum.n_out.size();
}

// k_final_groups_warp's body (fe::group_verdict) per group: vals576 the Miller values (val_off CSR over them, n_groups + 1),
// extra576 one value per group, status per set (group_off CSR).  ok[g] the verdict, gt576[g] the exponentiated value
// (zeros when a status or an empty group decides).
EXPORT int hs_final_groups(const uint8_t* vals576, const uint32_t* val_off, const uint8_t* extra576, const uint8_t* status,
                           const uint32_t* group_off, int n_groups, uint8_t* ok, uint8_t* gt576) {
    using namespace fe;
    const mw::Tables T = tables();
    for (int g = 0; g < n_groups; g++) {
        const uint32_t nv = val_off[g + 1] - val_off[g];
        std::vector<Fp12> vals(nv);
        for (uint32_t i = 0; i < nv; i++) fp12_in(vals[i], vals576 + 576ull * (val_off[g] + i));
        Fp12 extra, gt;
        fp12_in(extra, extra576 + 576ull * g);
        memset(&gt, 0, sizeof gt);
        std::vector<uint32_t> Rv(REGION_WORDS, 0xdeadbeefu);
        const bool one = group_verdict(Rv.data(), 0, T, status, group_off[g], group_off[g + 1], vals.data(), nv, &extra, &gt);
        ok[g] = one ? 1 : 0;
        bool zero = true;
        for (int w = 0; w < 12 * NL; w++) zero = zero && reinterpret_cast<const uint32_t*>(&gt)[w] == 0;
        if (zero) memset(gt576 + 576ull * g, 0, 576);
        else fp12_out(gt576 + 576ull * g, gt);
    }
    return 0;
}
