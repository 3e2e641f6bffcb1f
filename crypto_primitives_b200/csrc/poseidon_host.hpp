// poseidon_host.hpp -- host-side Poseidon parameter work (once per context).
//
//  * PoseidonGrainLFSR + find_poseidon_ark_and_mds: the reference's parameter generator,
//    R/sponge/poseidon/grain_lfsr.rs:16-181 and R/sponge/poseidon/traits.rs:105-146
//    (same bit stream; state kept as an 80-entry byte ring).
//  * derive_schedule: turns a PoseidonConfig (R/sponge/poseidon/mod.rs:26-45) into the round
//    schedule the CUDA kernels execute.  The reference's permute (mod.rs:98-121) applies a
//    dense t x t MDS in all RF+RP rounds; here the RP partial rounds use the equivalent
//    sparse form (1 row + 1 column per round) with round constants folded so that only lane 0
//    receives a constant.  The rewrite is exact field algebra, so outputs are bit-identical;
//    when a required (t-1)x(t-1) minor is singular the schedule falls back to the dense form.  For t = 3 it adds the
//    lane-0 recurrence of the partial rounds (derive_recurrence), which the one-hash-per-thread kernels run instead.
#pragma once
#include <algorithm>

#include "hostfp.hpp"
#include "poseidon.cuh"

namespace cpb {
namespace host {

// ------------------------------------------------------------------------- Grain LFSR
class GrainLFSR {
public:
    GrainLFSR(bool sbox_inverse, u64 prime_bits, u64 state_len, u64 rf, u64 rp) : prime_bits_(prime_bits) {
        for (int i = 0; i < 80; i++) st_[i] = 0;
        st_[1] = 1;                       // b0,b1: prime field          grain_lfsr.rs:25
        st_[5] = sbox_inverse ? 1 : 0;    // b2..b5: s-box               :28-32
        put(6, 17, prime_bits);           // :35-41
        put(18, 29, state_len);           // :44-50
        put(30, 39, rf);                  // :53-59
        put(40, 49, rp);                  // :62-68
        for (int i = 50; i < 80; i++) st_[i] = 1;   // :71-73
        head_ = 0;
        for (int i = 0; i < 160; i++) update();     // :177-181
    }

    // n bits, first drawn = most significant (grain_lfsr.rs:117-121,144-156), as 4 LE words.
    void draw(u64 out[4]) {
        out[0] = out[1] = out[2] = out[3] = 0;
        for (u64 i = 0; i < prime_bits_; i++) {
            u64 bitpos = prime_bits_ - 1 - i;
            if (next_filtered_bit()) out[bitpos / 64] |= 1ull << (bitpos % 64);
        }
    }

    FeVec rejection_sampling(const Field& F, size_t n) {     // :109-134
        FeVec r;
        while (r.size() < n) {
            u64 v[4];
            draw(v);
            if (!Field::geq(v, F.p)) r.push_back(F.from_canonical(v));
        }
        return r;
    }
    FeVec mod_p(const Field& F, size_t n) {                  // :136-160
        FeVec r;
        for (size_t i = 0; i < n; i++) {
            u64 v[4];
            draw(v);
            r.push_back(F.from_canonical(v));   // reduces mod p
        }
        return r;
    }

private:
    void put(int lo, int hi, u64 v) {
        for (int i = hi; i >= lo; i--) { st_[i] = v & 1; v >>= 1; }
    }
    int update() {                                            // :162-175
        int nb = st_[(head_ + 62) % 80] ^ st_[(head_ + 51) % 80] ^ st_[(head_ + 38) % 80] ^
                 st_[(head_ + 23) % 80] ^ st_[(head_ + 13) % 80] ^ st_[head_];
        st_[head_] = (unsigned char)nb;
        head_ = (head_ + 1) % 80;
        return nb;
    }
    int next_filtered_bit() {                                 // get_bits :87-107
        int b = update();
        while (!b) { update(); b = update(); }
        return update();
    }
    unsigned char st_[80];
    int head_;
    u64 prime_bits_;
};

struct PoseidonParams {
    int rate = 0, capacity = 0, full_rounds = 0, partial_rounds = 0;
    u64 alpha = 0;
    FeVec ark;   // (RF+RP) x t, Montgomery
    FeVec mds;   // t x t row-major, Montgomery
    int t() const { return rate + capacity; }
};

// traits.rs:105-146
inline void find_poseidon_ark_and_mds(const Field& F, u64 prime_bits, int rate, int rf, int rp, int skip,
                                      FeVec& ark, FeVec& mds) {
    int t = rate + 1;
    GrainLFSR lfsr(false, prime_bits, (u64)t, (u64)rf, (u64)rp);
    ark.clear();
    for (int r = 0; r < rf + rp; r++) {
        FeVec row = lfsr.rejection_sampling(F, (size_t)t);
        ark.insert(ark.end(), row.begin(), row.end());
    }
    for (int s = 0; s < skip; s++) (void)lfsr.mod_p(F, (size_t)(2 * t));
    FeVec xs = lfsr.mod_p(F, (size_t)t), ys = lfsr.mod_p(F, (size_t)t);
    mds.assign((size_t)t * t, F.zero());
    for (int i = 0; i < t; i++)
        for (int j = 0; j < t; j++) mds[(size_t)i * t + j] = F.inv(F.add(xs[i], ys[j]));
}

// Default-parameter entry tables of the reference's BLS12-381 test field (R/sponge/test.rs:13-32):
// (rate, alpha, full, partial, skip).  Other fields carry no table in the reference.
struct DefaultEntry { int rate; u64 alpha; int rf, rp, skip; };
inline bool default_entry(int field_id, int rate, bool optimized_for_weights, DefaultEntry& e) {
    if (field_id != 0) return false;   // PoseidonDefaultConfig is implemented per field; the reference does so for its BLS12-381 Fr test field only
    static const DefaultEntry C[7] = {{2, 17, 8, 31, 0}, {3, 5, 8, 56, 0}, {4, 5, 8, 56, 0}, {5, 5, 8, 57, 0},
                                      {6, 5, 8, 57, 0},  {7, 5, 8, 57, 0}, {8, 5, 8, 57, 0}};
    if (rate < 2 || rate > 8) return false;
    if (optimized_for_weights) e = DefaultEntry{rate, 257, 8, 13, 0};
    else e = C[rate - 2];
    return true;
}

// ------------------------------------------------------------------------- device schedule
// All offsets are in field elements into `consts` (8 x u32 / 4 x u64 Montgomery limbs each).
struct PoseidonSchedule {
    int t = 0, rate = 0, capacity = 0, rf = 0, rp = 0, sparse = 0;
    u64 alpha = 0;
    int off_c = 0;     // rf x t   constants added before the s-box of full round fr (0..rf-1)
    int off_m = 0;     // t x t    MDS
    int off_mpre = 0;  // t x t    matrix of the last first-half full round (= D0*M; M when dense)
    int off_cp0 = 0;   // t        constant vector added before the first partial round
    int off_pc = 0;    // rp       lane-0 constant added after partial round k-1 (entry k; entry 0 unused)
    int off_sp = 0;    // rp x (2t-1): per round the row [m00, w_hat[1..t-1]] then v[1..t-1]  (sparse)
    int off_arkp = 0;  // rp x t   original partial-round constants                     (dense schedules only; empty when sparse)
    int off_mod = 0;   // 1        the modulus limbs (plain integer): the kernels load them from here into registers
    int off_sc0 = 0;   // 1        S(C[0][0]): lane 0 after the first S-box when it entered the permutation as zero (fresh sponge)
    // Lane-0 recurrence of the partial rounds (t = 3 sparse schedules; see derive_recurrence).  recur == 0: not used, empty.
    int recur = 0;
    int off_rc = 0;    // 3 x 5    dot rows over the history (y_k, y_k-1, y_k-2, x_k, x_k-1): round 0, round 1, rounds >= 2
    int off_rk = 0;    // rp       constant added to the dot of round k (gives x_k+1; for k = rp-1 the sparse lane 0 after the last round)
    int off_rr = 0;    // 2x4 + 2  lanes 1, 2 after the last round from (y_rp-1, y_rp-2, lane 0, x_rp-1): two rows, two constants
    int n_elems = 0;
    std::vector<u64> consts;
};

namespace detail {
inline FeVec matmul(const Field& F, const FeVec& A, const FeVec& B, int n) {
    FeVec C((size_t)n * n, F.zero());
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
            Fe acc = F.zero();
            for (int k = 0; k < n; k++) acc = F.add(acc, F.mul(A[(size_t)i * n + k], B[(size_t)k * n + j]));
            C[(size_t)i * n + j] = acc;
        }
    return C;
}
inline FeVec matvec(const Field& F, const FeVec& A, const FeVec& x, int n) {
    FeVec y((size_t)n, F.zero());
    for (int i = 0; i < n; i++) {
        Fe acc = F.zero();
        for (int k = 0; k < n; k++) acc = F.add(acc, F.mul(A[(size_t)i * n + k], x[k]));
        y[i] = acc;
    }
    return y;
}
// Gauss-Jordan inverse of an m x m matrix; false when singular.
inline bool invert(const Field& F, FeVec A, int m, FeVec& out) {
    FeVec I((size_t)m * m, F.zero());
    for (int i = 0; i < m; i++) I[(size_t)i * m + i] = F.one();
    for (int c = 0; c < m; c++) {
        int piv = -1;
        for (int r = c; r < m; r++)
            if (!A[(size_t)r * m + c].is_zero()) { piv = r; break; }
        if (piv < 0) return false;
        if (piv != c)
            for (int k = 0; k < m; k++) {
                std::swap(A[(size_t)piv * m + k], A[(size_t)c * m + k]);
                std::swap(I[(size_t)piv * m + k], I[(size_t)c * m + k]);
            }
        Fe inv = F.inv(A[(size_t)c * m + c]);
        for (int k = 0; k < m; k++) {
            A[(size_t)c * m + k] = F.mul(A[(size_t)c * m + k], inv);
            I[(size_t)c * m + k] = F.mul(I[(size_t)c * m + k], inv);
        }
        for (int r = 0; r < m; r++) {
            if (r == c) continue;
            Fe f = A[(size_t)r * m + c];
            if (f.is_zero()) continue;
            for (int k = 0; k < m; k++) {
                A[(size_t)r * m + k] = F.sub(A[(size_t)r * m + k], F.mul(f, A[(size_t)c * m + k]));
                I[(size_t)r * m + k] = F.sub(I[(size_t)r * m + k], F.mul(f, I[(size_t)c * m + k]));
            }
        }
    }
    out = I;
    return true;
}

// Affine forms over the variables of the partial-round linear system (the S-box outputs taken as free inputs):
// entry 0 is the constant term, 1 and 2 lanes 1 and 2 on entry, 3 lane 0 on entry, 4 + k the S-box output y_k.
inline FeVec form_var(const Field& F, int nv, int v) {
    FeVec f((size_t)nv, F.zero());
    if (v >= 0) f[(size_t)v] = F.one();
    return f;
}
inline void form_axpy(const Field& F, FeVec& r, const Fe& c, const FeVec& a) {
    for (size_t i = 0; i < r.size(); i++) r[i] = F.add(r[i], F.mul(c, a[i]));
}
// Coefficients c (free ones 0) with f - sum_i c_i g_i constant, and that constant k; false when there are none.
inline bool solve_affine(const Field& F, const FeVec& f, const std::vector<FeVec>& g, FeVec& c, Fe& k) {
    const int n = (int)g.size(), rows = (int)f.size() - 1;
    std::vector<FeVec> A((size_t)rows, FeVec((size_t)n + 1));
    for (int v = 0; v < rows; v++) {
        for (int i = 0; i < n; i++) A[v][i] = g[i][(size_t)v + 1];
        A[v][n] = f[(size_t)v + 1];
    }
    std::vector<int> pivcol;
    int r = 0;
    for (int col = 0; col < n && r < rows; col++) {
        int piv = -1;
        for (int q = r; q < rows; q++)
            if (!A[q][col].is_zero()) { piv = q; break; }
        if (piv < 0) continue;
        std::swap(A[piv], A[r]);
        const Fe inv = F.inv(A[r][col]);
        for (auto& e : A[r]) e = F.mul(e, inv);
        for (int q = 0; q < rows; q++) {
            if (q == r || A[q][col].is_zero()) continue;
            const Fe m = A[q][col];
            for (int i = 0; i <= n; i++) A[q][i] = F.sub(A[q][i], F.mul(m, A[r][i]));
        }
        pivcol.push_back(col);
        r++;
    }
    for (int q = r; q < rows; q++)
        if (!A[q][n].is_zero()) return false;
    c.assign((size_t)n, F.zero());
    for (int j = 0; j < r; j++) c[(size_t)pivcol[j]] = A[j][n];
    k = f[0];
    for (int i = 0; i < n; i++) k = F.sub(k, F.mul(c[i], g[i][0]));
    return true;
}

// The partial rounds of a t = 3 sparse schedule as a recurrence on lane 0 alone.  Lanes 1, 2 form a linear system driven by
// the S-box outputs, so by Cayley-Hamilton on its 2x2 matrix B (z^2 + d1 z + d2) the lane-0 value x_k+1 after the constant
// addition of round k+1 is, for k >= 2,
//     x_k+1 = m00 y_k + b1 y_k-1 + b2 y_k-2 - d1 x_k - d2 x_k-1 + c_k,      y_k = x_k^alpha,
// with the same five coefficients in every round and c_k fixed by the round constants.  Rounds 0 and 1 get rows of their own over
// the lanes still held on entry (round 0: (y_0, s1, s2, x_0, 0); round 1: (y_1, y_0, s1, x_1, x_0), s2 eliminated through x_1), and
// after the last round lanes 1, 2 are affine in (y_rp-1, y_rp-2, lane 0, x_rp-1).  Every coefficient is solved for exactly on
// affine forms of the sparse rounds (sp, pc), so the kernels reproduce the sparse state bit for bit; false when a system has no
// solution (e.g. w_hat[2] of round 0 is zero, or the last two lane-0 values do not determine lanes 1, 2).
inline bool derive_recurrence(const Field& F, int rp, const FeVec& sp, const FeVec& pc, FeVec& rows, FeVec& ck, FeVec& rr) {
    const int w = 5, nv = 4 + rp;
    if (rp < 3) return false;                      // two bootstrap rounds, then at least one recurrence round
    auto var = [&](int v) { return form_var(F, nv, v); };
    FeVec l1 = var(1), l2 = var(2);
    std::vector<FeVec> x{var(3)};                 // x[k]: lane 0 after the constant addition of round k; x[rp]: after the last round
    for (int k = 0; k < rp; k++) {
        const Fe* row = &sp[(size_t)k * w];
        const FeVec y = var(4 + k);
        FeVec d((size_t)nv, F.zero());
        form_axpy(F, d, row[0], y);
        form_axpy(F, d, row[1], l1);
        form_axpy(F, d, row[2], l2);
        form_axpy(F, l1, row[3], y);
        form_axpy(F, l2, row[4], y);
        if (k + 1 < rp) d[0] = F.add(d[0], pc[(size_t)k + 1]);
        x.push_back(d);
    }
    rows.clear(); ck.clear(); rr.clear();
    for (int k = 0; k < rp; k++) {
        const std::vector<FeVec> h{var(4 + k), var(k >= 1 ? 3 + k : 1), var(k >= 2 ? 2 + k : k == 1 ? 1 : 2), x[(size_t)k],
                                   k >= 1 ? x[(size_t)k - 1] : var(-1)};
        FeVec c;
        Fe c0;
        if (!solve_affine(F, x[(size_t)k + 1], h, c, c0)) return false;
        if (k <= 2) rows.insert(rows.end(), c.begin(), c.end());
        else if (!std::equal(c.begin(), c.end(), rows.begin() + 2 * w)) return false;
        ck.push_back(c0);
    }
    const std::vector<FeVec> h{var(3 + rp), var(2 + rp), x[(size_t)rp], x[(size_t)rp - 1]};
    FeVec c1, c2;
    Fe k1, k2;
    if (!solve_affine(F, l1, h, c1, k1) || !solve_affine(F, l2, h, c2, k2)) return false;
    rr = c1;
    rr.insert(rr.end(), c2.begin(), c2.end());
    rr.push_back(k1);
    rr.push_back(k2);
    return true;
}
}  // namespace detail

inline PoseidonSchedule derive_schedule(const Field& F, const PoseidonParams& P, bool allow_sparse = true) {
    const int t = P.t(), rf = P.full_rounds, rp = P.partial_rounds, half = rf / 2;
    PoseidonSchedule S;
    S.t = t; S.rate = P.rate; S.capacity = P.capacity; S.rf = rf; S.rp = rp; S.alpha = P.alpha;

    const FeVec& M = P.mds;
    FeVec C((size_t)rf * t), Mpre = M, Cp0((size_t)t, F.zero()), pc((size_t)(rp > 0 ? rp : 1), F.zero());
    FeVec sp((size_t)(rp > 0 ? rp : 1) * (2 * t - 1), F.zero()), arkp;
    auto ark = [&](int r, int i) -> const Fe& { return P.ark[(size_t)r * t + i]; };
    for (int fr = 0; fr < rf; fr++) {
        int r = fr < half ? fr : half + rp + (fr - half);
        for (int i = 0; i < t; i++) C[(size_t)fr * t + i] = ark(r, i);
    }
    for (int k = 0; k < rp; k++)
        for (int i = 0; i < t; i++) arkp.push_back(ark(half + k, i));

    bool sparse = allow_sparse && rp > 0 && t >= 2 && half >= 1 && rf > half;
    if (sparse) {
        // backward factorisation  N_k = D_{k+1} * M = Sp_k * D_k,  D_rp = I
        FeVec D((size_t)t * t, F.zero());
        for (int i = 0; i < t; i++) D[(size_t)i * t + i] = F.one();
        const int m = t - 1;
        for (int k = rp - 1; k >= 0 && sparse; k--) {
            FeVec N = detail::matmul(F, D, M, t);
            FeVec Mhat((size_t)m * m), Minv;
            for (int i = 0; i < m; i++)
                for (int j = 0; j < m; j++) Mhat[(size_t)i * m + j] = N[(size_t)(i + 1) * t + (j + 1)];
            if (!detail::invert(F, Mhat, m, Minv)) { sparse = false; break; }
            for (int j = 0; j < m; j++) {   // w_hat^T = w^T * Mhat^-1
                Fe acc = F.zero();
                for (int i = 0; i < m; i++) acc = F.add(acc, F.mul(N[(size_t)0 * t + (i + 1)], Minv[(size_t)i * m + j]));
                sp[(size_t)k * (2 * t - 1) + 1 + j] = acc;
            }
            sp[(size_t)k * (2 * t - 1)] = N[0];   // m00 (row 0 of N equals row 0 of M)
            for (int i = 0; i < m; i++) sp[(size_t)k * (2 * t - 1) + t + i] = N[(size_t)(i + 1) * t + 0];
            for (auto& e : D) e = F.zero();
            D[0] = F.one();
            for (int i = 0; i < m; i++)
                for (int j = 0; j < m; j++) D[(size_t)(i + 1) * t + (j + 1)] = Mhat[(size_t)i * m + j];
        }
        if (sparse) {
            Mpre = detail::matmul(F, D, M, t);
            FeVec c0((size_t)t);
            for (int i = 0; i < t; i++) c0[i] = ark(half, i);
            Cp0 = detail::matvec(F, D, c0, t);
            // forward constant folding: lanes 1.. of each later partial constant move one round on
            FeVec d((size_t)t, F.zero());
            for (int k = 1; k < rp; k++) {
                FeVec md = detail::matvec(F, M, d, t);
                FeVec cp((size_t)t);
                for (int i = 0; i < t; i++) cp[i] = F.add(ark(half + k, i), md[i]);
                pc[k] = cp[0];
                d = cp;
                d[0] = F.zero();
            }
            FeVec post = detail::matvec(F, M, d, t);
            if (rf > half)
                for (int i = 0; i < t; i++) C[(size_t)half * t + i] = F.add(C[(size_t)half * t + i], post[i]);
            else sparse = false;   // no later full round to absorb the folded constants
        }
    }
    if (!sparse) {
        // dense fallback: partial rounds exactly as written in the reference
        for (int fr = 0; fr < rf; fr++) {
            int r = fr < half ? fr : half + rp + (fr - half);
            for (int i = 0; i < t; i++) C[(size_t)fr * t + i] = ark(r, i);
        }
        Mpre = M;
    }
    S.sparse = sparse ? 1 : 0;

    auto push = [&](const FeVec& v) {
        int off = (int)(S.consts.size() / 4);
        for (const Fe& e : v) S.consts.insert(S.consts.end(), e.l, e.l + 4);
        return off;
    };
    S.off_c = push(C);
    S.off_m = push(M);
    S.off_mpre = push(Mpre);
    S.off_cp0 = push(Cp0);
    S.off_pc = push(pc);
    S.off_sp = push(sp);
    if (sparse) arkp.clear();      // the original partial-round constants are read by the dense form only
    S.off_arkp = push(arkp);
    {
        Fe pm;
        memcpy(pm.l, F.p, 32);
        S.off_mod = push(FeVec(1, pm));
    }
    {
        Fe y = F.one(), b = C.empty() ? F.zero() : C[0];                       // C[0][0]^alpha (alpha = 0: the constant one, as the kernels' S-box)
        for (u64 e = P.alpha; e; e >>= 1) {
            if (e & 1) y = F.mul(y, b);
            b = F.mul(b, b);
        }
        S.off_sc0 = push(FeVec(1, y));
    }
    FeVec rrows, rk, rr;
    if (sparse && t == 3 && detail::derive_recurrence(F, rp, sp, pc, rrows, rk, rr)) {
        S.recur = 1;
        S.off_rc = push(rrows);
        S.off_rk = push(rk);
        S.off_rr = push(rr);
    }
    S.n_elems = (int)(S.consts.size() / 4);
    return S;
}

// The kernels' view of a schedule.
inline PoseidonDev make_dev(const PoseidonSchedule& S) {
    PoseidonDev D;
    D.t = S.t; D.rate = S.rate; D.cap = S.capacity; D.rf = S.rf; D.rp = S.rp; D.sparse = S.sparse; D.alpha = S.alpha;
    D.off_c = S.off_c; D.off_m = S.off_m; D.off_mpre = S.off_mpre; D.off_cp0 = S.off_cp0; D.off_pc = S.off_pc;
    D.off_sp = S.off_sp; D.off_arkp = S.off_arkp; D.off_mod = S.off_mod; D.off_sc0 = S.off_sc0; D.n_elems = S.n_elems; D.zero = 0;
    D.recur = S.recur; D.off_rc = S.off_rc; D.off_rk = S.off_rk; D.off_rr = S.off_rr;
    return D;
}

}  // namespace host
}  // namespace cpb
