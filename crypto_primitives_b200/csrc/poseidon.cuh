// poseidon.cuh -- the Poseidon permutation and the CRH / two-to-one evaluation built on it,
// one hash per thread, whole state in registers.
//
// Device counterpart of PoseidonSponge::permute (R/sponge/poseidon/mod.rs:66-121) and of
// crh::poseidon::{CRH::evaluate, TwoToOneCRH::compress} (R/crh/poseidon/mod.rs:30-40,66-79),
// i.e. new sponge -> absorb (mod.rs:124-153) -> squeeze one native element (mod.rs:323-345).
// Executes the schedule produced by host::derive_schedule (poseidon_host.hpp): same function,
// sparse partial rounds.  Everything here is CPB_HD so tests/host can run the identical code
// on the CPU (PTX primitives emulated) against the oracle before any GPU time is spent.
#pragma once
#include "fp.cuh"

namespace cpb {

struct PoseidonDev {
    int t, rate, cap, rf, rp, sparse;
    u64 alpha;
    int off_c, off_m, off_mpre, off_cp0, off_pc, off_sp, off_arkp, off_mod, off_sc0, n_elems;
    // Always 0.  Kernels add threadIdx.x * zero to the shared-memory address of every constant so
    // that ptxas keeps multiplier operands in ordinary registers: values loaded from a
    // warp-uniform address are promoted to uniform registers, and a multiply-add with a
    // uniform-register factor is emitted as IMAD.X + IMAD.HI.U32.X instead of one IMAD.WIDE.U32.X.
    int zero;
    // Lane-0 recurrence of the partial rounds (host::derive_recurrence); off unless the schedule sets it.
    int recur = 0, off_rc = 0, off_rk = 0, off_rr = 0;
};

template <class F, int T> CPB_HD void pos_add_vec(u32 (&s)[T][8], const u32* c) {
#pragma unroll
    for (int i = 0; i < T; i++) {
        u32 k[8];
        ld_elem(k, c + 8 * i);
        fp_add<F>(s[i], s[i], k);
    }
}

// (s0, s1, ..., s_{T-1}) <- (s1, ..., s_{T-1}, s0).  Lets a rolled loop visit every lane while
// the state stays in registers (register files cannot be indexed dynamically); a rotation is
// 8T moves against ~900 instructions of work per visit.
template <int T> CPB_HD void pos_rotl(u32 (&s)[T][8]) {
    u32 tmp[8];
    fp_copy(tmp, s[0]);
#pragma unroll
    for (int i = 0; i + 1 < T; i++) fp_copy(s[i], s[i + 1]);
    fp_copy(s[T - 1], tmp);
}

// x^alpha, left-to-right binary.  For the arkworks S-box exponents (3, 5, 17, 257 = 2^k+1)
// this is k squarings and one multiplication -- the optimal chain -- from a single pair of
// inlined multiplier bodies, which keeps the kernel's instruction footprint small.
// lazy (F::LAZY5 fields, alpha = 5, canonical x): the three products skip their conditional subtraction; x^2 < 1.19p, x^4 < 1.27p,
// x^5 < 1.24p for p/R < 0.19 -- what the dense rows take with EX = 1 (3 * 1.24 p < 4p).
template <class F> CPB_HD void pos_sbox(u32* x, u64 alpha, int top_bit, const u32* pm, bool lazy = false) {
    u32 x0[8];
    fp_copy(x0, x);
#pragma unroll 1
    for (int i = top_bit - 1; i >= 0; i--) {
        if constexpr (F::LAZY5) {
            fp_sqr_rt<F>(x, x, pm, lazy);
            if ((alpha >> i) & 1) fp_mul_rt<F>(x, x, x0, pm, lazy);
        } else {
            fp_sqr<F>(x, x, pm);
            if ((alpha >> i) & 1) fp_mul<F>(x, x, x0, pm);
        }
    }
}

// The permutation, one rolled loop over all RF+RP rounds with a single instance of each
// arithmetic body:  [add round constants] -> S-box on T lanes or lane 0 -> linear layer as
// lazy dot products (T rows of a dense matrix, or the one dense row of the sparse form
// followed by the rank-one column update).
// 1: every field uses pos_permute_split; 0: none; unset: per field (F::SPLIT_ROUNDS).  Measured on the t = 3 kernels:
// BN254 Fr (57 partial rounds, alpha = 5) +3 %; BLS12-381 Fr (31 partial rounds, alpha = 17) -1 % before and +0.9 %
// after the squaring lost 51 instructions -- so every field uses the split form now.
#ifdef CPB_POS_SPLIT
#define CPB_POS_SPLIT_FOR(F) (CPB_POS_SPLIT != 0)
#else
#define CPB_POS_SPLIT_FOR(F) (F::SPLIT_ROUNDS)
#endif
#ifndef CPB_SBOX5
#define CPB_SBOX5 1        // straight-line x^5 in the partial-round loop (+0.6 % on BN254 Fr; other exponents use the bit loop)
#endif
#ifndef CPB_COL_UNROLL_MAX
#define CPB_COL_UNROLL_MAX 4
#endif
#ifndef CPB_POS_RECUR
#define CPB_POS_RECUR 1    // t = 3: partial rounds as the lane-0 recurrence when the schedule has one (pos_partial_recur)
#endif

// Sparse schedules only: the same permutation with the partial rounds in a loop of their own.  The two
// halves of the full rounds share one body through a two-trip outer loop, so there is still a single
// instance of the dense round; the partial-round loop has no full/partial selection and no lane
// rotation, i.e. none of the register shuffles the merged loop pays at its control-flow joins.
//
// Two things the sponge knows and a bare permutation does not (PermuteHint): (i) in the first permutation of a fresh sponge the
// capacity lane 0 is zero, so its first S-box input is the round constant itself and S(c) comes from the schedule (off_sc0);
// (ii) when the permutation's result is only squeezed (no further permutation), the last round needs just the rows of the lanes
// that are read -- one of t for CRH::evaluate / TwoToOneCRH::compress.  Both leave every value that is used bit-identical.
struct PermuteHint {
    int lane0_zero;        // != 0: state lane 0 is zero on entry
    unsigned need;         // bit i set: lane i of the result is read; everything else is dead
};

// The partial rounds of a t = 3 sparse schedule as the lane-0 recurrence of host::derive_recurrence.  Per round: the S-box, then
// ONE five-term lazy dot over the history h = (y_k, y_k-1, y_k-2, x_k, x_k-1) -- 5 products and 1 Montgomery reduction, where the
// sparse form's 3-term row and two reduced column products take 5 products and 3 reductions (BN254 Fr: 384 instead of 512 wide
// multiply-adds).  Lanes 1, 2 are not carried through the rounds: the first two rounds read them from the history, and after the
// last round two 4-term dots rebuild them, so the state leaves bit for bit as the sparse rounds leave it.
// Ranges with `lazy` (BN254 Fr, alpha = 5; tests/test_poseidon_recurrence.py): x = d + c < 2p is kept unreduced except after the
// last round, the S-box output y < 1.6p, so the history sums below 8.8p (EX = 4: nine canonical terms' worth) and the terms of the
// rebuild below 6.2p (EX = 3).  Without it every value is canonical (EX = 0).
template <class F, bool LZ> CPB_HD void pos_partial_recur(u32 (&s)[3][8], const PoseidonDev& P, const u32* cs, const u32* pm, bool lazy,
                                                          int top_bit) {
    constexpr int EXH = LZ ? 4 : 0, EXR = LZ ? 3 : 0;
    const bool alpha_zero = P.alpha == 0;
    u32 h[5][8];
    fp_copy(h[1], s[1]);
    fp_copy(h[2], s[2]);
    fp_copy(h[3], s[0]);
    fp_zero(h[4]);
    const u32* row = cs + 8 * P.off_rc;      // rounds 0 and 1 have rows of their own, every later round uses the third
    const u32* ck = cs + 8 * P.off_rk;
#pragma unroll 1
    for (int k = 0; k < P.rp; k++, ck += 8) {
        fp_copy(h[0], h[3]);
#if CPB_SBOX5
        if (P.alpha == 5) {                   // straight-line x^5
            u32 x2[8];
            fp_sqr<F, LZ>(x2, h[0], pm);
            fp_sqr<F, LZ>(x2, x2, pm);
            fp_mul<F, LZ>(h[0], x2, h[0], pm);
        } else
#endif
        if (alpha_zero) fp_one<F>(h[0]);
        else pos_sbox<F>(h[0], P.alpha, top_bit, pm);
        u32 d[8], c[8];
        fp_dot<F, 5, EXH>(d, h, row, pm);
        if (k < 2) row += 8 * 5;
        ld_elem(c, ck);
        fp_copy(h[2], h[1]);
        fp_copy(h[1], h[0]);
        fp_copy(h[4], h[3]);
        if (lazy && k + 1 < P.rp) fp_add_noreduce(h[3], d, c);
        else fp_add<F>(h[3], d, c);
    }
    // h[1..4] = (y_rp-1, y_rp-2, lane 0 after the last round, x_rp-1)
    u32 g[4][8], c[8];
#pragma unroll
    for (int i = 0; i < 4; i++) fp_copy(g[i], h[i + 1]);
    const u32* rr = cs + 8 * P.off_rr;
    fp_copy(s[0], h[3]);
    fp_dot<F, 4, EXR>(s[1], g, rr, pm);
    ld_elem(c, rr + 8 * 8);
    fp_add<F>(s[1], s[1], c);
    fp_dot<F, 4, EXR>(s[2], g, rr + 8 * 4, pm);
    ld_elem(c, rr + 8 * 9);
    fp_add<F>(s[2], s[2], c);
}

template <class F, int T> CPB_HD void pos_permute_split(u32 (&s)[T][8], const PoseidonDev& P, const u32* cs, const u32* pm, const PermuteHint& H) {
    const int half = P.rf / 2;
    int top_bit = 0;
    for (int i = 63; i > 0; i--)
        if ((P.alpha >> i) & 1) { top_bit = i; break; }
    const bool alpha_zero = P.alpha == 0;
    // Lazy reduction (F::LAZY5: p/2^256 <= 0.19, i.e. BN254 Fr; alpha = 5; widths whose (T+1)-term rows need no overflow word).
    // Full rounds: the S-box of a canonical x skips its three conditional subtractions (x^5 < 1.24p, see pos_sbox) and the dense
    // rows take the T unreduced lanes as EX = 1 (T * 1.24p < (T+1)*p for T <= 4), returning canonical values.
    constexpr bool LZ = F::LAZY5 && !detail::dot_needs_x<F, T + 1>() && T <= 4;
    static_assert(!F::LAZY5 || 100 * ((u64)F::P(7) + 1) <= 19 * ((u64)1 << LIMB_BITS), "LAZY5 needs p/2^256 <= 0.19");
    const bool lazy = LZ && CPB_SBOX5 && P.alpha == 5;
    u32 n[T][8];
#pragma unroll
    for (int i = 0; i < T; i++) fp_zero(n[i]);
#pragma unroll 1
    for (int phase = 0; phase < 2; phase++) {
        const int cnt = phase == 0 ? half : P.rf - half;   // odd RF: floor(RF/2) rounds before, ceil(RF/2) after (mod.rs:98-121)
#pragma unroll 1
        for (int q = 0; q < cnt; q++) {
            pos_add_vec<F, T>(s, cs + 8 * (P.off_c + (phase * half + q) * T));
            const int first_j = (H.lane0_zero != 0 && phase == 0 && q == 0) ? 0 : -1;     // the lane whose S-box is the schedule constant
            const unsigned need = (phase == 1 && q == cnt - 1) ? H.need : ~0u;            // rows of this round that are used
#pragma unroll 1
            for (int j = 0; j < T; j++) {
                if (j == first_j) ld_elem(s[0], cs + 8 * P.off_sc0);         // S(0 + c) of the schedule
                else if (alpha_zero) fp_one<F>(s[0]);
                else pos_sbox<F>(s[0], P.alpha, top_bit, pm, lazy);
                pos_rotl<T>(s);
            }
            const u32* rows = cs + 8 * ((phase == 0 && q == half - 1) ? P.off_mpre : P.off_m);
            // (re)defined every round: the collector's old values are shifted through but never used, and without this they
            // would count as live across the partial rounds
#pragma unroll
            for (int i = 0; i < T; i++) fp_zero(n[i]);
#pragma unroll 1
            for (int i = 0; i < T; i++) {
                u32 d[8];
                fp_zero(d);
                if ((need >> i) & 1u) fp_dot<F, T, LZ ? 1 : 0>(d, s, rows + 8 * T * i, pm);
#pragma unroll
                for (int k = 0; k + 1 < T; k++) fp_copy(n[k], n[k + 1]);
                fp_copy(n[T - 1], d);
            }
#pragma unroll
            for (int i = 0; i < T; i++) fp_copy(s[i], n[i]);
        }
        if (phase == 0 && P.rp > 0) {
            pos_add_vec<F, T>(s, cs + 8 * P.off_cp0);
            if constexpr (T == 3 && CPB_POS_RECUR != 0) {
                if (P.recur) {
                    pos_partial_recur<F, LZ>(s, P, cs, pm, lazy, top_bit);
                    continue;                 // (the end of phase 0)
                }
            }
            const u32* row = cs + 8 * P.off_sp;
            const u32* pc = cs + 8 * (P.off_pc + 1);
            // Partial rounds, lazy lane 0: lane 0 lives in [0, 2p) from the constant
            // addition to the end of the round.  With a, b < 2p the Montgomery product (a*b + M*p)/R is below p*(4p/R + 1) <= 2p,
            // so x^2, x^4, x^5 need no conditional subtraction, nor does x = d + c (d, c < p).  Consumers: the row product
            // takes sum_j a_j < (T+1)*p (EX = 1: same code as T canonical terms when (T+2)*p <= 2^256, which is the
            // condition below) and returns a canonical d; the column products v_j * y are ordinary multiplications whose full
            // operand y + p stays below 2^256 and whose results are reduced, so lanes 1.. stay canonical.  Saves 4 conditional
            // subtractions (68 instructions) per partial round; bit-identical outputs.
#pragma unroll 1
            for (int k = 0; k < P.rp; k++, row += 8 * (2 * T - 1), pc += 8) {
#if CPB_SBOX5
                if (P.alpha == 5) {                   // straight-line x^5
                    u32 x2[8];
                    fp_sqr<F, LZ>(x2, s[0], pm);
                    fp_sqr<F, LZ>(x2, x2, pm);
                    fp_mul<F, LZ>(s[0], x2, s[0], pm);
                } else
#endif
                if (alpha_zero) fp_one<F>(s[0]);
                else pos_sbox<F>(s[0], P.alpha, top_bit, pm);
                u32 d[8];
                fp_dot<F, T, LZ ? 1 : 0>(d, s, row, pm);
                const u32* v = row + 8 * T;
                if (T <= CPB_COL_UNROLL_MAX) {
#pragma unroll
                    for (int j = 1; j < T; j++) {
                        u32 c[8], tmp[8];
                        ld_elem(c, v + 8 * (j - 1));
                        fp_mul<F>(tmp, s[0], c, pm);
                        fp_add<F>(s[j], s[j], tmp);
                    }
                } else {
#pragma unroll 1
                    for (int j = 1; j < T; j++) {
                        u32 c[8], tmp[8];
                        ld_elem(c, v + 8 * (j - 1));
                        fp_mul<F>(tmp, s[0], c, pm);
                        fp_add<F>(s[1], s[1], tmp);
                        fp_copy(tmp, s[1]);
#pragma unroll
                        for (int q = 1; q + 1 < T; q++) fp_copy(s[q], s[q + 1]);
                        fp_copy(s[T - 1], tmp);
                    }
                }
                if (k + 1 < P.rp) {
                    u32 c[8];
                    ld_elem(c, pc);
                    if (lazy) fp_add_noreduce(s[0], d, c);
                    else fp_add<F>(s[0], d, c);
                } else {
                    fp_copy(s[0], d);
                }
            }
        }
    }
}

template <class F, int T> CPB_HD void pos_permute(u32 (&s)[T][8], const PoseidonDev& P, const u32* cs, const u32* pm,
                                                  const PermuteHint& H = PermuteHint{0, ~0u}) {
    if constexpr (CPB_POS_SPLIT_FOR(F)) {
        if (P.sparse) {
            pos_permute_split<F, T>(s, P, cs, pm, H);
            return;
        }
    }
    const int half = P.rf / 2, total = P.rf + P.rp;
    int top_bit = 0;
    for (int i = 63; i > 0; i--)
        if ((P.alpha >> i) & 1) { top_bit = i; break; }
    const bool alpha_zero = P.alpha == 0;
    // row collector of the dense layers; defined once so that the shift below never reads an
    // indeterminate value (with the array declared inside the loop nvcc miscompiled t >= 5)
    u32 n[T][8];
#pragma unroll
    for (int i = 0; i < T; i++) fp_zero(n[i]);
#pragma unroll 1
    for (int r = 0; r < total; r++) {
        const bool full = r < half || r >= half + P.rp;
        const int k = r - half;                       // partial-round index when !full
        // --- round constants
        if (full) {
            const int fr = r < half ? r : r - P.rp;
            pos_add_vec<F, T>(s, cs + 8 * (P.off_c + fr * T));
        } else if (!P.sparse) {
            pos_add_vec<F, T>(s, cs + 8 * (P.off_arkp + k * T));
        } else if (k == 0) {
            pos_add_vec<F, T>(s, cs + 8 * P.off_cp0);
        }
        // --- S-box
        const int lanes = full ? T : 1;
#pragma unroll 1
        for (int j = 0; j < lanes; j++) {
            if (alpha_zero) fp_one<F>(s[0]);
            else pos_sbox<F>(s[0], P.alpha, top_bit, pm);
            if (full) pos_rotl<T>(s);
        }
        // --- linear layer
        const bool dense = full || !P.sparse;
        const u32* rows = dense ? cs + 8 * ((full && r == half - 1) ? P.off_mpre : P.off_m)
                                : cs + 8 * (P.off_sp + k * (2 * T - 1));
        const int nrows = dense ? T : 1;
        u32 d[8];
#pragma unroll 1
        for (int i = 0; i < nrows; i++) {
            fp_dot<F, T>(d, s, rows + 8 * T * i, pm);
            if (dense) {                        // collect row i; after T iterations n[i] holds row i
#pragma unroll
                for (int q = 0; q + 1 < T; q++) fp_copy(n[q], n[q + 1]);
                fp_copy(n[T - 1], d);
            }
        }
        if (dense) {
#pragma unroll
            for (int i = 0; i < T; i++) fp_copy(s[i], n[i]);
        } else {
            // s_j += v_j * s_0 for j >= 1 (old s_0), then s_0 <- row product d (+ next lane-0 constant)
            const u32* v = rows + 8 * T;
            if (T <= CPB_COL_UNROLL_MAX) {
#pragma unroll
                for (int j = 1; j < T; j++) {
                    u32 c[8], tmp[8];
                    ld_elem(c, v + 8 * (j - 1));
                    fp_mul<F>(tmp, s[0], c, pm);
                    fp_add<F>(s[j], s[j], tmp);
                }
            } else {
#pragma unroll 1
                for (int j = 1; j < T; j++) {
                    u32 c[8], tmp[8];
                    ld_elem(c, v + 8 * (j - 1));
                    fp_mul<F>(tmp, s[0], c, pm);
                    fp_add<F>(s[1], s[1], tmp);
                    fp_copy(tmp, s[1]);        // rotate lanes 1..T-1
#pragma unroll
                    for (int q = 1; q + 1 < T; q++) fp_copy(s[q], s[q + 1]);
                    fp_copy(s[T - 1], tmp);
                }
            }
            if (k + 1 < P.rp) {
                u32 c[8];
                ld_elem(c, cs + 8 * (P.off_pc + k + 1));
                fp_add<F>(s[0], d, c);
            } else {
                fp_copy(s[0], d);
            }
        }
    }
}

// New sponge -> absorb `len` elements at `in` -> squeeze `n_out` native elements to `out` (8 limbs each).
// n_out == 1 is crh::poseidon::CRH::evaluate (R/crh/poseidon/mod.rs:30-40).  Absorb semantics of
// R/sponge/poseidon/mod.rs:124-153: fill `rate` lanes, permute while more input remains; the squeeze
// (mod.rs:156-186, 323-345) permutes once from Absorbing mode (so an empty input still costs one
// permutation), then emits `rate` lanes per permutation.
template <class F, int T>
CPB_HD void pos_sponge(u32* out, long n_out, const u32* in, long len, const PoseidonDev& P, const u32* cs, const u32* pm) {
    u32 s[T][8];
#pragma unroll
    for (int i = 0; i < T; i++) fp_zero(s[i]);
    const int rate = P.rate, cap = P.cap;
    const long nblocks = len <= rate ? 1 : (len + rate - 1) / rate;
    const long nsq = n_out <= rate ? 1 : (n_out + rate - 1) / rate;
#pragma unroll 1
    for (long b = 0; b < nblocks + nsq - 1; b++) {
        if (b < nblocks) {
            const long pos = b * rate;
            const long rem = len - pos;
            const int cnt = rem > rate ? rate : (int)rem;
#pragma unroll
            for (int i = 0; i < T; i++) {
                int lane = i - cap;
                if (lane >= 0 && lane < cnt) {
                    u32 e[8];
                    ld_elem(e, in + 8 * (pos + lane));
                    fp_add<F>(s[i], s[i], e);
                }
            }
        }
        pos_permute<F, T>(s, P, cs, pm);
        if (b >= nblocks - 1) {
            const long q = b - (nblocks - 1);          // squeeze block index
            const long left = n_out - q * rate;
            const int cnt = left > rate ? rate : (int)left;
#pragma unroll
            for (int i = 0; i < T; i++) {
                int lane = i - cap;
                if (lane >= 0 && lane < cnt) st_elem(out + 8 * (q * rate + lane), s[i]);
            }
        }
    }
}

// The one-permutation case of pos_sponge (len <= rate, 1 <= n_out <= rate, capacity >= 1) -- every hash of a Merkle build and
// every CRH::evaluate / TwoToOneCRH::compress of up to `rate` elements -- with the permutation told what the sponge knows
// (PermuteHint): lane 0 enters as zero, and only lanes cap .. cap+n_out-1 of the result are read.
template <class F, int T>
CPB_HD void pos_hash_single(u32* out, int n_out, const u32* in, int len, const PoseidonDev& P, const u32* cs, const u32* pm) {
    u32 s[T][8];
    const int cap = P.cap;
#pragma unroll
    for (int i = 0; i < T; i++) {
        const int lane = i - cap;
        if (lane >= 0 && lane < len) ld_elem(s[i], in + 8 * lane);
        else fp_zero(s[i]);
    }
    pos_permute<F, T>(s, P, cs, pm, PermuteHint{1, ((1u << n_out) - 1u) << cap});
#pragma unroll
    for (int i = 0; i < T; i++) {
        const int lane = i - cap;
        if (lane >= 0 && lane < n_out) st_elem(out + 8 * lane, s[i]);
    }
}

template <class F, int T> CPB_HD void pos_crh(u32* out, const u32* in, long len, const PoseidonDev& P, const u32* cs, const u32* pm) {
    pos_sponge<F, T>(out, 1, in, len, P, cs, pm);
}

// Path::verify (R/merkle_tree/mod.rs:172-212) for the field-leaf Config: hash the leaf, fold the
// authentication path bottom-up choosing sides by the index bits, compare with the root.
// auth_path: plen elements ordered root side first (as Path.auth_path).  PL/PN, cl/cn: leaf / node schedules.
template <class F, int T>
CPB_HD bool pos_verify_path(const u32* leaf, long leaf_len, const u32* sibling, const u32* auth_path, int plen, unsigned long long index,
                            const u32* root, const PoseidonDev& PL, const u32* cl, const PoseidonDev& PN, const u32* cn, const u32* pm) {
    alignas(16) u32 pair[16];        // read back through 128-bit loads
    u32 cur[8];
    pos_crh<F, T>(cur, leaf, leaf_len, PL, cl, pm);
    u32 sib[8];
    ld_elem(sib, sibling);
#pragma unroll 1
    for (int level = plen; level >= 0; level--) {
        const bool right = (index & 1ull) != 0;       // computed node is the right child
#pragma unroll
        for (int j = 0; j < 8; j++) {
            pair[j] = right ? sib[j] : cur[j];
            pair[8 + j] = right ? cur[j] : sib[j];
        }
        pos_crh<F, T>(cur, pair, 2, PN, cn, pm);
        index >>= 1;
        if (level > 0) ld_elem(sib, auth_path + 8 * (level - 1));
    }
    u32 r[8];
    ld_elem(r, root);
    return fp_eq(cur, r);
}

}  // namespace cpb
