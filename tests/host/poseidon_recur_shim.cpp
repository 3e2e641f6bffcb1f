// CPU build of the device Poseidon code (crypto_primitives_b200/csrc/poseidon.cuh, PTX primitives emulated) with the schedule
// exactly as the library hands it to the kernels (host::make_dev), i.e. with the lane-0 recurrence of the t = 3 partial rounds
// whenever derive_schedule finds one.  Lets tests/test_poseidon_recurrence.py check the recurrence bit-for-bit against the oracle
// through every entry point that runs pos_permute_split.  Not part of the product.
#include "../../crypto_primitives_b200/csrc/poseidon_host.hpp"
#include <cstring>
#include <vector>
using namespace cpb;

static host::PoseidonSchedule schedule(int field, int rate, int cap, int rf, int rp, unsigned long long alpha, const uint64_t* ark,
                                       const uint64_t* mds) {
    host::Field F(host::field_modulus(field));
    host::PoseidonParams P;
    P.rate = rate; P.capacity = cap; P.full_rounds = rf; P.partial_rounds = rp; P.alpha = alpha;
    const int t = rate + cap;
    P.ark.resize((size_t)(rf + rp) * t);
    P.mds.resize((size_t)t * t);
    memcpy(P.ark.data(), ark, P.ark.size() * 32);
    memcpy(P.mds.data(), mds, P.mds.size() * 32);
    return host::derive_schedule(F, P, true);
}

// mode 0: CRH as the library's kernel selection runs it (one permutation with the sponge's hints when len <= rate, else the
// sponge); mode 1: always the generic sponge (no hints), n_out outputs; mode 2: bare permutation of t-element states.
template <class F, int T>
static void run(int mode, const PoseidonDev& D, const u32* cs, const u32* in, long len, long n_out, long n, u32* out) {
    u32 pm[8];
    ld_elem(pm, cs + 8 * D.off_mod);
    for (long i = 0; i < n; i++) {
        if (mode == 0 && len <= D.rate && D.cap >= 1) pos_hash_single<F, T>(out + 8 * i, 1, in + 8 * len * i, (int)len, D, cs, pm);
        else if (mode == 0) pos_crh<F, T>(out + 8 * i, in + 8 * len * i, len, D, cs, pm);
        else if (mode == 1) pos_sponge<F, T>(out + 8 * n_out * i, n_out, in + 8 * len * i, len, D, cs, pm);
        else {
            u32 s[T][8];
            for (int j = 0; j < T; j++) ld_elem(s[j], in + 8 * (T * i + j));
            pos_permute<F, T>(s, D, cs, pm);
            for (int j = 0; j < T; j++) st_elem(out + 8 * (T * i + j), s[j]);
        }
    }
}

template <class F>
static int run_t(int mode, const PoseidonDev& D, const u32* cs, const u32* in, long len, long n_out, long n, u32* out) {
    switch (D.t) {
        case 2: run<F, 2>(mode, D, cs, in, len, n_out, n, out); return 0;
        case 3: run<F, 3>(mode, D, cs, in, len, n_out, n, out); return 0;
        case 4: run<F, 4>(mode, D, cs, in, len, n_out, n, out); return 0;
    }
    return 1;
}

// returns -1 on error, else the schedule's `recur` flag
extern "C" int recur_run(int field, int mode, int rate, int cap, int rf, int rp, unsigned long long alpha, const uint64_t* ark,
                         const uint64_t* mds, const uint64_t* in, long len, long n_out, long n, uint64_t* out) {
    if (!host::field_modulus(field)) return -1;
    host::PoseidonSchedule S = schedule(field, rate, cap, rf, rp, alpha, ark, mds);
    PoseidonDev D = host::make_dev(S);
    const u32* cs = reinterpret_cast<const u32*>(S.consts.data());
    const u32* i32 = reinterpret_cast<const u32*>(in);
    u32* o32 = reinterpret_cast<u32*>(out);
    int rc = 1;
    switch (field) {
        case 0: rc = run_t<Bls12_381_Fr>(mode, D, cs, i32, len, n_out, n, o32); break;
        case 1: rc = run_t<Bn254_Fr>(mode, D, cs, i32, len, n_out, n, o32); break;
        case 2: rc = run_t<Jubjub_Fr>(mode, D, cs, i32, len, n_out, n, o32); break;
        case 3: rc = run_t<Bls12_377_Fr>(mode, D, cs, i32, len, n_out, n, o32); break;
    }
    return rc ? -1 : S.recur;
}

// The recurrence section of the schedule: rows (3 x 5), ck (rp), rr (10); also sparse (returned in flags[0]) and recur (flags[1]).
extern "C" int recur_schedule(int field, int rate, int cap, int rf, int rp, unsigned long long alpha, const uint64_t* ark,
                              const uint64_t* mds, uint64_t* rows, uint64_t* ck, uint64_t* rr, int* flags) {
    if (!host::field_modulus(field)) return -1;
    host::PoseidonSchedule S = schedule(field, rate, cap, rf, rp, alpha, ark, mds);
    flags[0] = S.sparse;
    flags[1] = S.recur;
    if (S.recur) {
        memcpy(rows, S.consts.data() + 4 * (size_t)S.off_rc, 15 * 32);
        memcpy(ck, S.consts.data() + 4 * (size_t)S.off_rk, (size_t)rp * 32);
        memcpy(rr, S.consts.data() + 4 * (size_t)S.off_rr, 10 * 32);
    }
    return 0;
}
