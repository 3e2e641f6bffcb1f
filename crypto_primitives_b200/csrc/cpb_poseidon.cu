// cpb_poseidon.cu -- CUDA kernels + C-ABI for the Poseidon part of the hot path and the
// field-leaf Merkle build on top of it (include/cpb200.h).
//
// Kernels (sm_100a, integer pipe, no tensor cores):
//   k_poseidon_crh      one CRH::evaluate per thread (R/crh/poseidon/mod.rs:30-40); with len==2
//                       it is also TwoToOneCRH::compress (:66-79) and one Merkle level
//                       (R/merkle_tree/mod.rs:454-515), because a level's children are contiguous
//                       in the heap-ordered node array.
//   k_poseidon_permute  one bare permutation per thread (R/sponge/poseidon/mod.rs:98-121).
//   k_field_convert     canonical <-> Montgomery.
// Round constants / MDS / sparse rows are staged into shared memory with one TMA bulk copy per
// CTA; inputs are read with 128-bit loads; state lives in registers.
#include <cstdlib>
#include <vector>

#include "poseidon_kernels.cuh"

namespace cpb {

// ------------------------------------------------------------------------------ common impl
std::string& last_error_ref() {
    static thread_local std::string s;
    return s;
}
cpb_status fail(cpb_status st, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    return st;
}
void keep_pool_memory(int device) {
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
}
int sm_count(int device) {
    static int cache[64];
    static std::mutex mu;
    std::lock_guard<std::mutex> g(mu);
    if (device < 0 || device >= 64) return 148;
    if (!cache[device]) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
        cache[device] = v;
    }
    return cache[device];
}

template <class F>
__global__ void k_field_convert(const u32* __restrict__ in, u32* __restrict__ out, long n, int to_mont) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 a[8], k[8];
    ld_elem(a, in + 8 * i);
    if (to_mont) {
        // inputs < 2^256 may exceed p: subtract p while >= p (at most 6 times for a 252-bit p... bounded loop)
        for (int it = 0; it < 18; it++) {
            u32 t[8];
            t[0] = sub_cc(a[0], F::P(0));
#pragma unroll
            for (int j = 1; j < 8; j++) t[j] = subc_cc(a[j], F::P(j));
            u32 borrow = subc(0, 0);
            if (borrow) break;
            fp_copy(a, t);
        }
#pragma unroll
        for (int j = 0; j < 8; j++) k[j] = F::R2(j);
    } else {
        fp_zero(k);
        k[0] = 1;
    }
    u32 pm[8];
    fp_modulus<F>(pm);
    fp_mul<F>(a, a, k, pm);
    st_elem(out + 8 * i, a);
}

}  // namespace cpb

using namespace cpb;

using namespace cpb;

namespace cpb {
CPB_POS_WIDTHS(CPB_POS_EXTERN, Bls12_381_Fr)
CPB_POS_WIDTHS(CPB_POS_EXTERN, Bn254_Fr)
CPB_POS_WIDTHS(CPB_POS_EXTERN, Jubjub_Fr)
CPB_POS_WIDTHS(CPB_POS_EXTERN, Bls12_377_Fr)
CPB_POS_EXTERN_TEAM(Bls12_381_Fr)
CPB_POS_EXTERN_TEAM(Bn254_Fr)
CPB_POS_EXTERN_TEAM(Jubjub_Fr)
CPB_POS_EXTERN_TEAM(Bls12_377_Fr)
}  // namespace cpb

namespace {

#define CPB_CASE_T(F, T, M, ...) case T: return M<F, T>(__VA_ARGS__);
#define CPB_FOR_T(F, M, ...)                                                                                   \
    switch (c->dev.t) {                                                                                        \
        CPB_CASE_T(F, 2, M, __VA_ARGS__) CPB_CASE_T(F, 3, M, __VA_ARGS__) CPB_CASE_T(F, 4, M, __VA_ARGS__)     \
        CPB_CASE_T(F, 5, M, __VA_ARGS__) CPB_CASE_T(F, 6, M, __VA_ARGS__) CPB_CASE_T(F, 7, M, __VA_ARGS__)     \
        CPB_CASE_T(F, 8, M, __VA_ARGS__) CPB_CASE_T(F, 9, M, __VA_ARGS__)                                      \
    }                                                                                                          \
    break;
#define CPB_FOR_FIELD(M, ...)                                                        \
    switch (c->field_id) {                                                           \
        case CPB_BLS12_381_FR: CPB_FOR_T(Bls12_381_Fr, M, __VA_ARGS__)               \
        case CPB_BN254_FR: CPB_FOR_T(Bn254_Fr, M, __VA_ARGS__)                       \
        case CPB_JUBJUB_FR: CPB_FOR_T(Jubjub_Fr, M, __VA_ARGS__)                     \
        case CPB_BLS12_377_FR: CPB_FOR_T(Bls12_377_Fr, M, __VA_ARGS__)               \
    }

// Largest level (in hashes) handled by the four-warp tree-top kernel: beyond ~6000 hashes the GPU's 592 warp
// schedulers are all busy with one hash per thread anyway, and the kernel's grid is capped at 128 CTAs of 32 hashes.
// CPB_TEAM_MAX overrides (0 disables; values above 4096 are clamped).
size_t team_max() {
    static long v = -1;
    if (v < 0) {
        const char* e = getenv("CPB_TEAM_MAX");
        v = e ? atol(e) : 4096;
        if (v > 4096) v = 4096;
        if (v < 0) v = 0;
    }
    return (size_t)v;
}
// Hand-over point of a subtree to the tree-top kernel when S subtrees are built concurrently: the four-warp kernel spends
// ~1.4x the multiplications of the one-hash-per-thread kernel to halve the dependent chain, which pays only once the GPU is
// latency-bound -- about 8192 hashes in flight over all streams (measured, profiles/r2_exp_team_max.txt: 2^21-leaf BN254
// tree, overhead over the bulk rate 2.9 / 2.3 / 1.9 / 2.0 ms for per-subtree limits 4096 / 2048 / 1024 / 256 at S = 8).
// CPB_TEAM_MAX, when set, is the per-subtree limit as given.
size_t team_max_for(size_t S) {
    if (getenv("CPB_TEAM_MAX")) return team_max();
    size_t v = 8192 / (S ? S : 1);
    return v < team_max() ? v : team_max();
}
bool team_capable(const cpb_poseidon_ctx* c) { return c->dev.t == 3 && c->dev.cap == 1 && c->dev.alpha >= 2; }

cpb_status launch_tree_top(cpb_poseidon_ctx* c, const TopJob& J, cudaStream_t st) {
    switch (c->field_id) {
        case CPB_BLS12_381_FR: return launch_tree_top_f<Bls12_381_Fr>(c, J, st);
        case CPB_BN254_FR: return launch_tree_top_f<Bn254_Fr>(c, J, st);
        case CPB_JUBJUB_FR: return launch_tree_top_f<Jubjub_Fr>(c, J, st);
        case CPB_BLS12_377_FR: return launch_tree_top_f<Bls12_377_Fr>(c, J, st);
    }
    return fail(CPB_BAD_PARAMS, "unknown field id %d", c->field_id);
}

}  // namespace

namespace cpb {
cpb_status launch_crh(cpb_poseidon_ctx* c, const u32* in, size_t len, u32* out, size_t n, cudaStream_t st, size_t n_out) {
    if (n == 0 || n_out == 0) return CPB_OK;
    if (team_capable(c) && len == 2 && n_out == 1 && n <= team_max()) {
        TopJob J;
        J.flat_in = in; J.flat_out = out; J.n_flat = (long)n;
        return launch_tree_top(c, J, st);
    }
    CPB_FOR_FIELD(launch_crh_ft, c, in, len, out, n_out, n, st)
    return fail(CPB_UNSUPPORTED, "state width t=%d is not built (this library: t = 2..9)", c->dev.t);
}
}  // namespace cpb

namespace {
cpb_status launch_verify(cpb_poseidon_ctx* c, cpb_poseidon_ctx* node, const u32* root, const u32* leaves, size_t leaf_len,
                         const u32* siblings, const u32* paths, int plen, const unsigned long long* indexes, unsigned char* ok,
                         size_t n, cudaStream_t st) {
    if (n == 0) return CPB_OK;
    CPB_FOR_FIELD(launch_verify_ft, c, node, root, leaves, leaf_len, siblings, paths, plen, indexes, ok, n, st)
    return fail(CPB_UNSUPPORTED, "state width t=%d is not built (this library: t = 2..9)", c->dev.t);
}
cpb_status launch_permute(cpb_poseidon_ctx* c, const u32* in, u32* out, size_t n, cudaStream_t st) {
    if (n == 0) return CPB_OK;
    CPB_FOR_FIELD(launch_permute_ft, c, in, out, n, st)
    return fail(CPB_UNSUPPORTED, "state width t=%d is not built (this library: t = 2..9)", c->dev.t);
}

}  // namespace

namespace cpb {

cpb_status check_ctx(const cpb_poseidon_ctx* c) {
    if (!c) return fail(CPB_NULL_POINTER, "null context");
    return CPB_OK;
}

// Inner levels of subtree k of S (S a power of two) from the leaf digests, heap order: global level l has
// 2^l nodes at [2^l - 1, 2^(l+1) - 1); subtree k owns the k-th 1/S of every level l >= log2 S
// (new_with_leaf_digest, R/merkle_tree/mod.rs:424-523).  S = 1, k = 0 is the whole tree.
cpb_status merkle_subtree_levels(cpb_poseidon_ctx* node, const u32* leaf_digests, size_t n, u32* nodes, size_t S, size_t k,
                                 cudaStream_t st, const MerkleHost* H, const ExchangeDev* X, int* small_from) {
    int h = 0;
    while (((size_t)1 << h) < n) h++;
    int lg = 0;
    while (((size_t)1 << lg) < S) lg++;
    const bool team = team_capable(node) && team_max() > 0;
    const size_t tmax = team_max_for(S);
    for (int l = h - 1; l >= lg; l--) {
        size_t cnt = ((size_t)1 << l) / S;
        if (team && cnt <= tmax) {
            // every remaining level of this subtree in ONE launch (k_poseidon_tree_top), optionally with the multi-GPU
            // root exchange and the replicated top levels fused in (X: only for the whole local tree, S == 1)
            TopJob J;
            J.leaf_digests = leaf_digests; J.nodes = nodes; J.h = h; J.lgS = lg; J.k = (long)k; J.l_start = l; J.l_end = lg;
            if (X && S == 1) J.x = *X;
            CPB_TRY(launch_tree_top(node, J, st));
            if (small_from) *small_from = l;                // the caller copies levels <= l out (all subtrees at once)
            else if (H)
                for (int q = l; q >= lg; q--) {
                    size_t c2 = ((size_t)1 << q) / S, off = (((size_t)1 << q) - 1) + k * c2;
                    CPB_CUDA(cudaMemcpyAsync(H->node_ptr(q, k * c2), nodes + 8 * off, c2 * 32, cudaMemcpyDeviceToHost, st));
                }
            return CPB_OK;
        }
        const u32* in = (l == h - 1) ? leaf_digests + 8 * (2 * k * cnt) : nodes + 8 * ((((size_t)1 << (l + 1)) - 1) + 2 * k * cnt);
        u32* out = nodes + 8 * ((((size_t)1 << l) - 1) + k * cnt);
        CPB_TRY(launch_crh(node, in, 2, out, cnt, st));
        // copy the level out right behind its kernel: the transfer overlaps the next levels and the other subtrees
        if (H) CPB_CUDA(cudaMemcpyAsync(H->node_ptr(l, k * cnt), out, cnt * 32, cudaMemcpyDeviceToHost, st));
    }
    if (X && S == 1) return fail(CPB_UNSUPPORTED, "the fused root exchange needs a rate-2, capacity-1 Poseidon two-to-one hash with alpha >= 2");
    return CPB_OK;
}
cpb_status merkle_levels(cpb_poseidon_ctx* node, const u32* leaf_digests, size_t n, u32* nodes, cudaStream_t st) {
    return merkle_subtree_levels(node, leaf_digests, n, nodes, 1, 0, st);
}

// Number of concurrently built subtrees: the top ~16 levels of a tree are latency-bound (fewer nodes than
// thread slots, one single-warp permutation latency each); building S subtrees on S streams hides the
// tails of all but the last behind bulk work.  CPB_MERKLE_STREAMS overrides (1 disables).
size_t merkle_streams(size_t n) {
    static int forced = -1;
    if (forced < 0) {
        const char* e = getenv("CPB_MERKLE_STREAMS");
        forced = e ? atoi(e) : 0;
    }
    size_t S = forced > 0 ? (size_t)forced : 8;
    if (S > 8) S = 8;
    while (S & (S - 1)) S &= S - 1;
    while (S > 1 && n / S < ((size_t)1 << 14)) S >>= 1;
    return S;
}

cpb_status ensure_side_streams(cpb_poseidon_ctx* c, size_t S) {
    std::lock_guard<std::mutex> lk(c->side_mu);
    for (size_t i = 0; i < S; i++)
        if (!c->side[i]) CPB_CUDA(cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking));
    return CPB_OK;
}

// leaf hashing (when leaves != nullptr) + all inner levels, S subtrees on S side streams joined on `st`
// X (optional): multi-GPU build -- after the local root, exchange the roots with the peers and compute the replicated top
// levels inside the last tree-top launch (ExchangeDev, poseidon_kernels.cuh).
cpb_status merkle_build_streams(cpb_poseidon_ctx* leaf, cpb_poseidon_ctx* node, const u32* leaves, size_t leaf_len, size_t n,
                                u32* leaf_nodes, u32* nodes, cudaStream_t st, const MerkleHost* H, const ExchangeDev* X) {
    size_t S = merkle_streams(n);
    if (S <= 1) {
        if (H && H->leaves && n * leaf_len) CPB_CUDA(cudaMemcpyAsync((void*)leaves, H->leaves, n * leaf_len * 32, cudaMemcpyHostToDevice, st));
        if (leaves) CPB_TRY(launch_crh(leaf, leaves, leaf_len, leaf_nodes, n, st));
        CPB_TRY(merkle_subtree_levels(node, leaf_nodes, n, nodes, 1, 0, st, H, X));
        if (H) CPB_CUDA(cudaMemcpyAsync(H->leaf_nodes, leaf_nodes, n * 32, cudaMemcpyDeviceToHost, st));
        return CPB_OK;
    }
    CPB_TRY(ensure_side_streams(node, S));
    int small_from = -1;                 // first (largest) level the subtrees' tree-top launches covered, when they ran
    cudaEvent_t start = nullptr, done[8] = {};
    CPB_CUDA(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
    cudaError_t e = cudaEventRecord(start, st);
    cpb_status rc = CPB_OK;
    size_t per = n / S;
    for (size_t k = 0; k < S && e == cudaSuccess && rc == CPB_OK; k++) {
        cudaStream_t sk = node->side[k];
        e = cudaStreamWaitEvent(sk, start, 0);
        if (e != cudaSuccess) break;
        if (H && H->leaves && leaf_len)
            e = cudaMemcpyAsync((void*)(leaves + 8 * leaf_len * (k * per)), H->leaves + 8 * leaf_len * (k * per), per * leaf_len * 32,
                                cudaMemcpyHostToDevice, sk);
        if (e != cudaSuccess) break;
        if (leaves) rc = launch_crh(leaf, leaves + 8 * leaf_len * (k * per), leaf_len, leaf_nodes + 8 * (k * per), per, sk);
        if (rc == CPB_OK && H)
            e = cudaMemcpyAsync(H->leaf_nodes + 8 * (k * per), leaf_nodes + 8 * (k * per), per * 32, cudaMemcpyDeviceToHost, sk);
        if (e != cudaSuccess) break;
        if (rc == CPB_OK) rc = merkle_subtree_levels(node, leaf_nodes, n, nodes, S, k, sk, H, nullptr, H ? &small_from : nullptr);
        if (rc != CPB_OK) break;
        e = cudaEventCreateWithFlags(&done[k], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventRecord(done[k], sk);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, done[k], 0);
    }
    cudaEventDestroy(start);
    for (size_t k = 0; k < S; k++)
        if (done[k]) cudaEventDestroy(done[k]);
    if (rc != CPB_OK) return rc;
    if (e != cudaSuccess) return fail(CPB_CUDA_ERROR, "merkle stream fork/join failed: %s", cudaGetErrorString(e));
    // top log2(S) levels on the caller's stream: one tree-top launch (with the fused exchange when X is given)
    int lg = 0, h = 0;
    while (((size_t)1 << lg) < S) lg++;
    while (((size_t)1 << h) < n) h++;
    if (team_capable(node) && team_max() > 0) {
        TopJob J;
        J.leaf_digests = leaf_nodes; J.nodes = nodes; J.h = h; J.lgS = 0; J.k = 0; J.l_start = lg - 1; J.l_end = 0;
        if (X) J.x = *X;
        CPB_TRY(launch_tree_top(node, J, st));
    } else {
        if (X) return fail(CPB_UNSUPPORTED, "the fused root exchange needs a rate-2, capacity-1 Poseidon two-to-one hash with alpha >= 2");
        for (int l = lg - 1; l >= 0; l--) {
            size_t cnt = (size_t)1 << l;
            CPB_TRY(launch_crh(node, nodes + 8 * ((((size_t)1 << (l + 1)) - 1)), 2, nodes + 8 * (cnt - 1), cnt, st));
        }
    }
    if (H) {
        // levels 0 .. small_from (the replicated top and, when the tree-top kernel ran, every small level of all the
        // subtrees): a contiguous prefix of the heap-ordered array -- one copy, or one per level for a shard (g > 0)
        const int last = small_from >= 0 ? small_from : lg - 1;
        if (H->g == 0) {
            CPB_CUDA(cudaMemcpyAsync(H->nodes, nodes, (((size_t)2 << last) - 1) * 32, cudaMemcpyDeviceToHost, st));
        } else {
            for (int l = last; l >= 0; l--)
                CPB_CUDA(cudaMemcpyAsync(H->node_ptr(l, 0), nodes + 8 * (((size_t)1 << l) - 1), ((size_t)1 << l) * 32, cudaMemcpyDeviceToHost, st));
        }
    }
    return CPB_OK;
}

// Kernel launches of merkle_build_streams(leaf != nullptr) for n leaves with this two-to-one context.
size_t count_launches(const cpb_poseidon_ctx* node, size_t n) {
    int h = 0;
    while (((size_t)1 << h) < n) h++;
    const size_t S = merkle_streams(n);
    int lg = 0;
    while (((size_t)1 << lg) < S) lg++;
    const bool team = team_capable(node) && team_max() > 0;
    size_t per_subtree = 1;                                   // the leaf hash
    for (int l = h - 1; l >= lg; l--) {
        size_t cnt = ((size_t)1 << l) / S;
        if (team && cnt <= team_max_for(S)) { per_subtree += 1; break; }
        per_subtree += 1;
    }
    size_t top = S > 1 ? (team ? 1 : (size_t)lg) : 0;
    return S * per_subtree + top;
}

bool pow2_gt1(size_t n) { return n > 1 && (n & (n - 1)) == 0; }

}  // namespace cpb

// ------------------------------------------------------------------------------ C ABI
extern "C" {

const char* cpb_last_error(void) { return last_error_ref().c_str(); }
int cpb_abi_version(void) { return CPB_ABI_VERSION; }
int cpb_version(void) { return 100; }

int cpb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; d++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

// Kernel launches one cpb_merkle_poseidon_build_dev over n leaves issues (leaf hash included): what bench.py reports as
// gpu_launches.  Mirrors merkle_build_streams above.
size_t cpb_merkle_poseidon_launch_count(const cpb_poseidon_ctx* node_ctx, size_t n) {
    if (!node_ctx || !pow2_gt1(n)) return 0;
    return count_launches(node_ctx, n);
}

// Page-lock a caller-owned host buffer so that the host-pointer entry points copy at full PCIe rate and overlap with
// hashing (a Rust Vec<Fr> is pageable; the shim can pin it once and reuse it).  cudaHostRegister / cudaHostUnregister.
cpb_status cpb_host_register(void* ptr, size_t bytes) {
    return cpb::guarded([&]() -> cpb_status {
    if (!ptr || !bytes) return fail(CPB_NULL_POINTER, "null buffer");
    CPB_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return CPB_OK;
    });
}
cpb_status cpb_host_unregister(void* ptr) {
    return cpb::guarded([&]() -> cpb_status {
    if (!ptr) return fail(CPB_NULL_POINTER, "null buffer");
    CPB_CUDA(cudaHostUnregister(ptr));
    return CPB_OK;
    });
}

cpb_status cpb_field_modulus(int field_id, uint64_t out[4]) {
    return cpb::guarded([&]() -> cpb_status {
    const uint64_t* m = host::field_modulus(field_id);
    if (!m) return fail(CPB_BAD_PARAMS, "unknown field id %d", field_id);
    if (!out) return fail(CPB_NULL_POINTER, "null out");
    memcpy(out, m, 32);
    return CPB_OK;
    });
}

static cpb_status field_convert(int field_id, int device, const uint64_t* in, uint64_t* out, size_t n, int to_mont) {
    if (!host::field_modulus(field_id)) return fail(CPB_BAD_PARAMS, "unknown field id %d", field_id);
    if (n == 0) return CPB_OK;
    if (!in || !out) return fail(CPB_NULL_POINTER, "null buffer");
    DeviceGuard g(device);
    if (!g.ok) return fail(CPB_NO_DEVICE, "cudaSetDevice(%d) failed", device);
    u32* d = nullptr;
    CPB_CUDA(cudaMalloc(&d, n * 32));
    cudaError_t e = cudaMemcpy(d, in, n * 32, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        int grid = (int)((n + 127) / 128);
        switch (field_id) {
            case 0: k_field_convert<Bls12_381_Fr><<<grid, 128>>>(d, d, (long)n, to_mont); break;
            case 1: k_field_convert<Bn254_Fr><<<grid, 128>>>(d, d, (long)n, to_mont); break;
            case 2: k_field_convert<Jubjub_Fr><<<grid, 128>>>(d, d, (long)n, to_mont); break;
            case 3: k_field_convert<Bls12_377_Fr><<<grid, 128>>>(d, d, (long)n, to_mont); break;
        }
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, d, n * 32, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(CPB_CUDA_ERROR, "field conversion failed: %s", cudaGetErrorString(e));
    return CPB_OK;
}
static cpb_status field_convert_dev(int field_id, int device, const uint64_t* in, uint64_t* out, size_t n, int to_mont, void* stream) {
    if (!host::field_modulus(field_id)) return fail(CPB_BAD_PARAMS, "unknown field id %d", field_id);
    if (n == 0) return CPB_OK;
    if (!in || !out) return fail(CPB_NULL_POINTER, "null buffer");
    DeviceGuard g(device);
    if (!g.ok) return fail(CPB_NO_DEVICE, "cudaSetDevice(%d) failed", device);
    cudaStream_t st = (cudaStream_t)stream;
    const u32* d_in = (const u32*)in;
    u32* d_out = (u32*)out;
    long left = (long)n, off = 0;
    while (left > 0) {                                  // grid.x limit is not an issue (2^31-1), but keep launches bounded
        long m = left < (1L << 28) ? left : (1L << 28);
        int grid = (int)((m + 127) / 128);
        switch (field_id) {
            case 0: k_field_convert<Bls12_381_Fr><<<grid, 128, 0, st>>>(d_in + 8 * off, d_out + 8 * off, m, to_mont); break;
            case 1: k_field_convert<Bn254_Fr><<<grid, 128, 0, st>>>(d_in + 8 * off, d_out + 8 * off, m, to_mont); break;
            case 2: k_field_convert<Jubjub_Fr><<<grid, 128, 0, st>>>(d_in + 8 * off, d_out + 8 * off, m, to_mont); break;
            case 3: k_field_convert<Bls12_377_Fr><<<grid, 128, 0, st>>>(d_in + 8 * off, d_out + 8 * off, m, to_mont); break;
        }
        CPB_CUDA(cudaGetLastError());
        left -= m; off += m;
    }
    return CPB_OK;
}
cpb_status cpb_field_to_montgomery_dev(int field_id, int device, const uint64_t* in, uint64_t* out, size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status { return field_convert_dev(field_id, device, in, out, n, 1, stream); });
}
cpb_status cpb_field_from_montgomery_dev(int field_id, int device, const uint64_t* in, uint64_t* out, size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status { return field_convert_dev(field_id, device, in, out, n, 0, stream); });
}
cpb_status cpb_field_to_montgomery(int field_id, int device, const uint64_t* in, uint64_t* out, size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    return field_convert(field_id, device, in, out, n, 1);
    });
}
cpb_status cpb_field_from_montgomery(int field_id, int device, const uint64_t* in, uint64_t* out, size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    return field_convert(field_id, device, in, out, n, 0);
    });
}

cpb_status cpb_poseidon_find_ark_and_mds(int field_id, uint64_t prime_bits, int rate, int full_rounds,
                                         int partial_rounds, int skip_matrices, uint64_t* ark_out, uint64_t* mds_out) {
    return cpb::guarded([&]() -> cpb_status {
    const uint64_t* mod = host::field_modulus(field_id);
    if (!mod) return fail(CPB_BAD_PARAMS, "unknown field id %d", field_id);
    if (!ark_out || !mds_out) return fail(CPB_NULL_POINTER, "null output");
    host::Field F(mod);
    if (prime_bits != (uint64_t)F.bits)   // assert_eq!(F::MODULUS_BIT_SIZE, prime_num_bits), grain_lfsr.rs:113
        return fail(CPB_BAD_PARAMS, "prime_bits %llu != MODULUS_BIT_SIZE %d", (unsigned long long)prime_bits, F.bits);
    if (rate < 1 || rate > 15 || full_rounds < 0 || partial_rounds < 0 || full_rounds > 1023 || partial_rounds > 1023 ||
        skip_matrices < 0)
        return fail(CPB_BAD_PARAMS, "bad shape");
    host::FeVec ark, mds;
    host::find_poseidon_ark_and_mds(F, prime_bits, rate, full_rounds, partial_rounds, skip_matrices, ark, mds);
    memcpy(ark_out, ark.data(), ark.size() * 32);
    memcpy(mds_out, mds.data(), mds.size() * 32);
    return CPB_OK;
    });
}

cpb_status cpb_poseidon_default_entry(int field_id, int rate, int optimized_for_weights, uint64_t* alpha, int* full_rounds,
                                      int* partial_rounds, int* skip_matrices) {
    return cpb::guarded([&]() -> cpb_status {
    host::DefaultEntry e;
    if (!host::default_entry(field_id, rate, optimized_for_weights != 0, e))
        return fail(CPB_BAD_PARAMS, "no default entry for field %d rate %d", field_id, rate);   // reference returns None / has no impl
    if (alpha) *alpha = e.alpha;
    if (full_rounds) *full_rounds = e.rf;
    if (partial_rounds) *partial_rounds = e.rp;
    if (skip_matrices) *skip_matrices = e.skip;
    return CPB_OK;
    });
}

cpb_status cpb_poseidon_ctx_create(int field_id, int rate, int capacity, int full_rounds, int partial_rounds,
                                   uint64_t alpha, const uint64_t* ark, const uint64_t* mds, int device,
                                   cpb_poseidon_ctx** out) {
    return cpb::guarded([&]() -> cpb_status {
    if (!out) return fail(CPB_NULL_POINTER, "null out");
    *out = nullptr;
    const uint64_t* mod = host::field_modulus(field_id);
    if (!mod) return fail(CPB_BAD_PARAMS, "unknown field id %d", field_id);
    if (!ark || !mds) return fail(CPB_NULL_POINTER, "null ark/mds");
    if (rate < 1 || capacity < 1 || rate + capacity > 16 || full_rounds < 0 || partial_rounds < 0 ||
        full_rounds + partial_rounds < 1)
        return fail(CPB_BAD_PARAMS, "bad Poseidon shape rate=%d capacity=%d RF=%d RP=%d", rate, capacity, full_rounds,
                    partial_rounds);
    host::Field F(mod);
    host::PoseidonParams P;
    P.rate = rate; P.capacity = capacity; P.full_rounds = full_rounds; P.partial_rounds = partial_rounds; P.alpha = alpha;
    int t = rate + capacity;
    P.ark.resize((size_t)(full_rounds + partial_rounds) * t);
    P.mds.resize((size_t)t * t);
    memcpy(P.ark.data(), ark, P.ark.size() * 32);
    memcpy(P.mds.data(), mds, P.mds.size() * 32);
    for (const auto& e : P.ark)
        if (!F.is_canonical(e)) return fail(CPB_BAD_PARAMS, "ark element not reduced");
    for (const auto& e : P.mds)
        if (!F.is_canonical(e)) return fail(CPB_BAD_PARAMS, "mds element not reduced");

    DeviceGuard g(device);
    if (!g.ok) { cudaGetLastError(); return fail(CPB_NO_DEVICE, "cudaSetDevice(%d) failed: no usable CUDA device", device); }
    int major = 0;
    CPB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(CPB_NO_DEVICE, "device %d is sm_%d0; this library is built for sm_100a only", device, major);

    keep_pool_memory(device);          // the tree-top launches take their progress words from the stream-ordered pool
    cpb_poseidon_ctx* c = new cpb_poseidon_ctx();
    c->field_id = field_id;
    c->device = device;
    c->sms = sm_count(device);
    c->sched = host::derive_schedule(F, P, true);
    c->dev = host::make_dev(c->sched);
    size_t bytes = c->sched.consts.size() * 8;
    if (bytes > 200 * 1024) { delete c; return fail(CPB_UNSUPPORTED, "round schedule (%zu B) exceeds shared memory", bytes); }
    cudaError_t e = cudaMalloc(&c->d_consts, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(c->d_consts, c->sched.consts.data(), bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        if (c->d_consts) cudaFree(c->d_consts);
        delete c;
        return fail(CPB_CUDA_ERROR, "context upload failed: %s", cudaGetErrorString(e));
    }
    *out = c;
    return CPB_OK;
    });
}

void cpb_poseidon_ctx_destroy(cpb_poseidon_ctx* c) {
    if (!c) return;
    DeviceGuard g(c->device);
    if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
    if (c->d_consts) cudaFree(c->d_consts);
    for (auto& s : c->side)
        if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
    c->s_in.release(); c->s_out.release(); c->s_aux.release();
    delete c;
}

int cpb_poseidon_ctx_is_sparse(const cpb_poseidon_ctx* c) { return c ? c->sched.sparse : 0; }
int cpb_poseidon_ctx_field(const cpb_poseidon_ctx* c) { return c ? c->field_id : -1; }
int cpb_poseidon_ctx_device(const cpb_poseidon_ctx* c) { return c ? c->device : -1; }

// ---- device-pointer entry points
cpb_status cpb_poseidon_permute_batch_dev(cpb_poseidon_ctx* c, const uint64_t* in, uint64_t* out, size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    DeviceGuard g(c->device);
    return launch_permute(c, (const u32*)in, (u32*)out, n, (cudaStream_t)stream);
    });
}
cpb_status cpb_poseidon_crh_batch_dev(cpb_poseidon_ctx* c, const uint64_t* in, size_t len, uint64_t* out, size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    DeviceGuard g(c->device);
    return launch_crh(c, (const u32*)in, len, (u32*)out, n, (cudaStream_t)stream);
    });
}
cpb_status cpb_poseidon_sponge_batch_dev(cpb_poseidon_ctx* c, const uint64_t* in, size_t len, uint64_t* out, size_t n_squeeze,
                                         size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    DeviceGuard g(c->device);
    return launch_crh(c, (const u32*)in, len, (u32*)out, n, (cudaStream_t)stream, n_squeeze);
    });
}
cpb_status cpb_merkle_poseidon_verify_batch_dev(cpb_poseidon_ctx* leaf, cpb_poseidon_ctx* node, const uint64_t* root,
                                                const uint64_t* leaves, size_t leaf_len, const uint64_t* leaf_sibling_hashes,
                                                const uint64_t* auth_paths, size_t path_len, const uint64_t* leaf_indexes,
                                                uint8_t* ok, size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(leaf));
    CPB_TRY(check_ctx(node));
    if (leaf->device != node->device || leaf->field_id != node->field_id || leaf->dev.t != node->dev.t)
        return fail(CPB_UNSUPPORTED, "leaf and node contexts must share device, field and state width");
    if (node->dev.rate < 2) return fail(CPB_UNSUPPORTED, "two-to-one with rate < 2 not supported");
    if (path_len > 62) return fail(CPB_BAD_PARAMS, "path too long");
    DeviceGuard g(leaf->device);
    return launch_verify(leaf, node, (const u32*)root, (const u32*)leaves, leaf_len, (const u32*)leaf_sibling_hashes,
                         (const u32*)auth_paths, (int)path_len, (const unsigned long long*)leaf_indexes, ok, n, (cudaStream_t)stream);
    });
}
cpb_status cpb_poseidon_compress_batch_dev(cpb_poseidon_ctx* c, const uint64_t* pairs, uint64_t* out, size_t n, void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    if (c->dev.rate < 2)   // two absorbs then one squeeze = one permutation only when rate >= 2
        return fail(CPB_UNSUPPORTED, "two-to-one with rate < 2 not supported");
    DeviceGuard g(c->device);
    return launch_crh(c, (const u32*)pairs, 2, (u32*)out, n, (cudaStream_t)stream);
    });
}
cpb_status cpb_merkle_poseidon_from_digests_dev(cpb_poseidon_ctx* node, const uint64_t* leaf_digests, size_t n,
                                                uint64_t* non_leaf_nodes, void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(node));
    if (!pow2_gt1(n)) return fail(CPB_NOT_POW2, "leaves.len() should be power of two and greater than one (got %zu)", n);
    if (node->dev.rate < 2) return fail(CPB_UNSUPPORTED, "two-to-one with rate < 2 not supported");
    DeviceGuard g(node->device);
    return merkle_build_streams(node, node, nullptr, 0, n, (u32*)leaf_digests, (u32*)non_leaf_nodes, (cudaStream_t)stream);
    });
}
cpb_status cpb_merkle_poseidon_build_dev(cpb_poseidon_ctx* leaf, cpb_poseidon_ctx* node, const uint64_t* leaves,
                                         size_t leaf_len, size_t n, uint64_t* leaf_nodes, uint64_t* non_leaf_nodes,
                                         void* stream) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(leaf));
    CPB_TRY(check_ctx(node));
    if (leaf->device != node->device || leaf->field_id != node->field_id)
        return fail(CPB_BAD_PARAMS, "leaf and node contexts must share device and field");
    if (!pow2_gt1(n)) return fail(CPB_NOT_POW2, "leaves.len() should be power of two and greater than one (got %zu)", n);
    if (node->dev.rate < 2) return fail(CPB_UNSUPPORTED, "two-to-one with rate < 2 not supported");
    DeviceGuard g(leaf->device);
    return merkle_build_streams(leaf, node, (const u32*)leaves, leaf_len, n, (u32*)leaf_nodes, (u32*)non_leaf_nodes,
                                (cudaStream_t)stream);
    });
}

// ---- host-pointer entry points: H2D, launch, D2H on the context stream
static cpb_status host_roundtrip_crh(cpb_poseidon_ctx* c, const uint64_t* in, size_t in_elems_per, size_t len,
                                     uint64_t* out, size_t out_elems_per, size_t n, int mode) {
    CPB_TRY(check_ctx(c));
    if (n == 0) return CPB_OK;
    if ((!in && in_elems_per) || !out) return fail(CPB_NULL_POINTER, "null buffer");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    size_t in_b = n * in_elems_per * 32, out_b = n * out_elems_per * 32;
    CPB_TRY(c->s_in.reserve(in_b ? in_b : 32));
    CPB_TRY(c->s_out.reserve(out_b));
    if (in_b) CPB_CUDA(cudaMemcpyAsync(c->s_in.ptr, in, in_b, cudaMemcpyHostToDevice, c->stream));
    if (mode == 0) CPB_TRY(launch_crh(c, (const u32*)c->s_in.ptr, len, (u32*)c->s_out.ptr, n, c->stream));
    else CPB_TRY(launch_permute(c, (const u32*)c->s_in.ptr, (u32*)c->s_out.ptr, n, c->stream));
    CPB_CUDA(cudaMemcpyAsync(out, c->s_out.ptr, out_b, cudaMemcpyDeviceToHost, c->stream));
    CPB_CUDA(cudaStreamSynchronize(c->stream));
    return CPB_OK;
}
cpb_status cpb_poseidon_permute_batch(cpb_poseidon_ctx* c, const uint64_t* in, uint64_t* out, size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    return host_roundtrip_crh(c, in, (size_t)c->dev.t, 0, out, (size_t)c->dev.t, n, 1);
    });
}
cpb_status cpb_poseidon_crh_batch(cpb_poseidon_ctx* c, const uint64_t* in, size_t len, uint64_t* out, size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    return host_roundtrip_crh(c, in, len, len, out, 1, n, 0);
    });
}
cpb_status cpb_poseidon_sponge_batch(cpb_poseidon_ctx* c, const uint64_t* in, size_t len, uint64_t* out, size_t n_squeeze, size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    if (n == 0 || n_squeeze == 0) return CPB_OK;
    if ((!in && len) || !out) return fail(CPB_NULL_POINTER, "null buffer");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    size_t in_b = n * len * 32, out_b = n * n_squeeze * 32;
    CPB_TRY(c->s_in.reserve(in_b ? in_b : 32));
    CPB_TRY(c->s_out.reserve(out_b));
    if (in_b) CPB_CUDA(cudaMemcpyAsync(c->s_in.ptr, in, in_b, cudaMemcpyHostToDevice, c->stream));
    CPB_TRY(launch_crh(c, (const u32*)c->s_in.ptr, len, (u32*)c->s_out.ptr, n, c->stream, n_squeeze));
    CPB_CUDA(cudaMemcpyAsync(out, c->s_out.ptr, out_b, cudaMemcpyDeviceToHost, c->stream));
    CPB_CUDA(cudaStreamSynchronize(c->stream));
    return CPB_OK;
    });
}
cpb_status cpb_merkle_poseidon_verify_batch(cpb_poseidon_ctx* leaf, cpb_poseidon_ctx* node, const uint64_t* root,
                                            const uint64_t* leaves, size_t leaf_len, const uint64_t* leaf_sibling_hashes,
                                            const uint64_t* auth_paths, size_t path_len, const uint64_t* leaf_indexes, uint8_t* ok,
                                            size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(leaf));
    CPB_TRY(check_ctx(node));
    if (n == 0) return CPB_OK;
    if (!root || (!leaves && leaf_len) || !leaf_sibling_hashes || (!auth_paths && path_len) || !leaf_indexes || !ok)
        return fail(CPB_NULL_POINTER, "null buffer");
    std::lock_guard<std::mutex> lk(leaf->mu);
    DeviceGuard g(leaf->device);
    size_t b_root = 32, b_leaves = n * leaf_len * 32, b_sib = n * 32, b_path = n * path_len * 32, b_idx = n * 8;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t o_leaves = up(b_root), o_sib = o_leaves + up(b_leaves), o_path = o_sib + up(b_sib), o_idx = o_path + up(b_path),
           total = o_idx + up(b_idx);
    CPB_TRY(leaf->s_in.reserve(total));
    CPB_TRY(leaf->s_out.reserve(n));
    char* d = (char*)leaf->s_in.ptr;
    cudaStream_t st = leaf->stream;
    CPB_CUDA(cudaMemcpyAsync(d, root, b_root, cudaMemcpyHostToDevice, st));
    if (b_leaves) CPB_CUDA(cudaMemcpyAsync(d + o_leaves, leaves, b_leaves, cudaMemcpyHostToDevice, st));
    CPB_CUDA(cudaMemcpyAsync(d + o_sib, leaf_sibling_hashes, b_sib, cudaMemcpyHostToDevice, st));
    if (b_path) CPB_CUDA(cudaMemcpyAsync(d + o_path, auth_paths, b_path, cudaMemcpyHostToDevice, st));
    CPB_CUDA(cudaMemcpyAsync(d + o_idx, leaf_indexes, b_idx, cudaMemcpyHostToDevice, st));
    CPB_TRY(cpb_merkle_poseidon_verify_batch_dev(leaf, node, (const uint64_t*)d, (const uint64_t*)(d + o_leaves), leaf_len,
                                                 (const uint64_t*)(d + o_sib), (const uint64_t*)(d + o_path), path_len,
                                                 (const uint64_t*)(d + o_idx), (uint8_t*)leaf->s_out.ptr, n, st));
    CPB_CUDA(cudaMemcpyAsync(ok, leaf->s_out.ptr, n, cudaMemcpyDeviceToHost, st));
    CPB_CUDA(cudaStreamSynchronize(st));
    return CPB_OK;
    });
}
cpb_status cpb_poseidon_compress_batch(cpb_poseidon_ctx* c, const uint64_t* pairs, uint64_t* out, size_t n) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(c));
    if (c->dev.rate < 2) return fail(CPB_UNSUPPORTED, "two-to-one with rate < 2 not supported");
    return host_roundtrip_crh(c, pairs, 2, 2, out, 1, n, 0);
    });
}

cpb_status cpb_merkle_poseidon_from_digests(cpb_poseidon_ctx* node, const uint64_t* leaf_digests, size_t n,
                                            uint64_t* non_leaf_nodes) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(node));
    if (!pow2_gt1(n)) return fail(CPB_NOT_POW2, "leaves.len() should be power of two and greater than one (got %zu)", n);
    if (!leaf_digests || !non_leaf_nodes) return fail(CPB_NULL_POINTER, "null buffer");
    std::lock_guard<std::mutex> lk(node->mu);
    DeviceGuard g(node->device);
    CPB_TRY(node->s_in.reserve(n * 32));
    CPB_TRY(node->s_out.reserve((n - 1) * 32));
    CPB_CUDA(cudaMemcpyAsync(node->s_in.ptr, leaf_digests, n * 32, cudaMemcpyHostToDevice, node->stream));
    CPB_TRY(cpb_merkle_poseidon_from_digests_dev(node, (const uint64_t*)node->s_in.ptr, n, (uint64_t*)node->s_out.ptr, node->stream));
    CPB_CUDA(cudaMemcpyAsync(non_leaf_nodes, node->s_out.ptr, (n - 1) * 32, cudaMemcpyDeviceToHost, node->stream));
    CPB_CUDA(cudaStreamSynchronize(node->stream));
    return CPB_OK;
    });
}

cpb_status cpb_merkle_poseidon_build(cpb_poseidon_ctx* leaf, cpb_poseidon_ctx* node, const uint64_t* leaves,
                                     size_t leaf_len, size_t n, uint64_t* leaf_nodes, uint64_t* non_leaf_nodes) {
    return cpb::guarded([&]() -> cpb_status {
    CPB_TRY(check_ctx(leaf));
    CPB_TRY(check_ctx(node));
    if (!pow2_gt1(n)) return fail(CPB_NOT_POW2, "leaves.len() should be power of two and greater than one (got %zu)", n);
    if ((!leaves && leaf_len) || !leaf_nodes || !non_leaf_nodes) return fail(CPB_NULL_POINTER, "null buffer");
    std::lock_guard<std::mutex> lk(leaf->mu);
    DeviceGuard g(leaf->device);
    size_t in_b = n * leaf_len * 32;
    CPB_TRY(leaf->s_in.reserve(in_b ? in_b : 32));
    CPB_TRY(leaf->s_out.reserve(n * 32));
    CPB_TRY(leaf->s_aux.reserve((n - 1) * 32));
    cudaStream_t st = leaf->stream;
    if (leaf->device != node->device || leaf->field_id != node->field_id)
        return fail(CPB_BAD_PARAMS, "leaf and node contexts must share device and field");
    if (node->dev.rate < 2) return fail(CPB_UNSUPPORTED, "two-to-one with rate < 2 not supported");
    MerkleHost H;
    H.leaves = (const u32*)leaves; H.leaf_nodes = (u32*)leaf_nodes; H.nodes = (u32*)non_leaf_nodes;
    CPB_TRY(merkle_build_streams(leaf, node, (const u32*)leaf->s_in.ptr, leaf_len, n, (u32*)leaf->s_out.ptr, (u32*)leaf->s_aux.ptr, st, &H));
    CPB_CUDA(cudaStreamSynchronize(st));
    return CPB_OK;
    });
}

}  // extern "C"
