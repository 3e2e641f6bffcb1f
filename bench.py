#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (driver contract; see DESIGN.md "Measurement").

Workload (BASELINE.json metric "Poseidon perms/sec & 2^24-leaf Merkle build s at 1/2/4/8 B200"):
one step = one full MerkleTree::new of 2^24 two-element leaves with Poseidon CRH leaves and
Poseidon two-to-one nodes over BN254 Fr (t=3, RF=8, RP=57, alpha=5) -- BASELINE.json configs[3].
It fits one GPU, so the same workload runs at N = 1, 2, 4, 8 (strong scaling): the leaves are
sharded contiguously over the ranks, each rank builds its subtree, ONE all-gather of the subtree
roots, top levels replicated (crypto_primitives_b200/distributed.py).

Inputs are a counter-based stream over the GLOBAL leaf index (bench_inputs.py, SURVEY.md §8d), so the
tree -- and its root -- is the same at every N.  The root is printed and compared with the oracle's
root committed in tests/golden/bench_goldens.json (tests/golden/make_bench_goldens.py); at N > 1 every
rank additionally rebuilds the whole tree on its own GPU once, outside the timed region, and compares
its slices of every level with it.

`value` = Poseidon permutations per second of the whole job = (2N-1) / step time, inputs resident in
HBM.  `e2e` = the same through the host-pointer C-ABI call (cpb_merkle_poseidon_build): leaves in
pinned host memory, H2D of the leaves and D2H of both node arrays inside the timed region (a pageable
run is reported next to it).  `configs` holds the other BASELINE configurations, each checked against
committed oracle results.

--impl reference : the C restatement of the reference CPU path (oracle/cref, all usable host threads)
on the 2^20-leaf prefix of the same leaf stream (the Rust reference cannot be built in this image).

--dump-outputs DIR : after the timed steps, write what the last one returned (root, leaf digests, inner
nodes) to DIR/*.npy (dump_tree), so that two builds can be compared output for output on the same inputs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench_inputs as BI  # noqa: E402

WORKLOADS = {
    # name: (field, log2 leaves, leaf_len, seed, description)
    "merkle_2^24_poseidon_bn254": ("bn254", 24, 2, BI.SEED_CONFIG4, "2^24-leaf Poseidon Merkle tree, BN254 Fr (t=3, RF=8, RP=57, alpha=5), 2-element leaves"),
    "merkle_2^20_poseidon_bls12_381": ("bls", 20, 2, BI.SEED_CONFIG2, "2^20-leaf Poseidon Merkle tree, BLS12-381 Fr default rate-2 (alpha=17, RF=8, RP=31)"),
}
DEFAULT_WORKLOAD = "merkle_2^24_poseidon_bn254"
HBM_PEAK_FALLBACK = 6650.0      # GB/s, B200_PROFILING.md fallback
CPU_LOG_SAMPLE = 20             # the CPU arm builds the tree over the first 2^20 leaves of the stream
MASK64 = (1 << 64) - 1


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def goldens():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "bench_goldens.json")))


def u64_list(t):
    """4-limb digest tensor/array -> list of unsigned limbs (JSON-able, comparable with the golden file)."""
    return [int(x) & MASK64 for x in (t.reshape(-1).tolist())]


DUMP_SAMPLE = 1 << 18           # digests per sampled array: 16 MB each as float64 words, about 36 MB per dump in all
DUMP_SEED = 0xB20000D0


def dump_tree(tree, out_dir):
    """Writes the arrays one tree build hands its caller: root.npy (8,), and leaf_nodes.npy / non_leaf_nodes.npy (k, 8) at a
    fixed, seeded sample of k <= DUMP_SAMPLE indices (ascending; heap order for the inner nodes), stored in *_index.npy.
    A digest is 4 little-endian 64-bit Montgomery limbs; each row holds its eight 32-bit words as float64, which is exact."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)

    def words(t):
        return t.contiguous().cpu().numpy().view(np.uint32).astype(np.float64)

    np.save(os.path.join(out_dir, "root.npy"), words(tree.root.reshape(1, -1))[0])
    rng = np.random.default_rng(DUMP_SEED)
    for name, a in (("leaf_nodes", tree.local_leaf_nodes), ("non_leaf_nodes", tree.local_nodes)):
        idx = np.sort(rng.choice(a.shape[0], min(DUMP_SAMPLE, a.shape[0]), replace=False))
        np.save(os.path.join(out_dir, f"{name}.npy"), words(a[torch.from_numpy(idx).to(a.device)]))
        np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))


# --------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        load = [x for x in sm if x > 500] or sm
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------- parameters
def poseidon_params(cp, field_key):
    if field_key == "bls":
        return cp.get_default_poseidon_parameters(cp.BLS12_381_FR, 2, False)
    f = cp.BN254_FR
    ark, mds = cp.find_poseidon_ark_and_mds(f, 254, 2, 8, 57, 0)       # SURVEY.md §8a a1
    return cp.PoseidonConfig(f, 8, 57, 5, mds, ark, 2, 1)


def oracle_poseidon(field_key):
    from oracle import cref, fields as OF, poseidon as OP
    if field_key == "bls":
        cfg = OP.get_default_poseidon_parameters(OF.BLS12_381_FR, 2, False)
    else:
        ark, mds = OP.find_poseidon_ark_and_mds(OF.BN254_FR, 254, 2, 8, 57, 0)
        cfg = OP.PoseidonConfig(OF.BN254_FR, 8, 57, 5, ark, mds, 2, 1)
    return cfg, cref.Poseidon(cfg)


def wide_madds_per_perm(field_key: str, t: int, rf: int, rp: int, alpha: int, crh: bool = False) -> int:
    """32x32->64 multiply-adds one permutation needs in the device code (csrc/fp.cuh, poseidon.cuh; sparse partial rounds):
    a product row costs 8 for a*b_i plus `red` for m*p (8; 6 for BLS12-381 Fr, whose p[0] = 1 and p[1] = 2^32-1 turn two
    of them into additions); fp_mul = 8 rows; fp_sqr = 28 cross + 8 diagonal products + 8 reduction rows;
    fp_dot<T> = 8 rows of (8T + red); S-box = floor(log2 alpha) squarings + (popcount(alpha) - 1) products;
    full round = t S-boxes + t dot products, partial round = 1 S-box + 1 dot product + (t-1) column products.
    (BN254 t=3: 61 896, BLS12-381 t=3: 44 784 -- the IMAD.WIDE counts of the committed ncu opcode mixes.)
    crh=True: the one-permutation hash kernels (CRH::evaluate / TwoToOneCRH::compress, poseidon.cuh PermuteHint) do not
    execute the first S-box of the zero capacity lane (its value is a schedule constant) nor the t-1 last-round rows whose
    lanes are never read; they are not counted either (61 056 / 43 856)."""
    red = 6 if field_key == "bls" else 8
    mul, sqr, dot = 8 * (8 + red), 36 + 8 * red, 8 * (8 * t + red)
    sbox = (alpha.bit_length() - 1) * sqr + (bin(alpha).count("1") - 1) * mul
    total = rf * (t * sbox + t * dot) + rp * (sbox + dot + (t - 1) * mul)
    return total - (sbox + (t - 1) * dot if crh else 0)


def merkle_launches(ctx, n: int) -> int:
    """Kernel launches of one cpb_merkle_poseidon_build_dev over n leaves (csrc/cpb_poseidon.cu: merkle_build_streams)."""
    from crypto_primitives_b200 import _native as N
    return int(N.lib.cpb_merkle_poseidon_launch_count(ctx, n))


# --------------------------------------------------------------------------------- CPU arm (oracle/cref)
def host_cpu_info():
    """Threads the CPU arm may use: the scheduler affinity mask, capped by a cgroup CPU quota when one is set."""
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        a, b = open("/sys/fs/cgroup/cpu.max").read().split()[:2]           # cgroup v2
        if a != "max":
            quota = float(a) / float(b)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())     # cgroup v1
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                quota = q / p
        except Exception:
            pass
    threads = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return {"threads": threads, "affinity": aff, "os_cpu_count": os.cpu_count(), "cgroup_quota_cpus": quota}


class CpuArm:
    """The C restatement of the reference CPU path (kind "port") on the 2^CPU_LOG_SAMPLE-leaf prefix of the workload's
    leaf stream: a complete tree of the same shape (leaf CRH + all its levels), 1/16 of the 2^24-leaf job; its root is
    node 15 of the full tree (heap order), which the golden file holds."""

    def __init__(self, workload):
        import numpy as np
        from oracle import cref
        self.np, self.cref = np, cref
        self.field_key, logn, self.leaf_len, self.seed, _ = WORKLOADS[workload]
        self.workload = workload
        self.log_sample = min(logn, CPU_LOG_SAMPLE)
        self.n = 1 << self.log_sample
        self.cfg, self.P = oracle_poseidon(self.field_key)
        self.info = host_cpu_info()
        self.leaves = cref.synth_field_mont(self.seed, self.n * self.leaf_len, self.cfg.p).reshape(self.n, self.leaf_len, 4)
        self.perms = 2 * self.n - 1
        self.root = None

    def step(self, threads=None):
        t0 = time.perf_counter()
        _, nn = self.cref.poseidon_merkle(self.P, self.P, self.leaves, threads=threads or self.info["threads"])
        dt = time.perf_counter() - t0
        self.root = [int(x) for x in nn[0]]
        return self.perms / dt, dt

    def single_thread_rate(self):
        m = 1 << 11
        t0 = time.perf_counter()
        self.P.crh_batch(self.leaves[:m], threads=1)
        return m / (time.perf_counter() - t0)

    def root_matches_golden(self):
        try:
            g = goldens()[self.workload]
            k = (1 << (g["log2_leaves"] - self.log_sample)) - 1                # heap index of the first subtree root at that depth
            return self.root == g["top_nodes_heap_order"][k]
        except Exception:
            return None

    def describe(self, value, dt):
        s1 = self.single_thread_rate()
        T = self.info["threads"]
        return {"value": value, "unit": "perms/s", "cores": T, "kind": "port",
                "sample": f"tree over the first 2^{self.log_sample} leaves of the same stream ({self.perms} permutations, {dt:.2f} s wall): 1/{1 << (WORKLOADS[self.workload][1] - self.log_sample)} of the job, same work per leaf",
                "host": self.info, "single_thread_perms_per_s": s1, "per_thread_perms_per_s": value / T,
                "parallel_efficiency": value / (T * s1), "root_matches_oracle_golden": self.root_matches_golden()}


def run_reference(args):
    """--impl reference: the CPU arm, on rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args.workload)
    vals, times = [], []
    for i in range(args.warmup + args.steps):
        v, dt = arm.step()
        if i >= args.warmup:
            vals.append(v); times.append(dt)
    value = statistics.median(vals)
    desc = WORKLOADS[args.workload][4]
    base = arm.describe(value, statistics.median(times))
    line = {"impl": "reference", "metric": "poseidon_perms_per_sec", "value": value, "unit": "perms/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.median(times), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u64x4 (256-bit Montgomery integer)", "data": "synthetic",
            "config": {"workload": args.workload, "description": desc,
                       "note": "C restatement of the reference CPU path (oracle/cref, persistent thread pool); the Rust reference cannot be built here",
                       "same_config": "same leaf stream, parameters and tree shape; each step builds the 2^%d-leaf prefix subtree (a throughput metric: perms/s does not depend on the tree size)" % arm.log_sample},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "perms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------- GPU arm
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import crypto_primitives_b200 as cp
    from crypto_primitives_b200 import _native as N
    from crypto_primitives_b200.distributed import CudaMixedBackend, CudaPoseidonBackend, Exchange, level_slices, sharded_merkle_build

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a one-GPU build: use it with --gpus 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    field_key, logn, leaf_len, seed, desc = WORKLOADS[args.workload]
    n_total = 1 << logn
    assert n_total % world == 0
    n_local = n_total // world
    params = poseidon_params(cp, field_key)
    fid = params.field.id
    backend = CudaPoseidonBackend(params, params, local_rank)
    # N > 1: the subtree roots are exchanged inside the last kernel of each rank's build over NVLink peer memory (CUDA IPC);
    # CPB_BENCH_EXCHANGE=nccl selects the torch.distributed all-gather for the headline instead (timed alongside anyway)
    use_fused = world > 1 and os.environ.get("CPB_BENCH_EXCHANGE", "fused") != "nccl"
    ex, ex_error = None, None
    if world > 1:
        try:
            ex = Exchange(local_rank)
        except Exception as e:                          # e.g. CUDA IPC not permitted in this container: every rank falls back together
            ex_error = repr(e)
        ok = torch.tensor([0 if ex is None else 1], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if not bool(ok.item()):
            ex, use_fused = None, False
    # this rank's slice of the global leaf stream: leaves [rank*n_local, (rank+1)*n_local)
    leaves = BI.field_elements_torch(torch, N, fid, seed, rank * n_local * leaf_len, n_local * leaf_len, local_rank).view(n_local, leaf_len, 4)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    gold = goldens()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_true(flag: bool) -> bool:
        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def step(fused=use_fused):
        return sharded_merkle_build(backend, leaves, gather="roots", exchange=ex if fused else None)

    perms_total = 2 * n_total - 1
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    times = []
    root = None
    tree = None
    for _ in range(args.steps):
        flush.zero_()                                   # evict L2 between timed iterations (not timed)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tree = step()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
        root = tree.root.clone()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_tree(tree, args.dump_outputs)
    t = torch.tensor([sum(times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = perms_total / (ms_per_step * 1e-3)

    # ---- N > 1: the other root exchange (NCCL all-gather issued from Python <-> fused peer-memory kernel), 3 steps
    other_ms = None
    if world > 1 and ex is not None:
        ts = []
        for i in range(4):
            flush.zero_()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(fused=not use_fused)
            e1.record()
            torch.cuda.synchronize()
            if i:
                ts.append(e0.elapsed_time(e1))
        tt = torch.tensor([sum(ts) / len(ts)], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        other_ms = float(tt.item())
        tree = step()
        torch.cuda.synchronize()
        root = tree.root.clone()
    if world > 1 and ex is None:
        other_ms = None

    # ---- parity of the timed result: the root against the oracle's committed root (every rank holds the root)
    g = gold.get(args.workload, {})
    root_u = u64_list(root.cpu())
    root_ok = all_true(root_u == g.get("root"))
    # ---- N > 1: every rank rebuilds the WHOLE tree on its own GPU and compares its slices of every level (untimed)
    slices_ok = None
    if world > 1:
        full_leaves = BI.field_elements_torch(torch, N, fid, seed, 0, n_total * leaf_len, local_rank).view(n_total, leaf_len, 4)
        ref_backend = CudaPoseidonBackend(params, params, local_rank)
        f_leaf, f_nodes = ref_backend.build_local(full_leaves)
        ok = torch.equal(tree.local_leaf_nodes, f_leaf[rank * n_local:(rank + 1) * n_local])
        for gstart, per, lstart in level_slices(n_total, world, rank):
            ok = ok and torch.equal(tree.local_nodes[lstart:lstart + per], f_nodes[gstart:gstart + per])
        ok = ok and torch.equal(tree.top_nodes, f_nodes[:world - 1]) and torch.equal(root, f_nodes[0])
        torch.cuda.synchronize()
        slices_ok = all_true(bool(ok))
        del full_leaves, f_leaf, f_nodes, ref_backend
        torch.cuda.empty_cache()

    # ---- e2e: host-pointer C-ABI call on this rank's shard, copies inside the timed region
    ctx = params.context(local_rank)
    h_leaves = torch.empty((n_local, leaf_len, 4), dtype=torch.int64, pin_memory=True)
    h_leaves.copy_(leaves)
    h_leaf_nodes = torch.empty((n_local, 4), dtype=torch.int64, pin_memory=True)
    h_nodes = torch.empty((max(n_local - 1, 1), 4), dtype=torch.int64, pin_memory=True)
    h_top = torch.empty((max(world - 1, 1), 4), dtype=torch.int64, pin_memory=True)

    def e2e_call(hl, hln, hn):
        if world > 1 and ex is None:
            N.check(N.lib.cpb_merkle_poseidon_build(ctx, ctx, N.C.cast(hl.data_ptr(), N.u64p), leaf_len, n_local,
                                                    N.C.cast(hln.data_ptr(), N.u64p), N.C.cast(hn.data_ptr(), N.u64p)))
            r = hn[0].to(dev, non_blocking=False).reshape(1, 4)
            roots = torch.empty((world, 4), dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(roots, r)
            return backend.from_digests(roots)[0].cpu()
        if world > 1:       # this rank's shard through the host-pointer sharded call: copies, hashing, root exchange, top levels
            N.check(N.lib.cpb_merkle_poseidon_build_sharded(ctx, ctx, ex.handle, N.C.cast(hl.data_ptr(), N.u64p), leaf_len, n_local,
                                                            N.C.cast(hln.data_ptr(), N.u64p), N.C.cast(hn.data_ptr(), N.u64p),
                                                            N.C.cast(h_top.data_ptr(), N.u64p)))
            return h_top[0]
        N.check(N.lib.cpb_merkle_poseidon_build(ctx, ctx, N.C.cast(hl.data_ptr(), N.u64p), leaf_len, n_local,
                                                N.C.cast(hln.data_ptr(), N.u64p), N.C.cast(hn.data_ptr(), N.u64p)))
        return hn[0]

    def e2e_time(hl, hln, hn, steps):
        e2e_call(hl, hln, hn)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = e2e_call(hl, hln, hn)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return perms_total / (float(dt.item()) / steps), r

    e2e_steps = max(1, min(args.steps, 3))
    e2e_value, e2e_root = e2e_time(h_leaves, h_leaf_nodes, h_nodes, e2e_steps)
    e2e_root_ok = all_true(u64_list(torch.as_tensor(e2e_root).cpu()) == g.get("root"))
    e2e_pageable = None
    if world == 1:                                       # what a Rust Vec<Fr> is unless the shim pins it (cpb_host_register)
        p_leaves = torch.empty((n_local, leaf_len, 4), dtype=torch.int64)
        p_leaves.copy_(h_leaves)
        p_ln = torch.empty((n_local, 4), dtype=torch.int64)
        p_n = torch.empty((max(n_local - 1, 1), 4), dtype=torch.int64)
        v, r = e2e_time(p_leaves, p_ln, p_n, 1)
        e2e_pageable = {"value": v, "unit": "perms/s", "root_matches_oracle": u64_list(torch.as_tensor(r)) == g.get("root")}
        del p_leaves, p_ln, p_n

    # ---- roofline of the dominant kernel (k_poseidon_crh, the leaf-hash launch), timed live with CUDA events
    out = torch.empty((n_local, 4), dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def time_kernel(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        ks = []
        for _ in range(reps):
            flush.zero_()
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record(); fn(); k1.record()
            torch.cuda.synchronize()
            ks.append(k0.elapsed_time(k1))
        return statistics.median(ks)

    k_ms = time_kernel(lambda: N.check(N.lib.cpb_poseidon_crh_batch_dev(ctx, leaves.data_ptr(), leaf_len, out.data_ptr(), n_local, st)))
    alg_bytes = n_local * (32 * leaf_len + 32)                      # SURVEY.md §8d: 32*L read + 32 written per leaf hash
    peaks = measured_peaks()
    peak = peaks["hbm_gbs"] if peaks else HBM_PEAK_FALLBACK
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    ncu = NCU_TRAFFIC[field_key]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu["bytes_per_hash"] * n_local, "traffic_source": ncu["source"],
                "kernel": "k_poseidon_crh (leaf level: %d hashes of %d elements)" % (n_local, leaf_len), "kernel_ms": k_ms,
                "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "B200_PROFILING.md fallback (of fallback)",
                "note": "the path is bound by the integer multiply pipe, not HBM (~6e4 IMAD-class instructions per 96 algorithmic bytes); see integer_pipe"}
    sm_clock = (clocks or {}).get("sm_mhz") or 1965.0

    def integer_pipe(fkey, prm, perms, ms, crh=False):
        w = wide_madds_per_perm(fkey, prm.rate + prm.capacity, prm.full_rounds, prm.partial_rounds, prm.alpha, crh)
        int_peak = 148 * 32 * sm_clock * 1e6            # IMAD.WIDE: 32 lanes/clk/SM (profiles/r2_ubench_imad.txt), x sampled SM clock
        return {"wide_madds_per_perm": w, "achieved_wide_madds_per_s": perms * w / (ms * 1e-3), "peak_wide_madds_per_s": int_peak,
                "frac": perms * w / (ms * 1e-3) / int_peak, "peak_source": "148 SMs x 32 lanes/clk (measured IMAD.WIDE issue rate) x sampled SM clock"}

    integer = integer_pipe(field_key, params, n_local, k_ms, crh=True)     # the leaf kernel: one-permutation CRH

    # ---- the other BASELINE configurations (each checked against committed oracle results)
    configs = {}
    cfg_sampler = ClockSampler(local_rank)
    if rank == 0:
        cfg_sampler.start()
    try:
        configs["config5_mixed_merkle_2^22"] = config5(torch, dist, cp, N, BI, CudaMixedBackend, sharded_merkle_build, gold, world, rank,
                                                       local_rank, flush, barrier, all_true, ex if use_fused else None)
    except Exception as e:                              # an extra, never a reason to lose the contract line
        configs["config5_mixed_merkle_2^22"] = {"error": repr(e)}
    if world == 1:
        for name, fn in (("config2_bls12_381", config2), ("config3_pedersen_2^20", config3)):
            try:
                configs[name] = fn(torch, cp, N, BI, gold, local_rank, flush, time_kernel, integer_pipe, peak)
            except Exception as e:
                configs[name] = {"error": repr(e)}
        try:
            configs["config1_crh_1024"] = config1_probe()
        except Exception as e:
            configs["config1_crh_1024"] = {"error": repr(e)}
    cfg_clocks = cfg_sampler.stop() if rank == 0 else None

    if rank == 0:
        launches_per_step = merkle_launches(ctx, n_local) + (0 if (world == 1 or use_fused) else 1)
        line = {"metric": "poseidon_perms_per_sec", "value": value, "unit": "perms/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "merkle_build_s": ms_per_step * 1e-3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (256-bit Montgomery integer)", "data": "synthetic",
                "config": {"workload": args.workload, "description": desc, "leaves_total": n_total, "leaves_per_gpu": n_local,
                           "parallelism": (f"leaf-sharded x{world}; subtree roots exchanged " +
                                           ("inside each rank's last kernel over NVLink peer memory (CUDA IPC), top levels fused in" if use_fused
                                            else "by one NCCL all-gather (torch.distributed)")) if world > 1 else "one GPU",
                           "other_exchange_ms_per_step": other_ms, "exchange_error": ex_error, "other_exchange": None if world == 1 else ("nccl all-gather" if use_fused else "fused peer-memory kernel"),
                           "l2": "flushed (256 MB write) between timed steps",
                           "perms_per_step": perms_total, "inputs": "SplitMix64 stream over the global leaf index (bench_inputs.py): identical tree at every N"},
                "root": root_u, "root_matches_oracle": root_ok, "slices_match_single_gpu_build": slices_ok,
                "oracle_root_source": "tests/golden/bench_goldens.json (oracle/cref via tests/golden/make_bench_goldens.py)",
                "clocks": clocks, "gpu_launches": launches_per_step * args.steps,
                "e2e": {"value": e2e_value, "unit": "perms/s", "h2d_bytes_per_step": n_local * leaf_len * 32 * world,
                        "d2h_bytes_per_step": (2 * n_local - 1) * 32 * world, "steps": e2e_steps, "root_matches_oracle": e2e_root_ok,
                        "api": "cpb_merkle_poseidon_build (host pointers, pinned)" if (world == 1 or ex is None) else "cpb_merkle_poseidon_build_sharded (host pointers, pinned; root exchange inside)",
                        "pageable": e2e_pageable},
                "roofline": roofline, "integer_pipe": integer, "configs": configs, "configs_clocks": cfg_clocks}
        if world == 1:
            arm = CpuArm(args.workload)
            v, dt = arm.step()
            line["cpu_baseline"] = arm.describe(v, dt)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# DRAM traffic of k_poseidon_crh from the committed `ncu --set full` captures (dram__bytes_read.sum + dram__bytes_write.sum of a
# 2^20-hash, len-2 launch), per hash.  Update together with the files named here.
NCU_TRAFFIC = {
    "bn254": {"bytes_per_hash": (67.246848e6 + 6.766848e6) / (1 << 20), "source": "profiles/r2_ncu_crh_bn254.txt (2^20-hash launch), scaled per hash"},
    "bls": {"bytes_per_hash": (67.188736e6 + 8.603136e6) / (1 << 20), "source": "profiles/r2_ncu_crh_bls.txt (2^20-hash launch), scaled per hash"},
}


def config1_probe():
    """BASELINE configs[0] -- the reference's own CPU-runnable case: crh::poseidon::CRH::evaluate on 1024 inputs of two
    BLS12-381 Fr elements (default rate-2 parameters).  CPU: the C restatement on ONE thread, as that config is stated;
    GPU: the host-pointer C-ABI call (copies included), median of 20.  Outputs compared."""
    import numpy as np
    import crypto_primitives_b200 as cp
    from crypto_primitives_b200 import _native as N
    from oracle import cref
    ocfg, P = oracle_poseidon("bls")
    x = cref.synth_field_mont(BI.SEED_CONFIG1, 1024 * 2, ocfg.p).reshape(1024, 2, 4)
    t0 = time.perf_counter()
    exp = P.crh_batch(x, threads=1)
    cpu_dt = time.perf_counter() - t0
    cfg = cp.get_default_poseidon_parameters(cp.BLS12_381_FR, 2, False)
    ctx = cfg.context(0)
    out = np.empty((1024, 4), dtype=np.uint64)
    times = []
    for _ in range(23):
        t0 = time.perf_counter()
        N.check(N.lib.cpb_poseidon_crh_batch(ctx, x.ctypes.data_as(N.u64p), 2, out.ctypes.data_as(N.u64p), 1024))
        times.append(time.perf_counter() - t0)
    gpu_dt = statistics.median(times[3:])
    return {"workload": "crh::poseidon::CRH::evaluate, BLS12-381 Fr, 1024 inputs x 2 elements",
            "cpu_single_thread": {"hashes_per_s": 1024 / cpu_dt, "ms": 1e3 * cpu_dt, "kind": "port"},
            "gpu_host_call": {"hashes_per_s": 1024 / gpu_dt, "ms": 1e3 * gpu_dt, "api": "cpb_poseidon_crh_batch (pageable host pointers, copies included)"},
            "outputs_equal": bool(np.array_equal(out, exp))}


def config2(torch, cp, N, BI, gold, dev_index, flush, time_kernel, integer_pipe, hbm_peak):
    """BASELINE configs[1]: 2^20-leaf Poseidon tree over BLS12-381 Fr on one B200, plus north_star's batched-permutation
    rate (2^22 bare permutations).  Root / sampled states against the committed oracle results."""
    from crypto_primitives_b200.distributed import CudaPoseidonBackend
    prm = poseidon_params(cp, "bls")
    ctx = prm.context(dev_index)
    st = torch.cuda.current_stream().cuda_stream
    n = 1 << 20
    leaves = BI.field_elements_torch(torch, N, prm.field.id, BI.SEED_CONFIG2, 0, 2 * n, dev_index).view(n, 2, 4)
    be = CudaPoseidonBackend(prm, prm, dev_index)
    ms_tree = time_kernel(lambda: be.build_local(leaves), reps=5)
    _, nodes = be.build_local(leaves)
    torch.cuda.synchronize()
    g = gold["merkle_2^20_poseidon_bls12_381"]
    tree = {"ms": ms_tree, "perms_per_s": (2 * n - 1) / (ms_tree * 1e-3), "root": u64_list(nodes[0].cpu()),
            "root_matches_oracle": u64_list(nodes[0].cpu()) == g["root"],
            "top_nodes_match_oracle": [u64_list(r) for r in nodes[:31].cpu()] == g["top_nodes_heap_order"]}
    m = 1 << 22
    states = BI.field_elements_torch(torch, N, prm.field.id, BI.SEED_CONFIG2_PERM, 0, 3 * m, dev_index).view(m, 3, 4)
    outs = torch.empty_like(states)
    ms_perm = time_kernel(lambda: N.check(N.lib.cpb_poseidon_permute_batch_dev(ctx, states.data_ptr(), outs.data_ptr(), m, st)), reps=5)
    gs = gold["permute_2^22_bls12_381"]["state_samples"]
    ok = all([u64_list(r) for r in outs[int(i)].cpu()] == v for i, v in gs.items())
    gbs = m * 192 / (ms_perm * 1e-3) / 1e9
    batched = {"ms": ms_perm, "perms_per_s": m / (ms_perm * 1e-3), "n": m, "sampled_states_match_oracle": bool(ok),
               "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                            "algorithmic_bytes_per_perm": 192},
               "integer_pipe": integer_pipe("bls", prm, m, ms_perm), "north_star_target_perms_per_s": 1e8}
    return {"workload": "BASELINE configs[1]: 2^20-leaf Poseidon Merkle tree + 2^22 batched permutations, BLS12-381 Fr, 1 GPU",
            "tree_2^20": tree, "batched_permutations_2^22": batched}


def pedersen_setup(cp):
    from crypto_primitives_b200.commitment.pedersen import Commitment
    from crypto_primitives_b200.crh.pedersen import Window
    return Commitment.setup(BI.StreamRng(BI.SEED_CONFIG3_PARAMS), Window(4, 256))


def config3(torch, cp, N, BI, gold, dev_index, flush, time_kernel, integer_pipe, hbm_peak):
    """BASELINE configs[2]: crh::pedersen + commitment::pedersen over Jubjub, window 4x256, 2^20 x 128-byte inputs, one B200."""
    dev = torch.device("cuda", dev_index)
    prm = pedersen_setup(cp)
    t0 = time.perf_counter()
    ctx = prm.context(dev_index)
    torch.cuda.synchronize()
    ctx_ms = 1e3 * (time.perf_counter() - t0)
    st = torch.cuda.current_stream().cuda_stream
    n = 1 << 20
    inp = BI.bytes_torch(torch, BI.SEED_CONFIG3, 0, 128 * n, dev).view(n, 128)
    rnd = BI.randomness_torch(torch, BI.SEED_CONFIG3_RAND, 0, n, dev)
    out_h = torch.empty((n, 2, 4), dtype=torch.int64, device=dev)
    out_c = torch.empty((n, 2, 4), dtype=torch.int64, device=dev)
    ms_crh = time_kernel(lambda: N.check(N.lib.cpb_pedersen_crh_batch_dev(ctx, inp.data_ptr(), 128, 128, out_h.data_ptr(), n, st)), reps=5)
    ms_com = time_kernel(lambda: N.check(N.lib.cpb_pedersen_commit_batch_dev(ctx, inp.data_ptr(), 128, 128, rnd.data_ptr(), out_c.data_ptr(), n, st)), reps=5)
    g = gold["pedersen_2^20_jubjub"]
    ok_h = all([u64_list(r) for r in out_h[int(i)].cpu()] == v for i, v in g["crh_xy"].items())
    ok_c = all([u64_list(r) for r in out_c[int(i)].cpu()] == v for i, v in g["commit_xy"].items())
    f = cp.BLS12_381_FR
    gen_ok = [str(v) for v in f.to_ints(prm.generators[0, 0])] == g["generator_0_0"]
    # opt-in: 20 input bits per table lookup (5.2 GB of tables for this window + the randomness generators): HBM capacity for integer-pipe work
    from crypto_primitives_b200.crh.pedersen import Parameters
    wide = Parameters(prm.curve, prm.window, prm.generators, prm.randomness_generator, chunk_bits=20)
    t0 = time.perf_counter()
    wctx = wide.context(dev_index)
    torch.cuda.synchronize()
    wide_ctx_ms = 1e3 * (time.perf_counter() - t0)
    out_w = torch.empty((n, 2, 4), dtype=torch.int64, device=dev)
    ms_w = time_kernel(lambda: N.check(N.lib.cpb_pedersen_crh_batch_dev(wctx, inp.data_ptr(), 128, 128, out_w.data_ptr(), n, st)), reps=5)
    ok_w = bool(torch.equal(out_w, out_h))
    alg = 128 + 64
    gbs = n * alg / (ms_crh * 1e-3) / 1e9
    lookups = -(-1024 // 18)
    return {"workload": "BASELINE configs[2]: Pedersen CRH + commitment, Jubjub, window 4x256, 2^20 x 128-byte inputs, 1 GPU",
            "crh": {"ms": ms_crh, "hashes_per_s": n / (ms_crh * 1e-3), "sampled_outputs_match_oracle": bool(ok_h)},
            "commit": {"ms": ms_com, "commits_per_s": n / (ms_com * 1e-3), "sampled_outputs_match_oracle": bool(ok_c)},
            "crh_20bit_tables": {"ms": ms_w, "hashes_per_s": n / (ms_w * 1e-3), "equals_default_tables_output": ok_w, "table_gb": 66 * 96 * 2**20 / 1e9,
                                 "context_create_ms": wide_ctx_ms, "note": "opt-in cpb_pedersen_ctx_create_ex(chunk_bits=20)"},
            "generators_match_oracle_setup": bool(gen_ok), "context_create_ms": ctx_ms,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "algorithmic_bytes_per_hash": alg,
                         "gathered_table_bytes_per_hash": lookups * 96,
                         "note": "default 18-bit table lookups: %d gathered 96-byte entries per hash from 1.8 GB of tables -- DRAM traffic ~%dx the algorithmic bytes "
                                 "by design, trading HBM bandwidth and capacity for fewer point additions; bound by the integer multiply pipe" % (lookups, lookups * 96 // alg)}}


def config5(torch, dist, cp, N, BI, CudaMixedBackend, sharded_merkle_build, gold, world, rank, dev_index, flush, barrier, all_true, ex=None):
    """BASELINE configs[4]: Pedersen leaf CRH (x-coordinate) + Poseidon two-to-one over BLS12-381 Fr, 2^22 x 128-byte leaves,
    leaf-sharded over the ranks of this run (BASELINE names 4 GPUs); root against the committed oracle root."""
    dev = torch.device("cuda", dev_index)
    n = 1 << 22
    n_local = n // world
    prm = pedersen_setup(cp)
    node = poseidon_params(cp, "bls")
    be = CudaMixedBackend(prm, node, dev_index)
    leaves = BI.bytes_torch(torch, BI.SEED_CONFIG5, 128 * rank * n_local, 128 * n_local, dev).view(n_local, 128)
    for _ in range(2):
        tree = sharded_merkle_build(be, leaves, gather="roots", exchange=ex)
    ts = []
    for _ in range(3):
        flush.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tree = sharded_merkle_build(be, leaves, gather="roots", exchange=ex)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    t = torch.tensor([statistics.median(ts)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    g = gold["mixed_merkle_2^22"]
    root = u64_list(tree.root.cpu())
    ok = all_true(root == g["root"])
    return {"workload": "BASELINE configs[4]: mixed tree, 2^22 x 128-byte leaves, Pedersen leaf hash + Poseidon two-to-one, BLS12-381 Fr",
            "n_gpus": world, "ms": ms, "merkle_build_s": ms * 1e-3, "hashes_per_step": {"pedersen": n, "poseidon": n - 1},
            "root": root, "root_matches_oracle": ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=list(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's root, leaf digests and inner nodes to DIR/*.npy (see dump_tree)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU build (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
