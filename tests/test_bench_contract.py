"""bench.py's CPU arm (`--impl reference`: the C restatement of the reference path on the host cores) runs without a GPU
and prints the contract's JSON line; under torchrun only rank 0 prints.  Also the file format of --dump-outputs and the
argument checks."""
import json
import os
import subprocess
import sys

from helpers import ROOT


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout.strip()


def test_reference_arm_prints_one_contract_line():
    out = _run()
    line = json.loads(out.splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "poseidon_perms_per_sec" and line["unit"] == "perms/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "perms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["steps"] == 1 and line["warmup"] == 0
    # the CPU arm's tree is the first 1/16 of the 2^24-leaf job: its root is node 15 of the committed oracle tree
    assert line["cpu_baseline"]["root_matches_oracle_golden"] is True
    assert line["cpu_baseline"]["host"]["threads"] == line["cpu_baseline"]["cores"]


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == ""


def test_dump_outputs_are_exact_float_images_of_a_fixed_sample(tmp_path):
    """--dump-outputs (bench.dump_tree): float64 32-bit words that give back the limbs exactly, at the same indices every run."""
    import types

    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n = 3 * bench.DUMP_SAMPLE // 2
    g = torch.Generator().manual_seed(5)
    leaf = torch.randint(-2**62, 2**62, (n, 4), dtype=torch.int64, generator=g)
    nodes = torch.randint(-2**62, 2**62, (n - 1, 4), dtype=torch.int64, generator=g)
    tree = types.SimpleNamespace(root=nodes[0], local_leaf_nodes=leaf, local_nodes=nodes)
    for d in ("a", "b"):
        bench.dump_tree(tree, str(tmp_path / d))

    def limbs(w):
        w = w.astype(np.uint64)
        return w[..., 0::2] | (w[..., 1::2] << np.uint64(32))

    assert np.array_equal(limbs(np.load(tmp_path / "a" / "root.npy")), nodes[0].numpy().view(np.uint64))
    total = 0
    for name, src in (("leaf_nodes", leaf), ("non_leaf_nodes", nodes)):
        words, idx = (np.load(tmp_path / "a" / f"{name}{s}.npy") for s in ("", "_index"))
        assert words.dtype == idx.dtype == np.float64 and words.shape == (bench.DUMP_SAMPLE, 8)
        assert np.array_equal(limbs(words), src.numpy().view(np.uint64)[idx.astype(np.int64)])
        assert np.array_equal(words, np.load(tmp_path / "b" / f"{name}.npy"))
        total += words.nbytes + idx.nbytes
    assert total <= 64 << 20


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=ROOT, timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr
