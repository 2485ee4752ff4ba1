"""bench.py contract checks: the reference arm prints one JSON line with the agreed keys; --dump-outputs writes the
tables of the last timed cycle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], check=True, capture_output=True, text=True,
                          cwd=ROOT).stdout.strip().splitlines()


def _load_dump(d):
    out = {}
    for f in sorted(os.listdir(d)):
        a = np.load(os.path.join(d, f))
        assert a.dtype in (np.float32, np.float64) and a.size, (f, a.dtype, a.shape)
        out[f[:-len(".npy")]] = a
    return out


def test_reference_arm_json_line():
    line = json.loads(_bench("--impl", "reference", "--config", "1", "--steps", "3", "--warmup", "1")[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_algorithmic_bytes_table_covers_every_timed_kernel():
    sys.path.insert(0, ROOT)
    import bench
    from kueue_b200 import abi, synth
    ab = bench.algorithmic_bytes(synth.make_snapshot(1))
    for name in abi.KERNEL_NAMES:
        # the kb_tas_find kernels are accounted in bench.run_tas (cfg5), "-" is an unused timing slot
        assert name in ab or name in ("k_lone", "k_tas_leaf", "k_tas_reduce", "k_tas_select", "-"), name


def test_reference_arm_dumps_its_last_cycle(tmp_path):
    import oracle
    from kueue_b200 import synth
    _bench("--impl", "reference", "--config", "1", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    got = _load_dump(tmp_path)
    want = oracle.run_cycle(synth.make_snapshot(1))
    names = ("decision", "mode", "borrow", "commit_rank", "ps_flavor", "ps_res_mode", "ps_tried_idx", "ps_count", "tgt_start",
             "tgt_adm", "tgt_reason", "node_usage")
    tables = {k: np.asarray(getattr(want, k))[:want.n_targets] if k in ("tgt_adm", "tgt_reason") else np.asarray(getattr(want, k))
              for k in names}
    assert sorted(got) == sorted(k for k, w in tables.items() if w.size), "empty tables are left out, all others written"
    for k in got:
        assert np.array_equal(got[k], tables[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("config", [1, 3])
def test_device_dump_equals_reference_dump(tmp_path, config):
    """The tables the device's last timed cycle returns are the oracle's, bit for bit (cfg3: the full-size headline)."""
    common = ["--config", str(config), "--steps", "3", "--warmup", "1", "--dump-outputs"]
    _bench("--impl", "reference", *common, str(tmp_path / "reference"))
    _bench("--no-cpu-baseline", "--no-drain", *common, str(tmp_path / "ours"))
    want, got = _load_dump(tmp_path / "reference"), _load_dump(tmp_path / "ours")
    assert sorted(got) == sorted(want)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
