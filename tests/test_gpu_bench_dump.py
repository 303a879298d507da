"""GPU suite (-m gpu): bench.py --dump-outputs writes the outputs of the benchmark step for its seeded inputs -- the launch chain
(layer i on its own row x[i]) and the dependent decode sequence (x[i+1] = first K outputs of layer i) -- checked against the
oracle with the benchmark's own parity tolerance."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import tmac_oracle as T

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_match_the_oracle(oracle, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--no-extras",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["metric"] == bench.METRIC
    assert sorted(os.listdir(tmp_path)) == ["launch_chain.npy", "sequence_dependent_chain.npy"]
    chain = np.load(tmp_path / "launch_chain.npy")
    seq = np.load(tmp_path / "sequence_dependent_chain.npy")
    assert chain.dtype == seq.dtype == np.float32 and chain.shape == seq.shape == (bench.LAYERS, bench.MOUT)

    cfg = T.Config(bench.MOUT, bench.K, bench.BITS, group_size=bench.GS, act_group_size=bench.AGS, zero_point=bench.ZP).resolved()
    A, S = T.pack_reference_layout(*bench.synth(100), cfg)
    x = bench.activations(200)

    def check(got, xrow):
        q, ls, lb = oracle.preprocessor(xrow[None], bench.AGS)
        want = oracle.qgemm(cfg, A, S, q, ls, lb)[0]
        assert np.abs(got - want).max() <= 1e-3 * np.abs(want).max()
    for i in (0, bench.LAYERS - 1):
        check(chain[i], x[i])
    check(seq[0], x[0])
    check(seq[bench.LAYERS - 1], seq[bench.LAYERS - 2][:bench.K])
