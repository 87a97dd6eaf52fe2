"""bench.py --dump-outputs: the arrays written are those of the last timed step, equal to the oracle's outputs
for that step's inputs, and --steps is the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def close(a, b, rtol=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= rtol * np.maximum(1.0, np.abs(b))))


def test_bench_dump_outputs_c2(cuda_device, tmp_path):
    if not CO.available():
        pytest.skip("oracle/_build/librpn_oracle.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    import bench
    W, K = 3, 5
    env = dict(os.environ, TFRPN_BENCH_LANES="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup",
                        str(W), "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and line["warmup"] == W

    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert sorted(got) == sorted(["bbox_deltas", "bbox_labels", "proposal_boxes", "proposal_scores",
                                  "proposal_valid", "proposal_keep"])
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    # the last timed step replays the CUDA graph of set (W + K - 1) % SETS, captured with that index as the
    # sampling offset of the target assignment
    wl = bench.Workload("C2")
    sets = wl.n_sets(4)
    j = (W + K - 1) % sets
    gtb, gtl, reg, cls = wl.make_inputs(0, sets)[j]
    hp = wl.hyper_params(O.get_hyper_params)
    anchors = O.generate_anchors(hp)
    B = wl.B
    od, ol = CO.rpn_targets(anchors, gtb, gtl, hp, seed=2026, offset=j, image_offset=0)
    wb, ws, wv, wk = CO.proposals(reg.reshape(B, -1, 4), cls.reshape(B, -1), anchors, hp, bench.PRE_NMS)
    assert np.array_equal(got["bbox_labels"], ol.reshape(B, -1))
    assert close(got["bbox_deltas"], od)
    assert np.array_equal(got["proposal_valid"], wv) and np.array_equal(got["proposal_keep"], wk)
    assert np.array_equal(got["proposal_scores"], ws) and close(got["proposal_boxes"], wb)
