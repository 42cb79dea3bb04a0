"""bench.py --dump-outputs: what it writes is what the timed batch call computed -- every record of the batch and the
masks of the sampled units against the cv2 oracle -- as float arrays within 64 MB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_timed_outputs(tmp_path):
    import vi_b200
    from oracle import ref_cv2 as R
    from vi_b200 import synth
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--images", "2",
                          "--distinct", "2", "--no-cpu", "--no-ingest", "--no-extra", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["gpu_launches"] == 2
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert {f"record_{k}" for k in vi_b200.RECORD_DTYPE.names} | {"sample_units", "seg_masks", "defect_masks"} == set(got)
    assert int((got["record_status"] == vi_b200.STATUS_NG).sum()) == line["ng_units"]
    boxes = vi_b200.generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)
    oracle = [R.inspect_frame(synth.make_frame(s, [b for b, _ in boxes]), boxes, R.Params(), (), None, True) for s in (0, 1)]
    for i, (recs, _, _) in enumerate(oracle):
        assert (got["record_image"][i] == i).all() and (got["record_unit"][i] == np.arange(len(boxes))).all()
        for k in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status', 'dx', 'dy'):
            assert got[f"record_{k}"][i].tolist() == [o[k] for o in recs], (i, k)
    assert len(got["sample_units"]) == 48
    for s, (i, u) in enumerate(got["sample_units"].astype(int)):
        _, segs, defs = oracle[i]
        assert np.array_equal(got["seg_masks"][s], segs[u]), (i, u)
        want = defs[u] if defs[u] is not None else np.zeros_like(segs[u])
        assert np.array_equal(got["defect_masks"][s], want), (i, u)
