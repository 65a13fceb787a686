"""CPU tier: `bench.py --dump-outputs` on the CPU arm at a tiny size — the dumped array is the MSM of the bench's
seeded inputs, exactly, in the documented layout (one float64 per byte of the 104-byte affine image)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_dumps_the_msm_of_its_seeded_inputs(cref, tmp_path):
    log_n = 6
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--log-n", str(log_n),
                          "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path)],
                         cwd=ROOT, capture_output=True, text=True, check=True).stdout
    line = json.loads(out.strip().splitlines()[-1])
    assert line["steps"] == 2
    got = np.load(tmp_path / "g1_msm_sum.npy")
    assert got.dtype == np.float64 and got.shape == (104,)
    import bench
    bseed, sseed = bench.rank_inputs_seeds(0)
    want = cref.msm_g1(cref.g1_random_bases(bseed, 1 << log_n), cref.fr_random(sseed, 1 << log_n))
    assert (got == want.astype(np.float64)).all()
    assert want[96] == 0  # not the point at infinity: the comparison is not vacuous
