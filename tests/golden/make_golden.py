"""Generate the committed golden fixtures from the CPU oracle (run once in the authoring container;
the oracle itself is `parity unpinned`, see oracle/__init__.py).

  v1_tta.npz : BASELINE.json config 2 -- synthetic 182x218x182 volume (seed 0), benchmark network
               (model 0), z-score (nonzero mask), step 0.5, Gaussian, 8x mirror TTA, fp32 oracle.
               Holds the argmax of a seeded half of the voxels as packed bits, the class-1 probability on
               a stride-6 lattice and both probabilities in a dense 32^3 block (fp32; tests/golden/fixtures.py
               save_v1 / load_v1), so the full-size GPU run is checked without the 7-minute CPU oracle.
  small_*.npz: tiny networks / volumes the oracle also re-computes live in the tests.

usage: python tests/golden/make_golden.py [v1_tta|v1_notta|all]
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import oracle as O  # noqa: E402
from golden import fixtures as F  # noqa: E402


def v1(tta: bool):
    torch.set_num_threads(int(os.environ.get("GOLDEN_THREADS", "6")))
    net = O.build_benchmark_network(0)
    tr = O.OracleTrainer(O.benchmark_plans(), net)
    raw = O.synthetic_flair((182, 218, 182), seed=0)
    data = raw.copy()
    data[0] = O.zscore_nnunet(raw[0], np.where(raw[0] != 0, 0, -1).astype(np.int8), True)
    t0 = time.time()
    seg, probs = tr.predict_preprocessed_data_return_seg_and_softmax(data, do_mirroring=tta, step_size=0.5,
                                                                     use_gaussian=True)
    dt = time.time() - t0
    name = "v1_tta.npz" if tta else "v1_notta.npz"
    F.save_v1(os.path.join(HERE, name), seg.astype(np.uint8), probs,
              zscore_mean_std=np.array([raw[0][raw[0] != 0].mean(), raw[0][raw[0] != 0].std()], dtype=np.float64),
              oracle_seconds=np.array([dt]))
    print(name, "done in %.1fs, fg=%.4f" % (dt, seg.mean()))


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("v1_tta", "all"):
        v1(True)
    if what in ("v1_notta", "all"):
        v1(False)
