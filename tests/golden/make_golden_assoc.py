"""Golden fixture for the association: outputs of the UNMODIFIED reference extension (dapalib extract / connect, compiled
from the reference's extensions/ into oracle/_ref/ by oracle/build_ref.py) on the seeded inputs of tests/test_assoc_gpu.py.
The extension launches CUDA kernels, so this runs on a GPU; the fixture lets the tests compare against it anywhere.

  assoc_ref_cases.npz, per case c and image b of that case:
    c<c>_b<b>_input_sha256 : SHA-256 of the float32 heat-maps followed by the float32 root-depth map (guards the generators)
    c<c>_b<b>_peaks        : float32 [sum n_j, 3] the 15 per-joint peak lists of extract(), concatenated
    c<c>_b<b>_npeaks       : int32 [15] n_j
    c<c>_b<b>_scores_sha256: SHA-256 of each of the 14 float32 [n_A, n_B] pair-score matrices of extract()
    c<c>_b<b>_bodies       : float32 [P, 15, 4] connect(hms, root_depth, 2, True)
  ("o" cases: connect() only, for the CPU oracle.)

Run:  python tests/golden/make_golden_assoc.py [out.npz]     (needs oracle/_ref built and a CUDA device)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import build_ref  # noqa: E402
from test_assoc_gpu import _sha as sha, oracle_cases, reference_cases  # noqa: E402


def main(path):
    ref = build_ref.load_ref()
    assert ref is not None, "oracle/_ref/dapalib_ref*.so is not built"
    out = {}
    for c, (hms, rd) in enumerate(reference_cases()):
        for b in range(hms.shape[0]):
            key = "c%d_b%d_" % (c, b)
            th = torch.from_numpy(hms[b]).cuda().contiguous()
            pc, sc = ref.extract(th)
            out[key + "input_sha256"] = np.array(sha(hms[b], rd[b]))
            out[key + "npeaks"] = np.array([p.shape[0] for p in pc], np.int32)
            out[key + "peaks"] = torch.cat([p.reshape(-1, 3) for p in pc]).cpu().numpy()
            out[key + "scores_sha256"] = np.array([sha(s.cpu().numpy()) for s in sc])
            out[key + "bodies"] = ref.connect(th, torch.from_numpy(rd[b]), 2, True).cpu().numpy().reshape(-1, 15, 4)
    hms, rd = oracle_cases()
    for b in range(hms.shape[0]):
        out["o_b%d_input_sha256" % b] = np.array(sha(hms[b], rd[b]))
        out["o_b%d_bodies" % b] = ref.connect(torch.from_numpy(hms[b]).cuda(), torch.from_numpy(rd[b]), 2,
                                               True).cpu().numpy().reshape(-1, 15, 4)
    for k, v in out.items():
        if not k.endswith("sha256"):
            assert v.dtype in (np.float32, np.int32), (k, v.dtype)
    np.savez_compressed(path, **out)
    print("assoc golden:", path, {k: v.shape for k, v in out.items() if k.endswith("bodies")})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "assoc_ref_cases.npz"))
