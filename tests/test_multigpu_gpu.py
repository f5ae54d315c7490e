"""GPU: sharding invariance (BASELINE.json config 3, SURVEY.md 8(d)/(e) "result independent of G").

 * one GPU: the records of 16 frames do not depend on how the frames are split into batches (8+8, 4x4, 16x1 ...) nor on the
   handle - the compute half of the invariance, runs on any box;
 * >= 2 GPUs: tests/dist_worker.py under torchrun - frames sharded over ranks, ONE ncclAllGather inside the graph, gathered
   bytes identical to the 1-GPU result on every rank (skipped on single-GPU boxes; builder-side logs of the 2- and 8-GPU
   runs are committed under profiles/)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from smap_b200 import schema

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_records_do_not_depend_on_batch_split_or_handle():
    from smap_b200.engine import Engine, scale_row

    sd = schema.make_state_dict(0, "identity")
    total = 16
    frames = torch.cat([schema.make_input(1, 512, 832, seed=2000 + i) for i in range(total)], 0).cuda()
    sc = dict(scale=832 / 1920, img_width=1920, img_height=1080, net_width=832, net_height=512, f_x=1920.0, f_y=1920.0,
              cx=960.0, cy=540.0)
    row = scale_row(sc)
    results = {}
    for B in (8, 4, 1):
        e = Engine(0, max_batch=B, in_h=512, in_w=832)
        e.load_state_dict(sd)
        scales = torch.from_numpy(np.stack([row] * B)).cuda()
        # 3 passes over the first block exercise eager run -> graph capture -> replay as well
        for _ in range(3):
            first = e.infer_device(frames[:B], scales).cpu()
        rec = torch.cat([e.infer_device(frames[k:k + B], scales).cpu() for k in range(0, total, B)], 0)
        assert torch.equal(rec[:B], first)
        results[B] = rec
        e.close()
    assert torch.equal(results[8], results[4]), "8-frame vs 4-frame batches"
    assert torch.equal(results[8], results[1]), "8-frame vs single-frame batches"


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs (logs of 2- and 8-GPU runs in profiles/)")
def test_sharded_allgather_equals_single_gpu_result():
    world = 8 if torch.cuda.device_count() >= 8 else 2
    port = 29500 + os.getpid() % 200
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_worker.py"), str(8 * world)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "MULTIGPU OK world=%d" % world in out.stdout
