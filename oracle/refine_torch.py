"""ORACLE - TEST INFRASTRUCTURE ONLY (imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs; never by the
product path).

CPU restatement of the RefineNet post-processing step (SURVEY.md 8(f) row f2):
  * model/refinenet.py:5-38      RefineNet_base: 4 x (Linear -> BatchNorm1d(eval) -> ReLU) + Linear, 75 -> 160 -> 256 ->
                                 256 -> 128 -> 45, driven by the reference's state-dict keys (block.layerN.{0,1}.*, block.layer5.*)
  * exps/stage3_root2/test_util.py:102-131  lift_and_refine_3d_pose: root-relative 2D/3D input assembly (fp64 numpy, cast to
                                 fp32), network, root re-addition in float32, score column.
Pinned by tests/golden/refine_cases.npz, produced by the unmodified reference code (tests/golden/make_golden.py) with
its Linear layers computed by linear() below: a BLAS's float32 GEMM sums in an order that depends on the CPU's instruction
set and on the number of rows, so its last bits are not reproducible across machines; linear() and batch_norm() round
in one fixed order on every machine.
"""
import numpy as np
import torch
import torch.nn.functional as F

LAYERS = [(75, 160), (160, 256), (256, 256), (256, 128), (128, 45)]


def refine_keys():
    """[(key, shape)] of the reference RefineNet state dict, in registration order (model/refinenet.py:8-17)."""
    out = []
    for i, (k, n) in enumerate(LAYERS[:4], start=1):
        p = "block.layer%d." % i
        out += [(p + "0.weight", (n, k)), (p + "0.bias", (n,)), (p + "1.weight", (n,)), (p + "1.bias", (n,)),
                (p + "1.running_mean", (n,)), (p + "1.running_var", (n,)), (p + "1.num_batches_tracked", ())]
    out += [("block.layer5.weight", (45, 128)), ("block.layer5.bias", (45,))]
    return out


def _np(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)


def linear(x, weight, bias=None):
    """F.linear for float32 with a fixed summation order: each output is a float32 running sum over k in index order,
    every step the exact float64 product added to it and the sum rounded to float32; the bias is added last.  (MKL's
    AVX-512 SGEMM kernel gives the same bits from 16 rows up.)  Drop-in for torch.nn.functional.linear."""
    x64, w64 = _np(x).astype(np.float64), _np(weight).astype(np.float64)
    acc = np.zeros((x64.shape[0], w64.shape[0]), np.float32)
    for k in range(x64.shape[1]):
        acc = (acc + x64[:, k:k + 1] * w64[:, k]).astype(np.float32)
    if bias is not None:
        acc = acc + _np(bias).astype(np.float32)
    return torch.from_numpy(acc)


def batch_norm(x, mean, var, weight, bias, eps=1e-5):
    """F.batch_norm in eval mode with the roundings of ATen's AVX2 / AVX-512 CPU kernel: alpha = (1 / sqrt(var + eps)) *
    weight in float32 steps; beta = bias - mean * alpha and x * alpha + beta each formed in float64 and rounded once to
    float32."""
    mean, var, weight, bias = (_np(t).astype(np.float32) for t in (mean, var, weight, bias))
    alpha = (np.float32(1) / np.sqrt(var + np.float32(eps))) * weight
    beta = (bias.astype(np.float64) - mean.astype(np.float64) * alpha).astype(np.float32)
    return torch.from_numpy((_np(x).astype(np.float64) * alpha + beta).astype(np.float32))


def mlp(sd, x):
    """model/refinenet.py:19-26 in eval mode.  x: float32 [n,75] -> float32 [n,45]."""
    for i in range(1, 5):
        p = "block.layer%d." % i
        x = linear(x, sd[p + "0.weight"], sd[p + "0.bias"])
        x = batch_norm(x, sd[p + "1.running_mean"], sd[p + "1.running_var"], sd[p + "1.weight"], sd[p + "1.bias"])
        x = F.relu(x)
    return linear(x, sd["block.layer5.weight"], sd["block.layer5.bias"])


def refine_inputs(pred2d, pred3d, root_n=2):
    """test_util.py:103-114 -> float32 [n,75]."""
    n = pred3d.shape[0]
    inp = np.zeros((n, 15, 5), np.float64)
    inp[:, root_n, :2] = pred2d[:, root_n, :2]
    inp[:, root_n, 2:] = pred3d[:, root_n, :3]
    for i in range(n):
        for j in range(15):
            if j != root_n and pred3d[i, j, 3] > 0:
                inp[i, j, :2] = pred2d[i, j, :2] - pred2d[i, root_n, :2]
                inp[i, j, 2:] = pred3d[i, j, :3] - pred3d[i, root_n, :3]
    return inp.reshape(n, 75).astype(np.float32)


def refine(pred2d, pred3d, sd, root_n=2):
    """test_util.py:102-131.  pred2d float32 [n,15,4], pred3d float64 [n,15,4] -> float64 [n,15,4]."""
    n = pred3d.shape[0]
    if n == 0:
        return np.zeros((0, 15, 4), np.float64)
    score = np.ones((n, 15, 1), np.float64)
    score[pred3d[:, root_n, 3] == 0] = 0
    with torch.no_grad():
        pred = mlp(sd, torch.from_numpy(refine_inputs(pred2d, pred3d, root_n))).numpy().reshape(n, 15, 3)
    for i in range(n):
        for j in range(15):
            if j != root_n:
                pred[i, j] += pred3d[i, root_n, :3]  # float32 += float64 -> computed in double, stored as float32
            else:
                pred[i, j] = pred3d[i, j, :3]
    return np.concatenate([pred, score], axis=2)
