"""Generates the committed golden fixtures by importing the REFERENCE (read-only, /root/reference) in the
build container.  The fixtures travel to the GPU box; /root/reference does not.

  backbone_64x96.npz : outputs of the unmodified reference model.smap.SMAP (CPU fp32) on a seeded input with
                       seeded weights (oracle.smap_torch.make_state_dict / make_input are pure generators, the
                       numbers come from the reference module's forward), for both BN settings, plus the
                       flip-TTA merge computed with the reference's own loop (exps/stage3_root2/test.py:55-70).
  lift_cases.npz     : inputs/outputs of the unmodified reference register_pred / generate_relZ / gen_3d_pose
                       (exps/stage3_root2/test_util.py, lib/utils/post_3d.py) driven exactly as
                       exps/stage3_root2/test.py:116-134 does, including cv2 INTER_NEAREST up-sampling.

  lift_gt_cases.npz  : the same with ground truth (register_pred's matching branch, test_util.py:21-39, float64 rows).
  shim_schema.npz    : the state-dict schema and seeded random initialisation of the reference SMAP and RefineNet.

Run:  python tests/golden/make_golden.py
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(REF, "exps", "stage3_root2"))

from oracle.smap_torch import make_input, make_state_dict  # noqa: E402


class NS(types.SimpleNamespace):
    pass


def golden_backbone():
    from model.smap import SMAP

    H, W = 64, 96
    cfg = NS(MODEL=NS(STAGE_NUM=3, UPSAMPLE_CHANNEL_NUM=256), DATASET=NS(KEYPOINT=NS(NUM=15), PAF=NS(NUM=14)),
             OUTPUT_SHAPE=(H // 4, W // 4), LOSS=NS(OHKM=True, TOPK=8, COARSE_TO_FINE=True))
    out = {}
    for bn, seed in (("identity", 11), ("random", 12)):
        m = SMAP(cfg).eval()
        m.load_state_dict(make_state_dict(seed, bn))
        x = make_input(2, H, W, seed=seed + 100)
        with torch.no_grad():
            o2d, dd, rd = m(x)
            f2d, _, _ = m(torch.flip(x, [-1]))
        out["%s_hm2d" % bn] = o2d.numpy().copy()
        out["%s_detd" % bn] = dd.numpy().copy()
        out["%s_rootd" % bn] = rd.numpy().copy()
        # flip merge exactly as test.py:55-70
        kpt_num = 15
        o = o2d.clone()
        f = torch.flip(f2d, dims=[-1])
        keypoint_pair = [0, 1, 2, 9, 10, 11, 12, 13, 14, 3, 4, 5, 6, 7, 8]
        paf_pair = [0, 1, 2, 3, 10, 11, 12, 13, 14, 15, 4, 5, 6, 7, 8, 9, 22, 23, 24, 25, 26, 27, 16, 17, 18, 19, 20, 21]
        pair = keypoint_pair + [v + kpt_num for v in paf_pair]
        for i in range(len(pair)):
            if i >= kpt_num and (i - kpt_num) % 2 == 0:
                o[:, i] += f[:, pair[i]] * -1
            else:
                o[:, i] += f[:, pair[i]]
        o[:, kpt_num:] *= 0.5
        out["%s_hm2d_flipmerged" % bn] = o.numpy().copy()
        out["%s_hm2d_flipraw" % bn] = f2d.numpy().copy()
    np.savez_compressed(os.path.join(HERE, "backbone_64x96.npz"), **out)
    print("backbone golden:", {k: v.shape for k, v in out.items()})


def _reference_env():
    """numpy aliases, PROJECT_HOME and an easydict stub so that exps/stage3_root2/test_util.py imports here."""
    np.int = int
    np.float = float
    os.environ.setdefault("PROJECT_HOME", "/tmp/smap_project_home")
    ed = types.ModuleType("easydict")

    class EasyDict(dict):
        def __getattr__(self, k):
            return self[k]

        def __setattr__(self, k, v):
            self[k] = v

    ed.EasyDict = EasyDict
    sys.modules["easydict"] = ed


def golden_lift():
    _reference_env()
    import cv2
    import test_util as T

    from cases import N_LIFT_CASES, lift_case_inputs

    cases = {}
    for ci in range(N_LIFT_CASES):
        b, det_d, root_d, (iw, ih) = lift_case_inputs(ci)
        s = min(832 / iw, 512 / ih)
        scale = {"scale": np.asarray(s), "img_width": np.asarray(iw), "img_height": np.asarray(ih),
                 "net_width": np.asarray(832), "net_height": np.asarray(512)}
        scale["f_x"] = scale["img_width"]
        scale["f_y"] = scale["img_width"]
        scale["cx"] = scale["img_width"] / 2
        scale["cy"] = scale["img_height"] / 2
        pb = torch.from_numpy(b.copy())
        if len(pb) > 0:
            pb[:, :, :2] *= 4  # test.py:117
        pb = pb.numpy()
        paf_up = cv2.resize(det_d.transpose(1, 2, 0), (832, 512), interpolation=cv2.INTER_NEAREST)  # test.py:123
        rd_up = cv2.resize(root_d, (832, 512), interpolation=cv2.INTER_NEAREST)
        pb = T.register_pred(pb, None)
        if len(pb) == 0:
            p2 = np.zeros((0, 15, 4), np.float32)
            p3 = np.zeros((0, 15, 4), np.float64)
            rdep = np.zeros((0,), np.float64)
        else:
            rdep = T.generate_relZ(pb, paf_up, rd_up, scale)
            p3 = T.gen_3d_pose(pb, rdep, scale)
            p2 = pb
        cases["c%d_pred2d" % ci] = np.asarray(p2, np.float32)
        cases["c%d_pred3d" % ci] = np.asarray(p3, np.float64)
        cases["c%d_rootdepth" % ci] = np.asarray(rdep, np.float64)
    small = cases
    np.savez_compressed(os.path.join(HERE, "lift_cases.npz"), **small)
    print("lift golden:", N_LIFT_CASES, "cases")


def golden_lift_gt():
    """lift_gt_cases.npz: the GT-matching branch - unmodified register_pred(pred, gt_bodys) (test_util.py:21-39; float64
    rows in GT order) followed by generate_relZ / gen_3d_pose with the GT intrinsics of test.py:86-95."""
    _reference_env()
    import cv2
    import test_util as T

    from cases import N_GT_CASES, lift_gt_case_inputs

    cases = {}
    for ci in range(N_GT_CASES):
        b, det_d, root_d, (iw, ih), gt = lift_gt_case_inputs(ci)
        s = min(832 / iw, 512 / ih)
        scale = {"scale": np.asarray(s), "img_width": np.asarray(iw), "img_height": np.asarray(ih),
                 "net_width": np.asarray(832), "net_height": np.asarray(512)}
        scale["f_x"] = gt[0, 0, 7]   # test.py:91-95 (11-column annotations)
        scale["f_y"] = gt[0, 0, 8]
        scale["cx"] = gt[0, 0, 9]
        scale["cy"] = gt[0, 0, 10]
        pb = torch.from_numpy(b.copy())
        if len(pb) > 0:
            pb[:, :, :2] *= 4  # test.py:117
        pb = pb.numpy()
        paf_up = cv2.resize(det_d.transpose(1, 2, 0), (832, 512), interpolation=cv2.INTER_NEAREST)
        rd_up = cv2.resize(root_d, (832, 512), interpolation=cv2.INTER_NEAREST)
        pb = T.register_pred(pb, gt)
        if len(pb) == 0:
            p2 = np.zeros((0, 15, 4), np.float64)
            p3 = np.zeros((0, 15, 4), np.float64)
            rdep = np.zeros((0,), np.float64)
        else:
            assert pb.dtype == np.float64 and len(pb) == len(gt)
            rdep = T.generate_relZ(pb, paf_up, rd_up, scale)
            p3 = T.gen_3d_pose(pb, rdep, scale)
            p2 = pb
        cases["c%d_pred2d" % ci] = np.asarray(p2, np.float64)
        cases["c%d_pred3d" % ci] = np.asarray(p3, np.float64)
        cases["c%d_rootdepth" % ci] = np.asarray(rdep, np.float64)
    np.savez_compressed(os.path.join(HERE, "lift_gt_cases.npz"), **cases)
    print("lift-gt golden:", N_GT_CASES, "cases; matched rows:",
          [int((cases["c%d_pred2d" % c][:, 2, 3] != 0).sum()) for c in range(N_GT_CASES)])


def golden_refine():
    """refine_cases.npz: outputs of the unmodified model/refinenet.py + test_util.lift_and_refine_3d_pose on the lift
    goldens (the 2D/3D poses the reference lift produced), with seeded weights.  torch.nn.functional.linear is replaced
    by oracle.refine_torch.linear (the same float32 linear with one fixed summation order), so that the fixture does not
    depend on which CPU and BLAS kernel made it."""
    _reference_env()
    import test_util as T
    from model.refinenet import RefineNet

    from cases import N_LIFT_CASES, refine_state_dict
    from oracle.refine_torch import linear

    torch.nn.functional.linear = linear

    lift = np.load(os.path.join(HERE, "lift_cases.npz"))
    net = RefineNet().eval()
    net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in refine_state_dict().items()})
    out = {}
    with torch.no_grad():
        for ci in range(N_LIFT_CASES):
            p2, p3 = lift["c%d_pred2d" % ci], lift["c%d_pred3d" % ci]
            if len(p3) == 0:
                out["c%d_refined" % ci] = np.zeros((0, 15, 4), np.float64)
                continue
            out["c%d_refined" % ci] = np.asarray(T.lift_and_refine_3d_pose(p2.copy(), p3.copy(), net, torch.device("cpu"), root_n=2),
                                                 np.float64)
    np.savez_compressed(os.path.join(HERE, "refine_cases.npz"), **out)
    print("refine golden:", {k: v.shape for k, v in list(out.items())[:4]})


def golden_results_json():
    """results_json.txt: json.dump of the dict the unmodified save_result builds (test_util.py:146-158) from the seeded
    records of tests/test_results_json.py::make_records(1, 7)."""
    _reference_env()
    import json

    import test_util as T

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_results_json import make_records

    rec = make_records(1, 7)
    result = {"model_pattern": "CMU", "3d_pairs": []}
    for b in range(len(rec)):
        n = int(rec["count"][b])
        if n == 0:
            continue  # test.py:130-131
        T.save_result(rec["pred2d"][b, :n], rec["pred3d"][b, :n], None, rec["root_depth"][b, :n], "img_%d.jpg" % b, result)
    with open(os.path.join(HERE, "results_json.txt"), "w") as f:
        json.dump(result, f)
    print("results json golden:", len(result["3d_pairs"]), "pairs")


def golden_preprocess():
    """preprocess_digests.json: SHA-256 of the float32 [3,512,832] tensors (and the scale dicts) the unmodified
    dataset/custom_dataset.py CustomDataset.aug_croppad + its torchvision transform produce for the seeded images of
    cases.preprocess_case_image; preprocess_small.npz: one full output (416x256 source) for a value-level comparison."""
    _reference_env()
    import hashlib
    import json

    from dataset.custom_dataset import CustomDataset

    from cases import PRE_GEOMS, preprocess_case_image

    cfg = NS(INPUT=NS(MEANS=[0.406, 0.456, 0.485], STDS=[0.225, 0.224, 0.229]))
    ds = CustomDataset(cfg, "/nonexistent_dataset_dir")
    out = {}
    for ci, (W, H) in enumerate(PRE_GEOMS):
        img = preprocess_case_image(ci)
        ds.image_shape = (img.shape[1], img.shape[0])     # custom_dataset.py:31
        net_img, scale = ds.aug_croppad(img)              # custom_dataset.py:33
        t = ds.transform(net_img).numpy()                 # custom_dataset.py:34
        assert t.shape == (3, 512, 832) and t.dtype == np.float32
        out["c%d" % ci] = {"geom": [W, H], "sha256": hashlib.sha256(np.ascontiguousarray(t).tobytes()).hexdigest(),
                           "u8_sha256": hashlib.sha256(np.ascontiguousarray(net_img).tobytes()).hexdigest(),
                           "scale": {k: float(v) for k, v in scale.items()}}
        if (W, H) == (416, 256):
            np.savez_compressed(os.path.join(HERE, "preprocess_small.npz"), tensor=t[:, ::4, ::4].copy(), ci=ci)
    with open(os.path.join(HERE, "preprocess_digests.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("preprocess golden:", len(out), "cases")


def golden_schema():
    """shim_schema.npz: keys, shapes, dtypes and SHA-256 (first 16 hex digits) of the values of the state dicts of the
    unmodified model/smap.py SMAP (torch.manual_seed(0)) and model/refinenet.py RefineNet (torch.manual_seed(3)) right
    after construction, i.e. their random initialisation."""
    import hashlib

    from model.refinenet import RefineNet
    from model.smap import SMAP

    cfg = NS(MODEL=NS(STAGE_NUM=3, UPSAMPLE_CHANNEL_NUM=256), DATASET=NS(KEYPOINT=NS(NUM=15), PAF=NS(NUM=14)),
             OUTPUT_SHAPE=(128, 208), LOSS=NS(OHKM=True, TOPK=8, COARSE_TO_FINE=True))
    out = {}
    for name, make, seed in (("smap", lambda: SMAP(cfg), 0), ("refinenet", RefineNet, 3)):
        torch.manual_seed(seed)
        sd = make().state_dict()
        out[name + "_keys"] = np.array(list(sd.keys()))
        out[name + "_shapes"] = np.array(["x".join(map(str, v.shape)) for v in sd.values()])
        out[name + "_dtypes"] = np.array([str(v.dtype) for v in sd.values()])
        out[name + "_sha256"] = np.array([hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest()[:16]
                                          for v in sd.values()])
    np.savez_compressed(os.path.join(HERE, "shim_schema.npz"), **out)
    print("schema golden:", len(out["smap_keys"]), "SMAP tensors,", len(out["refinenet_keys"]), "RefineNet tensors")


if __name__ == "__main__":
    which = sys.argv[1:] or ["backbone", "lift", "lift_gt", "refine", "json", "preprocess", "schema"]
    if "schema" in which:
        golden_schema()
    if "lift_gt" in which:
        golden_lift_gt()
    if "preprocess" in which:
        golden_preprocess()
    if "json" in which:
        golden_results_json()
    if "backbone" in which:
        golden_backbone()
    if "lift" in which:
        golden_lift()
    if "refine" in which:
        golden_refine()
