"""CPU: the drop-in modules expose exactly the reference's state-dict schema (keys, order, shapes) and random init.

Compared against the key lists the oracle restates (oracle/smap_torch.py, oracle/refine_torch.py), which
tests/test_oracle_golden.py pins to the reference, and against tests/golden/shim_schema.npz: the keys, shapes, dtypes and
value digests of the reference modules' own state dicts (tests/golden/make_golden.py).  No forward pass: the shims need
a B200 for that."""
import hashlib
import os
import sys
import types

import numpy as np
import torch

from oracle import refine_torch
from smap_b200 import schema

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIMS = os.path.join(ROOT, "smap_b200", "shims")


def _cfg():
    NS = types.SimpleNamespace
    return NS(MODEL=NS(STAGE_NUM=3, UPSAMPLE_CHANNEL_NUM=256), DATASET=NS(KEYPOINT=NS(NUM=15), PAF=NS(NUM=14)),
              OUTPUT_SHAPE=(128, 208), LOSS=NS(OHKM=True, TOPK=8, COARSE_TO_FINE=True))


def _import_from(path, names):
    """import `model.smap` / `model.refinenet` with `path` first on sys.path, isolated from other `model` packages"""
    saved = {k: v for k, v in sys.modules.items() if k == "model" or k.startswith("model.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, path)
    try:
        mods = [__import__(n, fromlist=["x"]) for n in names]
    finally:
        sys.path.remove(path)
        for k in [k for k in sys.modules if k == "model" or k.startswith("model.")]:
            del sys.modules[k]
        sys.modules.update(saved)
    return mods


def test_shim_schemas_match_the_restated_key_lists():
    smap_mod, refine_mod = _import_from(SHIMS, ["model.smap", "model.refinenet"])
    m = smap_mod.SMAP(_cfg())
    sd = m.state_dict()
    want = schema.make_state_dict(0, "identity")
    assert list(sd.keys()) == list(want.keys()) and len(sd) == 1876
    assert all(tuple(sd[k].shape) == tuple(want[k].shape) for k in sd)
    r = refine_mod.RefineNet()
    assert [(k, tuple(v.shape)) for k, v in r.state_dict().items()] == [(k, tuple(s)) for k, s in refine_torch.refine_keys()]


def _check_against_golden(gold, name, sd):
    keys = list(sd.keys())
    assert keys == list(gold[name + "_keys"])
    for k, shape, dtype, digest in zip(keys, gold[name + "_shapes"], gold[name + "_dtypes"], gold[name + "_sha256"]):
        v = sd[k]
        assert "x".join(map(str, v.shape)) == shape and str(v.dtype) == dtype, k
        assert hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest()[:16] == digest, "random init differs at " + k


def test_shims_match_the_reference_modules_key_for_key_and_init_for_init():
    gold = np.load(os.path.join(ROOT, "tests", "golden", "shim_schema.npz"))
    shim_smap, shim_refine = _import_from(SHIMS, ["model.smap", "model.refinenet"])
    torch.manual_seed(0)  # same construction order as the reference -> same RNG stream
    _check_against_golden(gold, "smap", shim_smap.SMAP(_cfg()).state_dict())
    torch.manual_seed(3)
    _check_against_golden(gold, "refinenet", shim_refine.RefineNet().state_dict())
    # strict loading of a state dict with the reference's keys and shapes
    ref_sd = {k: torch.zeros([int(d) for d in s.split("x") if d]) for k, s in zip(gold["refinenet_keys"], gold["refinenet_shapes"])}
    shim_refine.RefineNet().load_state_dict(ref_sd)


def test_oracle_and_product_generators_agree_bit_for_bit():
    """oracle/schema_ref.py (the checker's own generators) and smap_b200/schema.py (the product's) are separate files on
    purpose; the synthetic weights and frames they make must be the same bytes."""
    from oracle import schema_ref

    assert schema_ref.unit_specs() == schema.unit_specs()
    for bn in ("identity", "random"):
        a, b = schema_ref.make_state_dict(3, bn), schema.make_state_dict(3, bn)
        assert list(a.keys()) == list(b.keys())
        assert all(torch.equal(a[k], b[k]) for k in a)
    assert torch.equal(schema_ref.make_input(2, 64, 96, seed=5), schema.make_input(2, 64, 96, seed=5))
