"""GPU: association kernels (through the C ABI) bit-exact against the CPU oracle and against the outputs of the
UNMODIFIED reference extension on a B200 (tests/golden/assoc_ref_cases.npz, tests/golden/make_golden_assoc.py)."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import assoc
from smap_b200.synth import make_scene

pytestmark = pytest.mark.gpu
H, W = 128, 208


@pytest.fixture(scope="module")
def eng():
    from smap_b200.engine import Engine

    e = Engine(0, max_batch=8, in_h=512, in_w=832)
    yield e
    e.close()


@pytest.fixture(scope="module")
def ref_gold():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "assoc_ref_cases.npz"))


def scenes(seeds, persons=15):
    ss = [make_scene(s, persons) for s in seeds]
    return (np.stack([s["hms"] for s in ss]), np.stack([s["root_d"] for s in ss]), np.stack([s["det_d"] for s in ss]))


def random_heatmaps(seed, B=2):
    """Backbone-like garbage (random init heads): many peaks, exercises the 127 truncation."""
    rng = np.random.default_rng(seed)
    lo = rng.normal(0, 1, (B, 43, H // 4, W // 4)).astype(np.float32)
    hms = np.kron(lo, np.ones((1, 1, 4, 4), np.float32)) * 0.4 + rng.normal(0, 0.15, (B, 43, H, W)).astype(np.float32)
    rd = rng.uniform(0.5, 3, (B, H, W)).astype(np.float32)
    return hms.astype(np.float32), rd


def edge_cases():
    z = np.zeros((43, H, W), np.float32)
    cases = {"empty": z.copy()}
    a = z.copy()
    a[0, 10:12, 10:12] = 0.9
    a[1, 0, 5] = 0.9
    a[2, 20, 20] = 0.2
    a[2, 64, 100] = 0.7  # a root peak so grouping runs
    a[0, 40, 100] = 0.8
    cases["plateau_border_threshold"] = a
    b = z.copy()
    ys, xs = np.meshgrid(np.arange(2, 126, 4), np.arange(2, 206, 4), indexing="ij")
    for c in range(15):
        b[c, ys, xs] = 0.5 + 0.001 * ((xs + c) % 7)
    b[15:] = np.random.default_rng(0).normal(0, 0.5, (28, H, W))
    cases["saturated_127_peaks"] = b
    c = z.copy()
    c[0, 50, 50] = 1.0
    c[1, 50, 51] = 1.0
    c[2, 90, 90] = 1.0
    c[0, 90, 90] = 1.0
    cases["coincident_and_near"] = c
    return cases


def run_extract(eng, hms):
    p, s = eng.extract(torch.from_numpy(hms).cuda())
    torch.cuda.synchronize()
    return p.cpu().numpy(), s.cpu().numpy()


def check_extract(eng, hms):
    p, s = run_extract(eng, hms)
    for b in range(hms.shape[0]):
        op, os_ = assoc.extract(hms[b])
        assert np.array_equal(p[b], op), "peaks differ (image %d)" % b
        assert np.array_equal(s[b], os_), "pair scores differ (image %d)" % b


def check_connect(eng, hms, rd, root_idx=2, dist_flag=True):
    bodies, counts = eng.connect(torch.from_numpy(hms).cuda(), torch.from_numpy(rd).cuda(), root_idx, dist_flag)
    torch.cuda.synchronize()
    bodies, counts = bodies.cpu().numpy(), counts.cpu().numpy()
    for b in range(hms.shape[0]):
        ob = assoc.connect(hms[b], rd[b], root_idx, dist_flag)
        assert counts[b] == len(ob)
        assert np.array_equal(bodies[b, :len(ob)], ob), "bodies differ (image %d)" % b
        assert not bodies[b, len(ob):].any()


def test_extract_synthetic_scenes_bit_exact(eng):
    hms, _, _ = scenes(range(8))
    check_extract(eng, hms)


def test_extract_random_heatmaps_bit_exact(eng):
    hms, _ = random_heatmaps(1, B=3)
    check_extract(eng, hms)


@pytest.mark.parametrize("name", ["empty", "plateau_border_threshold", "saturated_127_peaks", "coincident_and_near"])
def test_extract_edge_cases(eng, name):
    check_extract(eng, edge_cases()[name][None])


def test_connect_synthetic_scenes_bit_exact(eng):
    hms, rd, _ = scenes(range(10, 18))
    check_connect(eng, hms, rd)
    check_connect(eng, hms, rd, dist_flag=False)


def test_connect_random_heatmaps_bit_exact(eng):
    hms, rd = random_heatmaps(2, B=3)
    check_connect(eng, hms, rd)


def test_connect_neck_root_serial_path(eng):
    hms, rd, _ = scenes(range(20, 22))
    check_connect(eng, hms, rd, root_idx=0)


@pytest.mark.parametrize("name", ["empty", "plateau_border_threshold", "saturated_127_peaks", "coincident_and_near"])
def test_connect_edge_cases(eng, name):
    hms = edge_cases()[name][None]
    rd = np.random.default_rng(3).uniform(0.5, 3, (1, H, W)).astype(np.float32)
    check_connect(eng, hms, rd)


def test_batch_invariance(eng):
    hms, rd, _ = scenes(range(30, 38))
    b8, c8 = eng.connect(torch.from_numpy(hms).cuda(), torch.from_numpy(rd).cuda())
    for i in range(8):
        b1, c1 = eng.connect(torch.from_numpy(hms[i:i + 1]).cuda(), torch.from_numpy(rd[i:i + 1]).cuda())
        assert torch.equal(b1[0], b8[i]) and c1[0] == c8[i]


# ---------------- the unmodified reference extension (its outputs on a B200, stored) ----------------
def reference_cases():
    sets = [scenes(range(40, 44))[:2], random_heatmaps(5, B=2)]
    ec = edge_cases()
    for name in ("plateau_border_threshold", "saturated_127_peaks", "coincident_and_near", "empty"):
        sets.append((ec[name][None], np.random.default_rng(3).uniform(0.5, 3, (1, H, W)).astype(np.float32)))
    return sets


def oracle_cases():
    return scenes(range(50, 53))[:2]


def _sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def test_against_unmodified_reference_extension(eng, ref_gold):
    pairs = [0, 1, 0, 2, 0, 9, 9, 10, 10, 11, 0, 3, 3, 4, 4, 5, 2, 12, 12, 13, 13, 14, 2, 6, 6, 7, 7, 8]
    for c, (hms, rd) in enumerate(reference_cases()):
        th = torch.from_numpy(hms).cuda()
        bodies, counts = eng.connect(th, torch.from_numpy(rd).cuda())
        peaks, scores = eng.extract(th)
        torch.cuda.synchronize()
        for b in range(hms.shape[0]):
            key = "c%d_b%d_" % (c, b)
            assert _sha(hms[b], rd[b]) == str(ref_gold[key + "input_sha256"]), "input generators changed (case %d)" % c
            npk = ref_gold[key + "npeaks"]
            ref_peaks = np.split(ref_gold[key + "peaks"], np.cumsum(npk)[:-1])
            for j in range(15):
                n = int(peaks[b, j, 0, 0].item())
                assert npk[j] == n
                assert np.array_equal(ref_peaks[j], peaks[b, j, 1:n + 1].cpu().numpy())
            for l in range(14):
                nA, nB = int(npk[pairs[2 * l]]), int(npk[pairs[2 * l + 1]])
                assert _sha(scores[b, l, :nA, :nB].cpu().numpy()) == ref_gold[key + "scores_sha256"][l], \
                    "pair scores differ from the reference"
            ref_b = ref_gold[key + "bodies"]
            n = int(counts[b].item())
            assert ref_b.shape == (n, 15, 4)
            assert np.array_equal(ref_b, bodies[b, :n].cpu().numpy()), "bodies differ from the reference"


def test_oracle_matches_unmodified_reference_extension(ref_gold):
    """Pins the CPU oracle itself against the reference (SURVEY.md 8(c))."""
    hms, rd = oracle_cases()
    for b in range(3):
        assert _sha(hms[b], rd[b]) == str(ref_gold["o_b%d_input_sha256" % b]), "input generators changed"
        ob = assoc.connect(hms[b], rd[b])
        assert np.array_equal(ref_gold["o_b%d_bodies" % b], ob)


# ---------------- lift ----------------
def test_lift_matches_oracle(eng):
    from oracle import lift_numpy
    from smap_b200.engine import scale_row

    hms, rd, dd = scenes(range(60, 64))
    bodies, counts = eng.connect(torch.from_numpy(hms).cuda(), torch.from_numpy(rd).cuda())
    geoms = [(1920, 1080), (640, 480), (1000, 1500), (832, 512)]
    scs = [lift_numpy.default_scale(*g) for g in geoms]
    scales = torch.from_numpy(np.stack([scale_row(s) for s in scs])).cuda()
    p2, p3, rdp, co = eng.lift(bodies, counts, torch.from_numpy(dd).cuda(), torch.from_numpy(rd).cuda(), scales)
    torch.cuda.synchronize()
    for b in range(4):
        n = int(counts[b].item())
        o2, o3, ordp = lift_numpy.lift(bodies[b, :n].cpu().numpy(), dd[b], rd[b], scs[b])
        m = len(o2)
        assert int(co[b].item()) == m
        assert np.array_equal(p2[b, :m].cpu().numpy(), o2)
        assert np.array_equal(rdp[b, :m].cpu().numpy(), ordp)
        np.testing.assert_allclose(p3[b, :m].cpu().numpy(), o3, rtol=1e-12, atol=1e-12)
        assert not p3[b, m:].any() and not p2[b, m:].any()


def test_lift_golden_cases(eng):
    """The committed reference-generated fixtures (tests/golden/lift_cases.npz)."""
    import os

    from cases import N_LIFT_CASES, lift_case_inputs
    from oracle import lift_numpy
    from smap_b200.engine import scale_row

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lift_cases.npz"))
    for ci in range(N_LIFT_CASES):
        b, det_d, root_d, (iw, ih) = lift_case_inputs(ci)
        P = len(b)
        bodies = np.zeros((1, 127, 15, 4), np.float32)
        bodies[0, :P] = b
        counts = torch.tensor([P], dtype=torch.int32).cuda()
        scales = torch.from_numpy(scale_row(lift_numpy.default_scale(iw, ih))[None]).cuda()
        p2, p3, rdp, co = eng.lift(torch.from_numpy(bodies).cuda(), counts, torch.from_numpy(det_d[None]).cuda(),
                                   torch.from_numpy(root_d[None]).cuda(), scales)
        m = int(co[0].item())
        assert m == len(g["c%d_pred2d" % ci])
        assert np.array_equal(p2[0, :m].cpu().numpy(), g["c%d_pred2d" % ci])
        assert np.array_equal(rdp[0, :m].cpu().numpy(), g["c%d_rootdepth" % ci])
        np.testing.assert_allclose(p3[0, :m].cpu().numpy(), g["c%d_pred3d" % ci], rtol=1e-12, atol=1e-12)


def test_config4_crowded_batch64(eng):
    """BASELINE.json configs[3]: crowded synthetic scenes (15 persons/frame), a 64-frame batch in chunks of 8."""
    for chunk in range(8):
        hms, rd, _ = scenes(range(1000 + chunk * 8, 1008 + chunk * 8), persons=15)
        check_connect(eng, hms, rd)
