"""The oracle (oracle/*.py) against the golden vectors produced by the unmodified
reference (oracle/gen_golden.py -> tests/golden/).  CPU only."""
import numpy as np
import PIL.Image as Image
import pytest
import torch
import torch.nn.functional as F

from conftest import golden
from oracle import model_oracle as MO
from oracle import outil_oracle as OO
from oracle import pair_oracle as PO
from oracle import synth
from oracle import warp_oracle as WO
from oracle.gen_golden import GOLDEN_THREADS

RANSAC_CASES = ["ransac_m120", "ransac_m636", "ransac_grid", "ransac_remainder_only", "ransac_none", "ransac_lowinlier"]


def test_wh_tensor_bit_exact():
    g = golden("wh_tensor")
    W, H = OO.getWHTensor(int(g["h"]), int(g["w"]))
    assert np.array_equal(W, g["W"]) and np.array_equal(H, g["H"])
    Wi, Hi = OO.getWHTensor_Int(int(g["h"]), int(g["w"]))
    assert np.array_equal(Wi, g["Wi"]) and np.array_equal(Hi, g["Hi"])


def test_mutual_matching_identical_pairs():
    g = golden("mutual_matching")
    i1, i2 = OO.mutualMatching(g["featA"], g["featB"])
    assert np.array_equal(i1, g["index1"]) and np.array_equal(i2, g["index2"])
    assert 11 not in i2                      # the all-zero target column never matches (SURVEY A.2)


@pytest.mark.parametrize("name", RANSAC_CASES)
def test_homography_prediction_score(name):
    g = golden(name)
    us = OO.unique_samples(g["samples"])[: len(g["chunk0_H"])]
    H = OO.Homography(g["match1"][us], g["match2"][us])
    assert np.array_equal(H, g["chunk0_H"])                       # same LAPACK -> same bits
    err = OO.Prediction(g["match1"], g["match2"], H[:8])
    np.testing.assert_allclose(err, g["chunk0_err8"], rtol=2e-4, atol=5e-6)   # x/z is ill-conditioned near z=0; exact fits are pure rounding noise
    dets = OO.det3(H)
    np.testing.assert_allclose(dets, g["chunk0_dets"], rtol=1e-4, atol=1e-7)
    _, counts = OO.ScoreRANSAC(g["match1"], g["match2"], float(g["tol"]), us)
    assert np.array_equal(counts, g["chunk0_counts"])


@pytest.mark.parametrize("name", RANSAC_CASES)
def test_ransac_bit_exact(name):
    g = golden(name)
    H, nb, inl, m2 = OO.RANSAC_from_samples(g["match1"], g["match2"], g["samples"], float(g["tol"]))
    if bool(g["is_none"]):
        assert H is None and nb == 0 and inl == [] and m2 == []
        return
    assert np.array_equal(H, g["H"])
    assert int(nb) == int(g["nbInlier"])
    assert np.array_equal(inl, g["isInlier"])


def test_ransac_typeerror_when_no_model():
    m1, m2, _ = synth.make_matches(3, 40, 0.0)
    s = synth.draw_samples(3, 40, 50)
    with pytest.raises(TypeError):
        OO.RANSAC_from_samples(m1, m2, s, 0.0)


def test_householder_null_vector_matches_lapack_sign():
    m1, m2, _ = synth.make_matches(21, 200, 0.6)
    s = OO.unique_samples(synth.draw_samples(21, 200, 300))
    A = OO.dlt_matrix(m1[s], m2[s])
    _, _, vh = np.linalg.svd(A)
    for n in range(len(A)):
        h = OO.householder_null_vector(A[n])
        assert np.max(np.abs(h - vh[n, 8])) < 1e-9


def test_feature_extractor():
    g = golden("feature_extractor")
    y = MO.feature_extractor(torch.from_numpy(g["x"]), synth.feature_extractor_state(int(g["seed"])))
    np.testing.assert_allclose(y.numpy(), g["y"], rtol=1e-4, atol=1e-4)


def test_fine_heads():
    g = golden("fine_heads")
    corr = MO.corr_neigh(torch.from_numpy(g["a"]), torch.from_numpy(g["b"]))
    np.testing.assert_allclose(corr.numpy(), g["corr"], rtol=1e-5, atol=1e-6)
    flow = MO.net_flow_coarse(torch.from_numpy(g["corr"]), synth.net_flow_coarse_state(1))
    np.testing.assert_allclose(flow.numpy(), g["flow"], rtol=1e-4, atol=1e-6)
    match = MO.net_matchability(torch.from_numpy(g["corr"]), synth.net_matchability_state(2))
    np.testing.assert_allclose(match.numpy(), g["match"], rtol=1e-4, atol=1e-6)


def test_resnet50_conv4():
    g = golden("resnet50_conv4")
    y = MO.resnet50_conv4(torch.from_numpy(g["x"]), synth.resnet50_conv4_state(int(g["seed"])))
    scale = np.abs(g["y"]).max()
    assert np.abs(y.numpy() - g["y"]).max() <= 1e-4 * scale


@pytest.mark.parametrize("tag,m21", [("hpatch", False), ("corr", True)])
def test_pred_flow_mask(tag, m21):
    g = golden("pred_flow_mask_" + tag)
    net = {"netFeatCoarse": synth.feature_extractor_state(0), "netFlowCoarse": synth.net_flow_coarse_state(1),
           "netMatch": synth.net_matchability_state(2)}
    Is, It = torch.from_numpy(g["Is"]), torch.from_numpy(g["It"])
    featt = F.normalize(MO.feature_extractor(It, net["netFeatCoarse"]))
    grid = WO.base_grid(48, 64)
    flowCoarse = WO.warp_grid(g["H"], 48, 64)
    flow12, match, f8, m8 = PO.pred_flow_mask(Is, featt, flowCoarse, grid, net, with_match21=m21)
    np.testing.assert_allclose(f8, g["flowDown8"], atol=1e-6)
    np.testing.assert_allclose(m8, g["matchDown8"], atol=1e-6)
    np.testing.assert_allclose(flow12.numpy(), g["flow12"], atol=1e-5)
    np.testing.assert_allclose(match, g["match"], atol=1e-5)


def test_get_flow_all():
    g = golden("get_flow_all")
    fg, _ = WO.get_flow_all(g["flow"], g["H"], g["mask"], 40, 56, th=float(g["th"]), multiH=True)
    np.testing.assert_allclose(fg.numpy(), g["flowGlobal"], atol=1e-6)


def test_coarse_align_variant_C():
    g = golden("coarse_align_C")
    c = PO.CoarseAlignOracle(synth.resnet50_conv4_state(0), nbScale=3, nbIter=500, tolerance=0.05, minSize=128,
                             scaleR=1.5, variant="C")
    c.setSource(Image.fromarray(g["src"]))
    c.setTarget(Image.fromarray(g["tgt"]))
    assert np.array_equal(np.asarray(c.Is), g["Is"]) and np.array_equal(np.asarray(c.It), g["It"])
    assert np.array_equal(c.WMultiScale, g["WMulti"]) and np.array_equal(c.HMultiScale, g["HMulti"])
    np.testing.assert_allclose(c.featt.numpy(), g["featt"], atol=2e-5)
    real = torch.randint
    torch.randint = lambda high, size, **k: torch.from_numpy(g["samples"]).clone()
    try:
        H, mask = c.getCoarse(np.zeros((c.It.size[1], c.It.size[0])))
    finally:
        torch.randint = real
    assert len(c.match1) == int(g["nbMatch"])
    np.testing.assert_allclose(H, g["H"], atol=1e-5)
    assert np.array_equal(mask, g["inlierMask"])


def test_coarse_align_variant_A():
    g = golden("coarse_align_A")
    c = PO.CoarseAlignOracle(synth.resnet50_conv4_state(0), nbScale=3, nbIter=500, tolerance=0.05, minSize=96,
                             scaleR=1.5, variant="A")
    c.setPair(Image.fromarray(g["src"]), Image.fromarray(g["tgt"]))
    assert np.array_equal(np.asarray(c.It), g["It"])
    assert np.array_equal(c.WMultiScale[c.index1], g["W1"]) and np.array_equal(c.Wt[c.index2], g["W2"])
    assert np.array_equal(c.WtInt[c.index2], g["W2i"]) and np.array_equal(c.HtInt[c.index2], g["H2i"])
    real = torch.randint
    for key_s, key_h, Mt in (("samples0", "H0", np.zeros_like(g["Mt"])), ("samples1", "H1", g["Mt"])):
        torch.randint = lambda high, size, **k: torch.from_numpy(g[key_s]).clone()
        try:
            H = c.getCoarse(Mt)
        finally:
            torch.randint = real
        np.testing.assert_allclose(H, g[key_h], atol=1e-5)
    assert len(c.match1) == int(g["nbMatch1"])


# ---- KITTI extras (evaluation/evalKITTI): golden outputs of the unmodified reference functions --------------------
def test_kitti_remove_small_cc():
    g = golden("kitti_remove_small_cc")
    for key in ("out_0", "out_0.01", "out_0.05", "out_1"):
        got = WO.remove_small_cc(g["match"], float(g["match_th"]), float(key.split("_")[1]))
        assert np.array_equal(got, g[key]), key
    assert (g["out_0.01"] != g["match"]).sum() > 0 and (g["out_0.05"] != g["out_0.01"]).sum() > 0      # the fixture bites


def test_kitti_pred_flow_mask_second_level():
    """evaluation/evalKITTI/evaluation.py:49-81 with the coarse flow on a 48x64 grid and the outputs on a 56x80 grid.
    The oracle runs with the golden's thread count: another count moves flowDown8 by ~2e-7 (reduction order), which the
    full-resolution composition amplifies to ~4e-6 in flow12 and match, above their 1e-6 bar."""
    g = golden("kitti_pred_flow_mask")
    net = {"netFeatCoarse": synth.feature_extractor_state(0), "netFlowCoarse": synth.net_flow_coarse_state(1),
           "netMatch": synth.net_matchability_state(2)}
    flowCoarse = WO.warp_grid(g["H"], 48, 64)
    threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        flow12, match, f8, m8 = PO.pred_flow_mask_kitti(torch.from_numpy(g["IsSample"]), torch.from_numpy(g["It"]), flowCoarse,
                                                        WO.base_grid(56, 80), net)
    finally:
        torch.set_num_threads(threads)
    np.testing.assert_allclose(f8.numpy(), g["flowDown8"], atol=1e-6)
    np.testing.assert_allclose(m8.numpy(), g["matchDown8"], atol=1e-6)
    np.testing.assert_allclose(flow12.numpy(), g["flow12"], atol=1e-6)
    np.testing.assert_allclose(match, g["match"], atol=1e-6)


@pytest.mark.parametrize("interp", [False, True])
def test_kitti_get_flow_all(interp):
    g = golden("kitti_get_flow_all")
    fg, _ = WO.get_flow_all_kitti(g["H"], g["flowd2"], g["flow"], g["mask"], 48, 80, th=float(g["th"]), cc_th=float(g["cc_th"]),
                                  multiH=True, interpolate=interp)
    np.testing.assert_allclose(fg.numpy(), g["flowGlobal_interp%d" % int(interp)], atol=1e-6)


def test_get_flow_corr():
    """evaluation/evalCorr/getResults.py:78-134 (flowGlobal and matchGlobal, three hypotheses)."""
    g = golden("get_flow_corr")
    fg, mg = WO.get_flow_corr(g["flow"], g["H"], g["mask"], th=float(g["th"]), multiH=True)
    np.testing.assert_allclose(fg.numpy(), g["flowGlobal"], atol=1e-6)
    np.testing.assert_allclose(mg.numpy(), g["matchGlobal"], atol=1e-6)


def test_coarse_align_variant_B():
    """evaluation/evalYFCC/coarseAlignFeatMatch.py:35-196 (variant C's API with ResizeMinSize) with a masked target."""
    g = golden("coarse_align_B")
    c = PO.CoarseAlignOracle(synth.resnet50_conv4_state(0), nbScale=3, nbIter=500, tolerance=0.05, minSize=96,
                             scaleR=1.5, variant="B")
    c.setSource(Image.fromarray(g["src"]))
    c.setTarget(Image.fromarray(g["tgt"]))
    assert np.array_equal(np.asarray(c.Is), g["Is"]) and np.array_equal(np.asarray(c.It), g["It"])
    assert np.array_equal(c.WMultiScale, g["WMulti"]) and np.array_equal(c.HMultiScale, g["HMulti"])
    real = torch.randint
    torch.randint = lambda high, size, **k: torch.from_numpy(g["samples"]).clone()
    try:
        H, mask = c.getCoarse(g["Mt"])
    finally:
        torch.randint = real
    assert len(c.match1) == int(g["nbMatch"])
    np.testing.assert_allclose(H, g["H"], atol=1e-5)
    assert np.array_equal(mask, g["inlierMask"]) and mask[0].sum() == 0          # the masked top rows hold no inlier


def test_warp_grid_reference_internal_consistency():
    """The pin the reference itself offers for kornia 0.1.4's ``HomographyWarper.warp_grid`` (not installed, not vendored):
    (1) the drivers add the fine flow to their OWN ``linspace`` grid (evaluation/evalHpatch/evaluation.py:187-189) and sample
    the coarse grid with it, which is only consistent if the identity homography reproduces that grid exactly; (2)
    ``Homography(X, Y)`` fits source = H * target (utils/outil.py:73-81) and its output goes straight into ``warp_grid``
    (evaluation.py:218), so the warped grid must carry the four target sample points onto their source points."""
    for h, w in ((48, 64), (30, 41), (2, 2)):
        ident = WO.warp_grid(np.eye(3, dtype=np.float32)[None], h, w)
        assert torch.equal(ident, WO.base_grid(h, w))
        assert torch.equal(WO.warp_grid(4.0 * np.eye(3, dtype=np.float32)[None], h, w), WO.base_grid(h, w))     # the scale of H cancels (a power of two: exactly)
    rs = np.random.RandomState(0)
    h, w = 33, 47
    # target points = the four corner nodes of the grid (x, y, 1); source points = a random projective image of them
    Y = np.array([[-1, -1, 1], [1, -1, 1], [-1, 1, 1], [1, 1, 1]], dtype=np.float32)
    Hgt = np.eye(3) + rs.uniform(-0.2, 0.2, (3, 3))
    Hgt[2, :2] = rs.uniform(-0.05, 0.05, 2)
    X = (Y @ Hgt.T)
    X = (X / X[:, 2:]).astype(np.float32)
    H = OO.Homography(X[None], Y[None])                       # (1,3,3): maps target -> source
    g = WO.warp_grid(H, h, w)[0].numpy()
    corners = np.stack([g[0, 0], g[0, w - 1], g[h - 1, 0], g[h - 1, w - 1]])
    assert np.abs(corners - X[:, :2]).max() < 1e-5
