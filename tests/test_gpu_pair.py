"""The API level: CoarseAlign variants, PredFlowMask, the pair loop and getFlow against the
reference's golden outputs and the CPU oracle (fp32 engine; flow tolerance 1e-3 from north_star)."""
import numpy as np
import PIL.Image as Image
import pytest
import torch

from conftest import golden
from oracle import pair_oracle as PO
from oracle import synth
from oracle import warp_oracle as WO

pytestmark = pytest.mark.gpu
FLOW_TOL = 1e-3


def networks(rf):
    net = {"netFeatCoarse": rf.model.FeatureExtractor(), "netCorr": rf.model.CorrNeigh(7),
           "netFlowCoarse": rf.model.NetFlowCoarse(7), "netMatch": rf.model.NetMatchability(7)}
    net["netFeatCoarse"].load_state_dict(synth.feature_extractor_state(0))
    net["netFlowCoarse"].load_state_dict(synth.net_flow_coarse_state(1))
    net["netMatch"].load_state_dict(synth.net_matchability_state(2))
    for m in net.values():
        m.cuda()
        m.eval()
    return net


def oracle_net():
    return {"netFeatCoarse": synth.feature_extractor_state(0), "netFlowCoarse": synth.net_flow_coarse_state(1),
            "netMatch": synth.net_matchability_state(2)}


class fixed_randint:
    def __init__(self, arrays):
        self.arrays = list(arrays)

    def __enter__(self):
        self.real = torch.randint
        it = iter(self.arrays)
        torch.randint = lambda high, size, **k: torch.from_numpy(next(it)).to(k.get("device", "cpu"))
        return self

    def __exit__(self, *a):
        torch.randint = self.real


def test_coarse_align_variant_C_vs_reference(rf):
    g = golden("coarse_align_C")
    c = rf.CoarseAlignC(3, 500, 0.05, "Homography", 128, scaleR=1.5, resnet_state_dict=synth.resnet50_conv4_state(0), verbose=False)
    c.setSource(Image.fromarray(g["src"]))
    c.setTarget(Image.fromarray(g["tgt"]))
    assert np.array_equal(np.asarray(c.Is), g["Is"]) and np.array_equal(np.asarray(c.It), g["It"])
    assert np.array_equal(c.WMultiScale.cpu().numpy(), g["WMulti"]) and np.array_equal(c.HMultiScale.cpu().numpy(), g["HMulti"])
    assert np.abs(c.featt.cpu().numpy() - g["featt"]).max() < 1e-4
    assert tuple(c.featsMultiScale.shape) == (1024, len(g["WMulti"]))
    assert np.abs(c.featsMultiScale.sum(0).cpu().numpy() - g["feats_sum"]).max() < 1e-3
    assert tuple(c.IsTensor.shape) == (1, 3, 96, 128) and float(c.IsTensor.max()) <= 1.0
    with fixed_randint([g["samples"]]):
        H, mask = c.getCoarse(np.zeros((c.It.size[1], c.It.size[0])))
    assert len(c.match1) == int(g["nbMatch"])
    np.testing.assert_allclose(H, g["H"], atol=1e-5)
    assert H.dtype == np.float32 and np.array_equal(mask, g["inlierMask"])


def test_coarse_align_variant_A_vs_reference(rf):
    g = golden("coarse_align_A")
    c = rf.CoarseAlignA(3, 500, 0.05, "Homography", 96, 2, False, 1.5, True, False,
                        resnet_state_dict=synth.resnet50_conv4_state(0), verbose=False)
    c.setPair(Image.fromarray(g["src"]), Image.fromarray(g["tgt"]))
    assert np.array_equal(np.asarray(c.It), g["It"])
    for name, key in (("W1MutualMatch", "W1"), ("H1MutualMatch", "H1m"), ("W2MutualMatch", "W2"), ("H2MutualMatch", "H2m"),
                      ("W2MutualMatchInt", "W2i"), ("H2MutualMatchInt", "H2i")):
        assert np.array_equal(getattr(c, name).cpu().numpy(), g[key]), name
    with fixed_randint([g["samples0"], g["samples1"]]):
        H0 = c.getCoarse(np.zeros_like(g["Mt"]))
        n0 = len(c.match1)
        H1 = c.getCoarse(g["Mt"])
    assert n0 == int(g["nbMatch0"]) and len(c.match1) == int(g["nbMatch1"])
    np.testing.assert_allclose(H0, g["H0"], atol=1e-5)
    np.testing.assert_allclose(H1, g["H1"], atol=1e-5)
    # too few matches -> None (coarseAlignFeatMatch.py:171-172)
    assert c.getCoarse(np.ones_like(g["Mt"])) is None


@pytest.mark.parametrize("tag,m21", [("hpatch", False), ("corr", True)])
def test_pred_flow_mask_vs_reference(rf, tag, m21):
    g = golden("pred_flow_mask_" + tag)
    net = networks(rf)
    Is, It = torch.from_numpy(g["Is"]).cuda(), torch.from_numpy(g["It"]).cuda()
    featt = torch.nn.functional.normalize(net["netFeatCoarse"](It))
    flowCoarse = rf.kornia_geometry.HomographyWarper(48, 64).warp_grid(torch.from_numpy(g["H"]).cuda())
    grid = rf.pipeline.base_grid(48, 64)
    flow12, match, f8, m8 = rf.pipeline.PredFlowMask(Is, featt, flowCoarse, grid, net, with_match21=m21)
    assert np.abs(f8 - g["flowDown8"]).max() < FLOW_TOL and np.abs(m8 - g["matchDown8"]).max() < FLOW_TOL
    assert np.abs(flow12.cpu().numpy() - g["flow12"]).max() < FLOW_TOL
    far = (np.abs(np.abs(g["flow12"]) - 1) > 1e-3).all(-1)[0]
    assert np.abs(match - g["match"])[far].max() < FLOW_TOL
    print("max |flow12 - ref| = %.3g" % np.abs(flow12.cpu().numpy() - g["flow12"]).max())


@pytest.mark.parametrize("eng", ["tf32", "f16"])
@pytest.mark.parametrize("tag,m21", [("hpatch", False), ("corr", True)])
def test_pred_flow_mask_tensor_core_engines_vs_reference(rf, eng, tag, m21):
    """The fine-flow stage of the tensor-core engines ('f16' is bench.py's default) against the UNMODIFIED reference's
    golden PredFlowMask output for a fixed coarse homography: what the reference saves (flowDown8 / matchDown8) and the
    full-resolution flow on the pixels that sample the coarse grid away from its border stay within north_star's 1e-3
    (measured on B200: tf32 1.6e-4 / 1.5e-4 / 1.6e-4, f16 2.4e-4 / 2.0e-4 / 2.2e-4).  Within a pixel of the border
    grid_sample's zero padding makes the flow discontinuous in the sampling position, which amplifies 10-bit-operand
    differences (tf32 1.4e-3, f16 1.05e-3 there): bounded by 3e-3."""
    g = golden("pred_flow_mask_" + tag)
    rf.model.set_engine(eng)
    try:
        net = networks(rf)
        Is, It = torch.from_numpy(g["Is"]).cuda(), torch.from_numpy(g["It"]).cuda()
        featt = torch.nn.functional.normalize(net["netFeatCoarse"](It))
        flowCoarse = rf.kornia_geometry.HomographyWarper(48, 64).warp_grid(torch.from_numpy(g["H"]).cuda())
        flow12, match, f8, m8 = rf.pipeline.PredFlowMask(Is, featt, flowCoarse, rf.pipeline.base_grid(48, 64), net, with_match21=m21)
    finally:
        rf.model.set_engine("fp32")
    d8, dm8 = np.abs(f8 - g["flowDown8"]).max(), np.abs(m8 - g["matchDown8"]).max()
    _, flowUp = WO.compose_fine(torch.from_numpy(g["flowDown8"][:1]), WO.warp_grid(g["H"][:1], 48, 64), WO.base_grid(48, 64), clamp=True)
    fu = flowUp[0].numpy()
    interior = (np.abs(fu[..., 0]) < 1 - 4.0 / 64) & (np.abs(fu[..., 1]) < 1 - 4.0 / 48)
    d = np.abs(flow12.cpu().numpy() - g["flow12"])[0]
    print("[%s %s] |flowDown8 - ref| %.3g, |matchDown8 - ref| %.3g, |flow12 - ref| interior %.3g / all %.3g"
          % (eng, tag, d8, dm8, d[interior].max(), d.max()))
    assert d8 < FLOW_TOL and dm8 < FLOW_TOL and interior.mean() > 0.5 and d[interior].max() < FLOW_TOL
    assert d.max() < 3e-3


def test_get_flow_all_vs_reference(rf):
    g = golden("get_flow_all")
    fg = rf.pipeline.getFlow_all(g["flow"], g["H"], g["mask"], 40, 56, th=float(g["th"]), multiH=True)
    ref, m = WO.get_flow_all(g["flow"], g["H"], g["mask"], 40, 56, th=float(g["th"]), multiH=True)
    far = (np.abs(m.numpy() - float(g["th"])) > 1e-4).all(0)[..., 0]     # merge picks flip only at the threshold
    assert np.abs(fg.cpu().numpy() - g["flowGlobal"])[0][far].max() < 1e-5


def test_multi_hypothesis_loop_runs(rf):
    src, tgt, _ = synth.make_pair(12, 96, 128)
    c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False,
                        resnet_state_dict=synth.resnet50_conv4_state(0), verbose=False)
    torch.manual_seed(1000)
    out = rf.pipeline.align_pair(c, networks(rf), Image.fromarray(src), Image.fromarray(tgt), maxCoarse=3, with_match21=True)
    nH = len(out["flow12"])
    assert 1 <= nH <= 4 and out["H"].shape == (nH, 3, 3) and out["flowDown8"].shape == (nH, 2, 12, 16)


def test_device_preproc_pyramid_equals_host(rf):
    src, tgt, _ = synth.make_pair(13, 120, 160)
    rsd = synth.resnet50_conv4_state(0)
    a = rf.CoarseAlignA(3, 100, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
    b = rf.CoarseAlignA(3, 100, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
    b.device_preproc = True
    a.setPair(Image.fromarray(src), Image.fromarray(tgt))
    b.setPair(Image.fromarray(src), Image.fromarray(tgt))
    assert np.array_equal(np.asarray(a.It), np.asarray(b.It)) and np.array_equal(np.asarray(a.Is), np.asarray(b.Is))
    assert torch.equal(a.featsMultiScale, b.featsMultiScale) and torch.equal(a._idx1, b._idx1)


def test_async_single_hypothesis_path_equals_the_loop(rf):
    """align_pair_single (no host sync until the final D2H) == align_pair(maxCoarse=0) when both use the same samples."""
    src, tgt, _ = synth.make_pair(14, 96, 128)
    Is, It = Image.fromarray(src), Image.fromarray(tgt)
    rsd = synth.resnet50_conv4_state(0)
    net = networks(rf)
    c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
    raw = synth.draw_samples(5, 2 ** 31 - 1, 1000)
    a = rf.pipeline.align_pair_single(c, net, Is, It, samples=raw)
    with fixed_randint([raw % a["nbMatch"]]):
        b = rf.pipeline.align_pair(c, net, Is, It, maxCoarse=0)
    assert np.array_equal(a["H"], b["H"])
    assert np.array_equal(a["flowDown8"], b["flowDown8"]) and np.array_equal(a["matchDown8"], b["matchDown8"])
    assert torch.equal(a["flow12"][0], b["flow12"][0]) and np.array_equal(a["match"][0], b["match"][0])


def test_config1_quick_start_align2images_vs_oracle(rf):
    """BASELINE config 1: a 240x320 pair through quick_start/align2images.py semantics (variant C, ResizeMaxSize,
    minSize 320, nbScale 7, scaleR 1.2, one homography) against the CPU oracle with the same samples."""
    src, tgt, _ = synth.make_pair(21, 240, 320)
    Is, It = Image.fromarray(src), Image.fromarray(tgt)
    rsd = synth.resnet50_conv4_state(0)
    oc = PO.CoarseAlignOracle(rsd, nbScale=7, nbIter=1000, tolerance=0.05, minSize=320, scaleR=1.2, variant="C", seed=1000)
    ref = PO.align2images(oc, oracle_net(), Is, It)
    assert oc.featsMultiScale.shape[1] == 2107 and oc.featt.shape[2] * oc.featt.shape[3] == 300       # SURVEY A.5
    c = rf.CoarseAlignC(7, 1000, 0.05, "Homography", 320, scaleR=1.2, resnet_state_dict=rsd, verbose=False)
    with fixed_randint([oc.last_samples]):
        out = rf.pipeline.align2images(c, networks(rf), Is, It)
    assert ref is not None and out is not None
    same = len(c.match1) == len(oc.match1) and np.array_equal(c.match2.cpu().numpy(), oc.match2)
    print("config1: matches %d/%d identical=%s" % (len(c.match1), len(oc.match1), same))
    assert same, "config 1 (fp32 engine): the match list must be the oracle's"
    np.testing.assert_allclose(out["bestPrm"], ref["bestPrm"], atol=1e-5)
    assert np.array_equal(out["inlierMask"], ref["inlierMask"])
    assert np.abs(out["flowDown"].cpu().numpy() - ref["flowDown"].numpy()).max() < FLOW_TOL
    assert np.abs(out["flow12"].cpu().numpy() - ref["flow12"].numpy()).max() < FLOW_TOL
    assert np.abs(out["img1_fine"].cpu().numpy() - ref["img1_fine"].numpy()).max() < 5e-3


def test_coarse_align_variant_B_vs_reference(rf):
    """CoarseAlignB (evaluation/evalYFCC/coarseAlignFeatMatch.py:35-196) vs the reference's golden H / inlier mask / match
    count with a masked target and the same samples."""
    g = golden("coarse_align_B")
    c = rf.CoarseAlignB(3, 500, 0.05, "Homography", 96, 1, True, True, True, False, 1.5, resnet_state_dict=synth.resnet50_conv4_state(0), verbose=False)
    c.setSource(Image.fromarray(g["src"]))
    c.setTarget(Image.fromarray(g["tgt"]))
    assert np.array_equal(np.asarray(c.Is), g["Is"]) and np.array_equal(np.asarray(c.It), g["It"])
    assert np.array_equal(c.WMultiScale.cpu().numpy(), g["WMulti"]) and np.array_equal(c.HMultiScale.cpu().numpy(), g["HMulti"])
    with fixed_randint([g["samples"]]):
        H, mask = c.getCoarse(g["Mt"])
    assert len(c.match1) == int(g["nbMatch"])
    np.testing.assert_allclose(H, g["H"], atol=1e-5)
    assert np.array_equal(mask, g["inlierMask"])


def test_coarse_align_variant_B_api(rf):
    """evalYFCC variant: C's API with ResizeMinSize; use_cuda=False and segNet=True are refused loudly."""
    src, tgt, _ = synth.make_pair(22, 96, 128)
    rsd = synth.resnet50_conv4_state(0)
    b = rf.CoarseAlignB(3, 500, 0.05, "Homography", 96, 1, True, True, True, False, 1.5, resnet_state_dict=rsd, verbose=False)
    b.setSource(Image.fromarray(src))
    b.setTarget(Image.fromarray(tgt))
    assert b.It.size == (128, 96)
    torch.manual_seed(1000)
    H, mask = b.getCoarse(np.zeros((96, 128)))
    assert H is not None and H.shape == (3, 3) and mask.shape == (6, 8)
    with pytest.raises(rf._lib.RFError):
        rf.CoarseAlignB(3, 500, 0.05, "Homography", 96, 1, True, False, True, False, 1.5, resnet_state_dict=rsd, verbose=False)
    with pytest.raises(NotImplementedError):
        rf.CoarseAlignB(3, 500, 0.05, "Homography", 96, 1, True, True, True, True, 1.5, resnet_state_dict=rsd, verbose=False)


def test_graphed_aligner_replays_match_eager(rf):
    """GraphedAligner (CUDA graph per input size) == align_pair_single on the same inputs, over several replays and
    for two different pairs through the same graph (the samples differ per replay, so compare what is sample independent
    and the full result against an eager run with the graph's own H)."""
    rsd = synth.resnet50_conv4_state(0)
    net = networks(rf)
    c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
    ga = rf.pipeline.GraphedAligner(c, net)
    for seed in (15, 16, 15):
        src, tgt, _ = synth.make_pair(seed, 96, 128)
        s, t = torch.from_numpy(src).cuda(), torch.from_numpy(tgt).cuda()
        out = ga(s, t)
        assert out["H"].shape == (1, 3, 3) and out["nbMatch"] > 4 and out["nbInlier"] >= 4
        # eager fine stage with the graph's H must give the graph's flow
        c2 = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
        c2.setPair(Image.fromarray(src), Image.fromarray(tgt))
        featt = rf.pipeline.fine_features(net["netFeatCoarse"], c2.ItTensor)
        fc = rf.ops.warp_grid(torch.from_numpy(out["H"]).cuda(), 96, 128)
        f12, m, f8, _ = rf.pipeline.PredFlowMask_device(c2.IsTensor, featt, fc, (96, 128), net)
        assert np.abs(f8.cpu().numpy() - out["flowDown8"]).max() < 1e-6
        assert torch.allclose(f12, out["flow12"][0], atol=1e-6)
    assert len(ga.graphs) == 1


def test_device_resident_multi_hypothesis_loop_equals_host_loop(rf):
    """align_pair_device (masks on the device, 12 bytes per hypothesis to the host) == align_pair (host numpy masks, the
    reference's loop) when both see the same samples."""
    src, tgt, _ = synth.make_pair(12, 96, 128)
    Is, It = Image.fromarray(src), Image.fromarray(tgt)
    rsd = synth.resnet50_conv4_state(0)
    net = networks(rf)
    c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
    raws = [synth.draw_samples(30 + k, 2 ** 31 - 1, 1000) for k in range(6)]
    a = rf.pipeline.align_pair_device(c, net, Is, It, maxCoarse=3, with_match21=True, samples=raws)
    nH = len(a["flow12"])
    assert 1 <= nH <= 4 and len(a["nbMatch"]) == nH
    # the host loop draws one sample set per getCoarse call, including a last rejected / failed one
    counts = a["nbMatch"] + [a["nbMatch"][-1]] * 3
    with fixed_randint([raws[k] % max(counts[k], 1) for k in range(6)]):
        b = rf.pipeline.align_pair(c, net, Is, It, maxCoarse=3, with_match21=True)
    n = min(nH, len(b["flow12"]))
    assert n >= 1
    np.testing.assert_allclose(a["H"][:n], b["H"][:n], atol=1e-6)
    np.testing.assert_allclose(a["flowDown8"][:n], b["flowDown8"][:n], atol=1e-6)
    np.testing.assert_allclose(a["match"][0], b["match"][0], atol=1e-6)


def test_kitti_shaped_pair_runs(rf):
    """BASELINE config 5 shape: 376x1241 pair at coarseSize 800 (nbScale 3, scaleR 1.2 -> source grids 198x60 / 165x50 / 137x41,
    NA = 25747; target 165x50, NB = 8250), one hypothesis through the sync-free path.  No oracle at this size (minutes on the
    CPU): checks sizes, finiteness and that the coarse homography of a synthetic homography pair is recovered."""
    src, tgt, Hgt = synth.make_pair(31, 376, 1241)
    rsd = synth.resnet50_conv4_state(0)
    net = networks(rf)
    c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 800, 2, False, 1.2, True, False, resnet_state_dict=rsd, verbose=False)
    c.device_preproc = True
    torch.manual_seed(1000)
    out = rf.pipeline.align_pair_single(c, net, torch.from_numpy(src).cuda(), torch.from_numpy(tgt).cuda())
    assert c._feats_rows.shape == (25747, 1024) and c._featt_rows.shape == (8250, 1024)
    assert out["H"].shape == (1, 3, 3) and np.isfinite(out["H"]).all() and out["nbMatch"] >= 4
    h, w = c.target_size[1], c.target_size[0]
    assert (h, w) == (800, 2640) and out["flow12"][0].shape == (1, h, w, 2) and torch.isfinite(out["flow12"][0]).all()
    assert out["flowDown8"].shape == (1, 2, h // 8, w // 8)
    Hn = out["H"][0] / out["H"][0][2, 2]
    print("KITTI-shaped pair: %d matches, %d inliers, |H - Hgt|max = %.3f" % (out["nbMatch"], out["nbInlier"], np.abs(Hn - Hgt / Hgt[2, 2]).max()))


def test_concurrent_aligner_equals_graphed_aligner(rf):
    """ConcurrentAligner: two pairs in flight on two streams (own models / graphs / pinned buffers per lane) return, pair
    by pair, what a single GraphedAligner returns.  The deterministic stages (pyramid, trunk, correlation -> match count)
    must be identical - they would not be if the lanes shared a buffer; RANSAC draws its samples inside the graphs, so
    H / flow are only checked for being a valid result of the same shape."""
    rf.model.set_engine("f16")
    rf.outil.corr_precision = 2
    try:
        rsd = synth.resnet50_conv4_state(0)

        def make_models():
            c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
            return c, networks(rf)
        pairs = [tuple(torch.from_numpy(a).pin_memory() for a in synth.make_pair(30 + i, 96, 128)[:2]) for i in range(4)]
        single = rf.pipeline.GraphedAligner(*make_models())
        ref = [single(s, t) for s, t in pairs]
        multi = rf.pipeline.ConcurrentAligner(make_models, lanes=2)
        outs = multi(pairs[:2]) + multi(pairs[2:])
        outs2 = multi(pairs[:2]) + multi(pairs[2:3])          # buffers are reused; a short batch is fine
        assert len(outs) == 4 and len(outs2) == 3
        outs3 = multi.run(pairs + pairs[:3])                  # 7 pairs through 2 lanes without round barriers, results in input order
        assert len(outs3) == 7
        for o, r in zip(outs3, ref + ref[:3]):
            assert o["nbMatch"] == r["nbMatch"] and o["flowDown8"].shape == r["flowDown8"].shape
        for o, r in list(zip(outs, ref)) + list(zip(outs2, ref[:3])):
            assert o["nbMatch"] == r["nbMatch"] and o["nbMatch"] >= 4
            assert len(o["H"]) == len(r["H"])
            if len(o["H"]):
                assert o["H"].shape == (1, 3, 3) and np.isfinite(o["H"]).all() and o["nbInlier"] >= 4
                assert o["flowDown8"].shape == r["flowDown8"].shape and np.isfinite(o["flowDown8"]).all()
                assert o["match"][0].shape == r["match"][0].shape
            print("pair: matches %d, inliers single %d / concurrent %d" % (o["nbMatch"], r["nbInlier"], o["nbInlier"]))
        g0 = multi.lanes[0].graphs[next(iter(multi.lanes[0].graphs))]
        assert multi.replayed_kernels == 14 * g0["n_kernels"] and g0["n_kernels"] > 50
    finally:
        rf.model.set_engine("fp32")
        rf.outil.corr_precision = 0


def test_concurrent_aligner_lanes_are_reproducible_after_manual_seed(rf):
    """Each lane's graphs draw their RANSAC samples from the lane's own generator state, so lanes released together do not
    race on one generator's offset: after ConcurrentAligner.manual_seed the same pairs give bit-identical results."""
    rf.model.set_engine("f16")
    rf.outil.corr_precision = 2
    try:
        rsd = synth.resnet50_conv4_state(0)

        def make_models():
            c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
            return c, networks(rf)
        pairs = [tuple(torch.from_numpy(a).cuda() for a in synth.make_pair(40 + i, 96, 128)[:2]) for i in range(4)]
        multi = rf.pipeline.ConcurrentAligner(make_models, lanes=4)
        multi.prepare(*pairs[0])
        runs = []
        for _ in range(2):
            multi.manual_seed(3)
            runs.append(multi.run(pairs * 3))
        for a, b in zip(*runs):
            assert np.array_equal(a["H"], b["H"]) and a["nbInlier"] == b["nbInlier"] and np.array_equal(a["flowDown8"], b["flowDown8"])
    finally:
        rf.model.set_engine("fp32")
        rf.outil.corr_precision = 0


def test_graphed_aligner_results_survive_later_replays_and_graph_eviction(rf):
    """ADVICE r1: (1) a result kept across replays must not be overwritten (flow12 used to alias the graph's static buffer);
    (2) graphs are LRU-bounded and an evicted graph takes the activation buffers only it used with it - replaying the
    survivors and re-capturing the evicted size afterwards still gives the eager results."""
    rsd = synth.resnet50_conv4_state(0)
    net = networks(rf)
    c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
    ga = rf.pipeline.GraphedAligner(c, net, max_graphs=2)
    sizes = [(96, 128), (80, 112), (64, 96)]
    pairs = [tuple(torch.from_numpy(a).cuda() for a in synth.make_pair(40 + i, h, w)[:2]) for i, (h, w) in enumerate(sizes)]

    def eager(i):
        c2 = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 96, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
        c2.device_preproc = True
        torch.manual_seed(7)
        return rf.pipeline.align_pair_single(c2, net, *pairs[i])

    torch.manual_seed(7)
    first = ga(*pairs[0])
    keep = first["flow12"][0].clone()
    torch.manual_seed(8)
    second = ga(*pairs[0])                                    # same size: the same graph replayed with other samples
    assert torch.equal(first["flow12"][0], keep) and first["flow12"][0].data_ptr() != second["flow12"][0].data_ptr()
    for i in (1, 2, 0, 1, 2):                                 # three sizes through two graph slots: evictions + re-captures
        ga.prepare(*pairs[i])                                 # (re-)capture first: its warm-up runs draw from the generator
        torch.manual_seed(7)
        out = ga(*pairs[i])
        ref = eager(i)
        assert len(ga.graphs) <= 2
        assert np.array_equal(out["H"], ref["H"]) and np.array_equal(out["flowDown8"], ref["flowDown8"])
        assert torch.equal(out["flow12"][0], ref["flow12"][0])
