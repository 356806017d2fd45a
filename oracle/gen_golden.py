"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference)
on the CPU in the build container.  Test infrastructure; run once:

    python -m oracle.gen_golden            # needs /root/reference, writes tests/golden/

The reference hard-codes ``.cuda()`` (utils/outil.py:86, coarseAlignFeatMatch.py)
and pretrained downloads; the harness monkeypatches, on its own side only,
``torch.Tensor.cuda`` / ``nn.Module.cuda`` -> identity, ``torch.cuda.FloatTensor`` ->
``torch.FloatTensor``, ``torchvision.models.resnet50`` -> seeded random weights
(oracle/synth.py), ``torch.randint`` -> recorded/replayed samples, and stubs for
absent imports (``scipy.misc.imresize``, ``segEval``, ``kornia``).  Functions that
live in driver *scripts* (PredFlowMask, getFlow_all) are extracted from the
script's AST at run time and executed as they are.  No reference source is
copied into this repository; only inputs/outputs are stored.
"""
import ast
import contextlib
import importlib.util
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

from . import synth
from . import warp_oracle as WO

REF = os.environ.get("RF_REFERENCE", "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# torch-CPU threads the golden outputs are computed with: the reduction order of the convolutions depends on it
GOLDEN_THREADS = 8


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@contextlib.contextmanager
def cpu_as_cuda():
    """Harness-side shims so the reference's hard-coded CUDA calls run on the CPU."""
    import torch.nn as nn
    saved = (torch.Tensor.cuda, nn.Module.cuda, getattr(torch.cuda, "FloatTensor", None), torch.cuda.empty_cache)
    torch.Tensor.cuda = lambda self, *a, **k: self
    nn.Module.cuda = lambda self, *a, **k: self
    torch.cuda.FloatTensor = torch.FloatTensor
    torch.cuda.empty_cache = lambda: None
    try:
        yield
    finally:
        torch.Tensor.cuda, nn.Module.cuda = saved[0], saved[1]
        torch.cuda.FloatTensor = saved[2]
        torch.cuda.empty_cache = saved[3]


@contextlib.contextmanager
def replay_randint(samples_list, record):
    """Make ``torch.randint`` (utils/outil.py:120) return prepared sample arrays
    (or record what the real one draws when ``samples_list`` is None)."""
    real = torch.randint
    it = iter(samples_list) if samples_list is not None else None

    def fake(high, size, **kw):
        kw.pop("device", None)
        if it is not None:
            s = torch.from_numpy(np.asarray(next(it))).clone()
        else:
            s = real(high, size, **kw)
        record.append((int(high), s.numpy().copy()))
        return s
    torch.randint = fake
    try:
        yield
    finally:
        torch.randint = real


def ref_outil():
    return _load("ref_outil", os.path.join(REF, "utils", "outil.py"))


def ref_model():
    sys.path.insert(0, os.path.join(REF, "model"))
    try:
        return _load("ref_model", os.path.join(REF, "model", "model.py"))
    finally:
        sys.path.pop(0)


def extract_function(path, name, extra_ns):
    """Compile one top-level function of a reference *script* without running the script."""
    src = open(path).read()
    tree = ast.parse(src)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            code = compile(ast.Module(body=[node], type_ignores=[]), path, "exec")
            ns = dict(extra_ns)
            exec(code, ns)
            return ns[name]
    raise KeyError(name)


def save(name, **arrs):
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
    print("wrote", name, {k: getattr(v, "shape", None) for k, v in arrs.items()})


# --------------------------------------------------------------------------
def gen_outil():
    outil = ref_outil()
    rs = np.random.RandomState(7)
    # getWHTensor / getWHTensor_Int (utils/outil.py:21-29)
    feat = torch.zeros(1, 4, 5, 7)
    W, H = outil.getWHTensor(feat)
    Wi, Hi = outil.getWHTensor_Int(feat)
    save("wh_tensor", h=np.int64(5), w=np.int64(7), W=W.numpy(), H=H.numpy(), Wi=Wi.numpy(), Hi=Hi.numpy())

    # mutualMatching (utils/outil.py:32-45): non-negative unit columns, one all-zero target column
    C, NA, NB = 48, 300, 70
    A = np.abs(rs.randn(C, NA)).astype(np.float32)
    B = np.abs(rs.randn(C, NB)).astype(np.float32)
    B[:, :30] = A[:, rs.permutation(NA)[:30]] + 0.05 * np.abs(rs.randn(C, 30)).astype(np.float32)
    A /= np.linalg.norm(A, axis=0, keepdims=True)
    B /= np.linalg.norm(B, axis=0, keepdims=True)
    B[:, 11] = 0
    i1, i2 = outil.mutualMatching(torch.from_numpy(A), torch.from_numpy(B))
    save("mutual_matching", featA=A, featB=B, index1=i1.numpy(), index2=i2.numpy())

    # Homography / Prediction / ScoreRANSAC / RANSAC (utils/outil.py:68-164)
    cases = {
        "ransac_m120": dict(seed=11, M=120, nbIter=1000, tol=0.05, frac=0.6),
        "ransac_m636": dict(seed=12, M=636, nbIter=1000, tol=0.05, frac=0.6),
        "ransac_grid": dict(seed=13, M=300, nbIter=1000, tol=0.05, frac=0.5, grid=(30, 40)),
        "ransac_remainder_only": dict(seed=14, M=80, nbIter=60, tol=0.05, frac=0.7),
        "ransac_none": dict(seed=15, M=60, nbIter=400, tol=0.0, frac=0.0),
        "ransac_lowinlier": dict(seed=16, M=200, nbIter=1000, tol=0.02, frac=0.15),
    }
    with cpu_as_cuda():
        for name, c in cases.items():
            m1, m2, Hgt = synth.make_matches(c["seed"], c["M"], c["frac"], grid=c.get("grid"))
            samples = synth.draw_samples(c["seed"], c["M"], c["nbIter"])
            rec = []
            with replay_randint([samples], rec):
                H, nb, inl, m2in = outil.RANSAC(c["nbIter"], torch.from_numpy(m1), torch.from_numpy(m2),
                                                c["tol"], 4, outil.Homography)
            # first chunk scores, for a per-hypothesis check
            us = samples[[len(set(r)) == 4 for r in samples.tolist()]]
            n0 = min(100, len(us))
            H0, cnt0 = outil.ScoreRANSAC(torch.from_numpy(m1), torch.from_numpy(m2), c["tol"],
                                         torch.from_numpy(us[:n0]), outil.Homography)
            dets0 = torch.det(H0)
            err0 = outil.Prediction(torch.from_numpy(m1)[None], torch.from_numpy(m2)[None], H0[:8])
            save(name, match1=m1, match2=m2, samples=samples, tol=np.float64(c["tol"]),
                 is_none=np.bool_(H is None),
                 H=(np.zeros((3, 3), np.float32) if H is None else H),
                 nbInlier=np.int64(0 if H is None else nb),
                 isInlier=(np.zeros(c["M"], bool) if H is None else inl),
                 chunk0_H=H0.numpy(), chunk0_counts=cnt0.numpy(), chunk0_dets=dets0.numpy(),
                 chunk0_err8=err0.numpy())


def gen_models():
    model = ref_model()
    torch.manual_seed(0)
    x = torch.rand(1, 3, 48, 64)
    fe = model.FeatureExtractor()
    fe.load_state_dict(synth.feature_extractor_state(0))
    fe.eval()
    y = fe(x)
    save("feature_extractor", x=x.numpy(), y=y.numpy(), seed=np.int64(0))

    a = F.normalize(torch.randn(1, 256, 6, 8))
    b = F.normalize(torch.randn(1, 256, 6, 8))
    corr = model.CorrNeigh(7).eval()(a, b)
    nf = model.NetFlowCoarse(7)
    nf.load_state_dict(synth.net_flow_coarse_state(1))
    nf.eval()
    nm = model.NetMatchability(7)
    nm.load_state_dict(synth.net_matchability_state(2))
    nm.eval()
    save("fine_heads", a=a.numpy(), b=b.numpy(), corr=corr.numpy(), flow=nf(corr, False).numpy(),
         match=nm(corr, False).numpy())

    import torchvision
    net = torchvision.models.resnet50(weights=None)
    missing = net.load_state_dict(synth.resnet50_conv4_state(0), strict=False)
    assert all(k.startswith(("layer4", "fc")) for k in missing.missing_keys), missing
    trunk = torch.nn.Sequential(net.conv1, net.bn1, net.relu, net.maxpool, net.layer1, net.layer2, net.layer3).eval()
    xr = torch.randn(1, 3, 64, 96)
    with torch.no_grad():
        yr = trunk(xr)
    save("resnet50_conv4", x=xr.numpy(), y=yr.numpy(), seed=np.int64(0))


def _ref_networks(model):
    net = {"netFeatCoarse": model.FeatureExtractor(), "netCorr": model.CorrNeigh(7),
           "netFlowCoarse": model.NetFlowCoarse(7), "netMatch": model.NetMatchability(7)}
    net["netFeatCoarse"].load_state_dict(synth.feature_extractor_state(0))
    net["netFlowCoarse"].load_state_dict(synth.net_flow_coarse_state(1))
    net["netMatch"].load_state_dict(synth.net_matchability_state(2))
    for m in net.values():
        m.eval()
    return net


def gen_pred_flow_mask():
    """PredFlowMask as written in the two driver scripts, on a 48x64 pair."""
    model = ref_model()
    net = _ref_networks(model)
    src, tgt, Hgt = synth.make_pair(3, 48, 64)
    Is = torch.from_numpy(src).permute(2, 0, 1)[None].float() / 255
    It = torch.from_numpy(tgt).permute(2, 0, 1)[None].float() / 255
    Hm = torch.tensor(Hgt / np.linalg.norm(Hgt), dtype=torch.float32)[None]
    grid = WO.base_grid(48, 64)
    flowCoarse = WO.warp_grid(Hm, 48, 64)
    with cpu_as_cuda(), torch.no_grad():
        featt = F.normalize(net["netFeatCoarse"](It))
        for tag, script in (("hpatch", "evaluation/evalHpatch/evaluation.py"), ("corr", "evaluation/evalCorr/evaluation.py")):
            fn = extract_function(os.path.join(REF, script), "PredFlowMask", {"torch": torch, "F": F})
            flow12, match, f8, m8 = fn(Is, featt, flowCoarse, grid, net)
            save("pred_flow_mask_" + tag, Is=Is.numpy(), It=It.numpy(), H=Hm.numpy(), flow12=flow12.numpy(),
                 match=match, flowDown8=f8, matchDown8=m8)
    return f8, m8, Hm


def gen_get_flow(tmpdir="/tmp/rf_golden_getflow"):
    """getFlow_all (evaluation/evalHpatch/getResults.py:16-63) on two hypotheses."""
    os.makedirs(tmpdir + "/fine", exist_ok=True)
    os.makedirs(tmpdir + "/coarse", exist_ok=True)
    rs = np.random.RandomState(5)
    flow = (rs.randn(2, 2, 6, 8) * 0.02).astype(np.float32)
    mask = rs.rand(2, 2, 6, 8).astype(np.float32)
    Hs = np.stack([np.eye(3) + rs.uniform(-0.05, 0.05, (3, 3)) for _ in range(2)]).astype(np.float32)
    np.save(tmpdir + "/fine/flow_0_2H.npy", flow)
    np.save(tmpdir + "/fine/mask_0_2H.npy", mask)
    np.save(tmpdir + "/coarse/flow_0_2H.npy", Hs)

    class Warper:                      # kornia is absent: the oracle's restatement stands in
        def __init__(self, h, w):
            self.h, self.w = h, w

        def warp_grid(self, H):
            return WO.warp_grid(H, self.h, self.w)
    fn = extract_function(os.path.join(REF, "evaluation/evalHpatch/getResults.py"), "getFlow_all",
                          {"torch": torch, "F": F, "np": np, "os": os})
    outH, outW = 40, 56
    grid = WO.base_grid(outH, outW)
    fg = fn(0, tmpdir + "/fine", tmpdir + "/coarse", ["flow_0_2H.npy"], True, Warper(outH, outW), grid, 0.5, outW, outH)
    save("get_flow_all", flow=flow, mask=mask, H=Hs, flowGlobal=fg.numpy(), th=np.float64(0.5))


def _coarse_align_common(path, name, stubs):
    for k, v in stubs.items():
        sys.modules.setdefault(k, v)
    sys.path.insert(0, os.path.join(REF, "utils"))
    try:
        return _load(name, path)
    finally:
        sys.path.pop(0)


def gen_coarse_align():
    """CoarseAlign variant C (quick_start) and variant A (evalHpatch) on a 96x128 pair."""
    import PIL.Image as Image
    import torchvision
    src, tgt, Hgt = synth.make_pair(5, 96, 128)
    Is, It = Image.fromarray(src), Image.fromarray(tgt)
    real_resnet50 = torchvision.models.resnet50

    def seeded_resnet50(*a, **k):
        net = real_resnet50(weights=None)
        net.load_state_dict(synth.resnet50_conv4_state(0), strict=False)
        return net
    torchvision.models.resnet50 = seeded_resnet50
    seg = types.ModuleType("segEval")
    res = types.ModuleType("resnet50")
    res.resnet50 = seeded_resnet50
    misc = types.ModuleType("scipy.misc")
    misc.imresize = None
    import scipy
    scipy.misc = misc
    try:
        with cpu_as_cuda():
            # variant C
            modC = _coarse_align_common(os.path.join(REF, "quick_start/coarseAlignFeatMatch.py"), "ref_coarse_C", {})
            cC = modC.CoarseAlign(3, 500, 0.05, "Homography", 128, scaleR=1.5)
            cC.setSource(Is)
            cC.setTarget(It)
            rec = []
            torch.manual_seed(1000)
            with replay_randint(None, rec):
                H, mask = cC.getCoarse(np.zeros((It.size[1], It.size[0])))
            assert H is not None
            save("coarse_align_C", src=src, tgt=tgt, H=H, inlierMask=mask, samples=rec[0][1], nbMatch=np.int64(rec[0][0]),
                 featt=cC.featt.numpy(), feats_sum=cC.featsMultiScale.sum(0).numpy(),
                 WMulti=cC.WMultiScale.numpy(), HMulti=cC.HMultiScale.numpy(),
                 Is=np.asarray(cC.Is), It=np.asarray(cC.It))
            # variant B (evalYFCC): variant C's API with ResizeMinSize and a use_cuda switch
            modB = _coarse_align_common(os.path.join(REF, "evaluation/evalYFCC/coarseAlignFeatMatch.py"), "ref_coarse_B",
                                        {"segEval": seg, "resnet50": res, "scipy.misc": misc})
            cB = modB.CoarseAlign(3, 500, 0.05, "Homography", 96, 1, True, False, True, False, 1.5)
            cB.setSource(Is)
            cB.setTarget(It)
            MtB = np.zeros((cB.It.size[1], cB.It.size[0]), dtype=np.float32)
            MtB[: cB.It.size[1] // 5] = 1            # mask out the top fifth of the target
            rec = []
            with replay_randint(None, rec):
                torch.manual_seed(1000)
                HB, maskB = cB.getCoarse(MtB)
            assert HB is not None
            save("coarse_align_B", src=src, tgt=tgt, Mt=MtB, H=HB, inlierMask=maskB, samples=rec[0][1], nbMatch=np.int64(rec[0][0]),
                 WMulti=cB.WMultiScale.numpy(), HMulti=cB.HMultiScale.numpy(), Is=np.asarray(cB.Is), It=np.asarray(cB.It))
            # variant A
            modA = _coarse_align_common(os.path.join(REF, "evaluation/evalHpatch/coarseAlignFeatMatch.py"), "ref_coarse_A",
                                        {"segEval": seg, "resnet50": res, "scipy.misc": misc})
            cA = modA.CoarseAlign(3, 500, 0.05, "Homography", 96, 2, False, 1.5, True, False)
            cA.setPair(Is, It)
            Mt = np.zeros((cA.It.size[1], cA.It.size[0]), dtype=np.float32)
            Mt[:, : cA.It.size[0] // 4] = 1          # mask out the left quarter of the target
            rec = []
            with replay_randint(None, rec):
                torch.manual_seed(1000)
                HA0 = cA.getCoarse(np.zeros_like(Mt))
                torch.manual_seed(1000)
                HA1 = cA.getCoarse(Mt)
            save("coarse_align_A", src=src, tgt=tgt, H0=HA0, H1=HA1, Mt=Mt,
                 samples0=rec[0][1], samples1=rec[1][1], nbMatch0=np.int64(rec[0][0]), nbMatch1=np.int64(rec[1][0]),
                 W1=cA.W1MutualMatch.numpy(), H1m=cA.H1MutualMatch.numpy(), W2=cA.W2MutualMatch.numpy(),
                 H2m=cA.H2MutualMatch.numpy(), W2i=cA.W2MutualMatchInt.numpy(), H2i=cA.H2MutualMatchInt.numpy(),
                 Is=np.asarray(cA.Is), It=np.asarray(cA.It))
    finally:
        torchvision.models.resnet50 = real_resnet50


class _LabelShim:
    """skimage is not installed: ``measure.label(binary, background=0)`` (8-connected components of a 2-D array, the
    skimage default) is served by ``scipy.ndimage.label`` with a full 3x3 structure.  Harness-side stand-in for an absent
    third-party dependency: the component NUMBERING may differ from skimage's, the components do not."""

    @staticmethod
    def label(binary, background=0):
        import scipy.ndimage as nd
        return nd.label(binary, structure=np.ones((3, 3), dtype=np.int32))[0]


def gen_kitti():
    """The KITTI-only pieces as written in evaluation/evalKITTI: PredFlowMask with a coarse flow of another size than the
    output grid (the second level, evaluation.py:296-302), remove_small_cc (:85-100) and getResults.py's two-level
    getFlow_all (:95-141, with and without the EDT hole filling)."""
    import scipy.ndimage as nd
    model = ref_model()
    net = _ref_networks(model)
    src, tgt, Hgt = synth.make_pair(4, 48, 64)
    Is = torch.from_numpy(src).permute(2, 0, 1)[None].float() / 255
    It = torch.from_numpy(tgt).permute(2, 0, 1)[None].float() / 255
    Hm = torch.tensor(Hgt / np.linalg.norm(Hgt), dtype=torch.float32)[None]
    ev = os.path.join(REF, "evaluation/evalKITTI/evaluation.py")
    with cpu_as_cuda(), torch.no_grad():
        fn = extract_function(ev, "PredFlowMask", {"torch": torch, "F": F})
        # level-2 shapes: images at 48x64 (the "resized" target), coarse flow on that grid, outputs on a 56x80 "original" grid
        flowCoarse = WO.warp_grid(Hm, 48, 64)
        IsSample = F.grid_sample(Is, flowCoarse)
        grid_org = WO.base_grid(56, 80)
        flow12, match, f8, m8 = fn(IsSample, It, flowCoarse, grid_org, net)
        save("kitti_pred_flow_mask", Is=Is.numpy(), It=It.numpy(), H=Hm.numpy(), IsSample=IsSample.numpy(), flow12=flow12.numpy(),
             match=match, flowDown8=f8.numpy(), matchDown8=m8.numpy())
    # remove_small_cc on a blobby map
    rs = np.random.RandomState(9)
    raw = nd.gaussian_filter(rs.rand(60, 96), 2.0)
    m = ((raw - raw.min()) / (raw.max() - raw.min())).astype(np.float32)
    m = np.where(m > 0.55, 1.0, m).astype(np.float32)
    m[3:5, 90:93] = 1.0
    m[40, 2] = 1.0
    rcc = extract_function(ev, "remove_small_cc", {"np": np, "measure": _LabelShim})
    outs = {}
    for cc_th in (0.0, 0.01, 0.05, 1.0):
        outs["out_%g" % cc_th] = rcc(m.copy(), 0.99, cc_th)
    save("kitti_remove_small_cc", match=m, match_th=np.float64(0.99), **outs)
    # getResults.getFlow_all (two levels, files on disk)
    gr = os.path.join(REF, "evaluation/evalKITTI/getResults.py")
    tmp = "/tmp/rf_golden_kitti"
    os.makedirs(tmp, exist_ok=True)
    nH = 2
    Hs = np.stack([np.eye(3) + rs.uniform(-0.04, 0.04, (3, 3)) for _ in range(nH)]).astype(np.float32)
    flowd2 = (rs.randn(nH, 2, 3, 5) * 0.02).astype(np.float32)
    flow = (rs.randn(nH, 2, 6, 10) * 0.01).astype(np.float32)
    mask = np.clip(nd.gaussian_filter(rs.rand(nH, 2, 6, 10), (0, 0, 1, 1)) * 2.2, 0, 1).astype(np.float32)
    np.save(tmp + "/Homograpy_7_2.npy", Hs)
    np.save(tmp + "/Finetune_D2_7_2.npy", flowd2)
    np.save(tmp + "/Finetune_7_2.npy", flow)
    np.save(tmp + "/Finetune_Mask_7_2.npy", mask)
    np.save(tmp + "/BG_7_2H.npy", np.ones((48, 80), bool))

    class Warper:                      # kornia is absent: the oracle's restatement stands in
        def __init__(self, h, w):
            self.h, self.w = h, w

        def warp_grid(self, H):
            return WO.warp_grid(H, self.h, self.w)
    ns = {"torch": torch, "F": F, "np": np, "os": os, "nd": nd, "measure": _LabelShim}
    ns["remove_small_cc"] = extract_function(gr, "remove_small_cc", ns)
    ns["interpolate_flow_match"] = extract_function(gr, "interpolate_flow_match", ns)
    gfa = extract_function(gr, "getFlow_all", ns)
    h, w = 48, 80
    grid = WO.base_grid(h, w)
    res = {}
    for interp in (False, True):
        fg = gfa("7", tmp, 2, "Finetune", Warper(h, w), True, grid, 0.6, 0.01, interp)
        res["flowGlobal_interp%d" % int(interp)] = fg.numpy()
    save("kitti_get_flow_all", H=Hs, flowd2=flowd2, flow=flow, mask=mask, th=np.float64(0.6), cc_th=np.float64(0.01), **res)


def gen_get_flow_corr(tmpdir="/tmp/rf_golden_getflow_corr"):
    """evaluation/evalCorr/getResults.py:78-134 ``getFlow`` (flowGlobal AND matchGlobal) on three hypotheses."""
    import scipy.ndimage as nd
    for d in ("fine", "coarse"):
        os.makedirs(os.path.join(tmpdir, d), exist_ok=True)
    rs = np.random.RandomState(8)
    nH = 3
    flow = (rs.randn(nH, 2, 5, 7) * 0.02).astype(np.float32)
    mask = np.clip(nd.gaussian_filter(rs.rand(nH, 2, 5, 7), (0, 0, 1, 1)) * 2.0, 0, 1).astype(np.float32)
    Hs = np.stack([np.eye(3) + rs.uniform(-0.05, 0.05, (3, 3)) for _ in range(nH)]).astype(np.float32)
    np.save(tmpdir + "/fine/flow_4_3H.npy", flow)
    np.save(tmpdir + "/fine/mask_4_3H.npy", mask)
    np.save(tmpdir + "/fine/maskBG_4_3H.npy", np.ones((40, 56), bool))
    np.save(tmpdir + "/coarse/flow_4_3H.npy", Hs)

    class Warper:                      # kornia is absent: the oracle's restatement stands in
        def __init__(self, h, w):
            self.h, self.w = h, w

        def warp_grid(self, H):
            return WO.warp_grid(H, self.h, self.w)
    tgm = types.SimpleNamespace(HomographyWarper=Warper)
    fn = extract_function(os.path.join(REF, "evaluation/evalCorr/getResults.py"), "getFlow",
                          {"torch": torch, "F": F, "np": np, "os": os, "tgm": tgm})
    fg, mg = fn(4, tmpdir + "/fine", ["flow_4_3H.npy"], tmpdir + "/coarse", tmpdir + "/fine", True, 0.55)
    save("get_flow_corr", flow=flow, mask=mask, H=Hs, flowGlobal=fg.numpy(), matchGlobal=mg.numpy(), th=np.float64(0.55))


def gen_metrics():
    """The two metric FUNCTIONS the getResults scripts define (the rest of their metric code is inline in the scripts):
    ``epe`` (evaluation/evalHpatch/getResults.py:147-157) and ``alignmentError`` (evaluation/evalCorr/getResults.py:15-38)."""
    rs = np.random.RandomState(21)
    epe = extract_function(os.path.join(REF, "evaluation/evalHpatch/getResults.py"), "epe", {"torch": torch})
    a = torch.from_numpy(rs.rand(500, 2).astype(np.float32) * 239)
    b = a + torch.from_numpy(rs.randn(500, 2).astype(np.float32))
    ae = extract_function(os.path.join(REF, "evaluation/evalCorr/getResults.py"), "alignmentError", {"torch": torch, "np": np})
    hB, wB, hA, wA = 48, 64, 40, 72
    flow = torch.from_numpy(rs.uniform(-1, 1, (1, hB, wB, 2)).astype(np.float32))
    match2 = torch.from_numpy((rs.rand(1, hB, wB, 1) > 0.4).astype(np.float32))
    n = 60
    XB, YB = rs.uniform(0, wB - 1, n).astype(np.float32), rs.uniform(0, hB - 1, n).astype(np.float32)
    XA, YA = rs.uniform(0, wA - 1, n).astype(np.float32), rs.uniform(0, hA - 1, n).astype(np.float32)
    # make a third of the keypoints agree with the flow so that the counts are not all zero
    xb, yb = XB.astype(np.int64), YB.astype(np.int64)
    for k in range(0, n, 3):
        XA[k] = (flow[0, yb[k], xb[k], 0].item() + 1) * 0.5 * (wA - 1) + rs.uniform(-2, 2)
        YA[k] = (flow[0, yb[k], xb[k], 1].item() + 1) * 0.5 * (hA - 1) + rs.uniform(-2, 2)
    pixelGrid = np.around(np.logspace(0, np.log10(36), 8).reshape(-1, 8))
    cnt, nb = ae(wB, hB, wA, hA, XA, YA, XB, YB, flow, match2, pixelGrid)
    save("metrics", epe_in=a.numpy(), epe_tgt=b.numpy(), epe=np.float64(epe(a, b).item()), flow=flow.numpy(), match2=match2.numpy(),
         XA=XA, YA=YA, XB=XB, YB=YB, pixelGrid=pixelGrid, dims=np.array([wB, hB, wA, hA]), counts=np.asarray(cnt), nbAlign=np.int64(nb))


DROPIN_SCRIPTS = ["quick_start/align2images.py", "evaluation/evalHpatch/evaluation.py", "evaluation/evalCorr/evaluation.py",
                  "evaluation/evalKITTI/evaluation.py", "evaluation/evalYFCC/evaluation.py", "evaluation/evalHpatch/getResults.py",
                  "evaluation/evalCorr/getResults.py", "evaluation/evalKITTI/getResults.py"]


def script_uses(path):
    """What one driver script uses of the drop-in modules, read from its AST: attributes of ``outil`` / ``model`` / ``tgm``,
    the positional count and keyword names of every ``CoarseAlign(...)`` assignment, the attributes read on names bound to a
    CoarseAlign instance, and the names imported from ``coarseAlignFeatMatch``."""
    tree = ast.parse(open(path).read())
    mod_attrs, ctor_calls, inst_attrs, imports = set(), [], set(), set()
    inst_names = set()
    for node in ast.walk(tree):
        if isinstance(node, ast.Assign) and isinstance(node.value, ast.Call) and isinstance(node.value.func, ast.Name) \
                and node.value.func.id == "CoarseAlign":
            ctor_calls.append({"nargs": len(node.value.args), "keywords": [k.arg for k in node.value.keywords if k.arg]})
            for t in node.targets:
                if isinstance(t, ast.Name):
                    inst_names.add(t.id)
        if isinstance(node, ast.ImportFrom) and node.module == "coarseAlignFeatMatch":
            imports.update(al.name for al in node.names)
    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name):
            if node.value.id in ("outil", "model", "tgm"):
                mod_attrs.add(node.value.id + "." + node.attr)
            if node.value.id in inst_names:
                inst_attrs.add(node.attr)
    return {"module_attrs": sorted(mod_attrs), "coarse_align_calls": ctor_calls,
            "coarse_align_attrs": sorted(inst_attrs), "coarse_align_imports": sorted(imports)}


def gen_script_uses():
    """tests/golden/dropin_script_uses.json: the drop-in API surface each of the reference's driver scripts relies on."""
    import json
    os.makedirs(OUT, exist_ok=True)
    uses = {s: script_uses(os.path.join(REF, s)) for s in DROPIN_SCRIPTS}
    with open(os.path.join(OUT, "dropin_script_uses.json"), "w") as f:
        json.dump(uses, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote dropin_script_uses", {s: len(u["module_attrs"]) for s, u in uses.items()})


def main():
    assert os.path.isdir(REF), "reference checkout not found at %s" % REF
    torch.set_num_threads(GOLDEN_THREADS)
    gen_script_uses()
    gen_outil()
    gen_models()
    gen_pred_flow_mask()
    gen_get_flow()
    gen_kitti()
    gen_get_flow_corr()
    gen_metrics()
    gen_coarse_align()


if __name__ == "__main__":
    main()
