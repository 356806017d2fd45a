"""The drop-in boundary against the reference's REAL driver scripts (SURVEY 8b).

CPU part: each use a driver script makes of the drop-in modules - names imported from them, constructor calls and their
argument counts / keywords, methods and attributes read on the CoarseAlign object, on the networks and on the warper - is
checked against this package's mirrors.  Those uses were read from the scripts' ASTs by ``oracle/gen_golden.py``
(``gen_script_uses``) and are stored in tests/golden/dropin_script_uses.json, so the check needs no reference checkout.
The GPU part re-enacts the statement sequence of quick_start/align2images.py in a driver of its own, run byte-for-byte
through ``dropin.main`` with torch's own F.grid_sample / F.interpolate between the calls exactly as the script mixes them,
and compares what it saves with the CPU oracle."""
import inspect
import json
import os
import sys

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with open(os.path.join(GOLDEN, "dropin_script_uses.json")) as _f:
    SCRIPT_USES = json.load(_f)
SCRIPTS = ["quick_start/align2images.py", "evaluation/evalHpatch/evaluation.py", "evaluation/evalCorr/evaluation.py",
           "evaluation/evalKITTI/evaluation.py", "evaluation/evalYFCC/evaluation.py", "evaluation/evalHpatch/getResults.py",
           "evaluation/evalCorr/getResults.py", "evaluation/evalKITTI/getResults.py"]


@pytest.mark.parametrize("script", SCRIPTS)
def test_reference_script_api_surface_is_covered(rf, script):
    from ransac_flow_b200 import dropin
    uses = SCRIPT_USES[script]
    variant = dropin.variant_for(os.path.join(os.sep, script))
    cls = {"A": rf.CoarseAlignA, "B": rf.CoarseAlignB, "C": rf.CoarseAlignC}[variant]
    mirrors = {"outil": rf.outil, "model": rf.model, "tgm": rf.kornia_geometry}
    for use in uses["module_attrs"]:
        m, a = use.split(".")
        assert hasattr(mirrors[m], a), "%s uses %s, which the mirror lacks" % (script, use)
    sig = inspect.signature(cls.__init__)
    for call in uses["coarse_align_calls"]:                    # the script's own positional count and keyword names must bind
        args = [None] * (1 + call["nargs"])
        kwargs = {k: None for k in call["keywords"]}
        sig.bind(*args, **kwargs)
    for a in uses["coarse_align_attrs"]:
        assert hasattr(cls, a) or a in ("Is", "It", "IsTensor", "ItTensor", "featt", "scaleList", "Wt", "Ht", "featsMultiScale"), \
            "%s reads CoarseAlign.%s" % (script, a)
    # the bare module names the script imports resolve after install()
    saved = {k: sys.modules.get(k) for k in ("coarseAlignFeatMatch", "outil", "model", "kornia", "kornia.geometry")}
    try:
        dropin.install(variant)
        for name in uses["coarse_align_imports"]:
            assert hasattr(sys.modules["coarseAlignFeatMatch"], name)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


DRIVER = '''
# a driver written against the REFERENCE's module names only (run through ransac_flow_b200.dropin)
from coarseAlignFeatMatch import CoarseAlign
import outil
import model as model
import kornia.geometry as tgm
import argparse, numpy as np, torch, PIL.Image as Image
import torch.nn.functional as F

ap = argparse.ArgumentParser()
for k in ("--img1", "--img2", "--resumePth", "--outdir"):
    ap.add_argument(k, type=str)
args = ap.parse_args()
src, tgt = Image.open(args.img1).convert("RGB"), Image.open(args.img2).convert("RGB")
nets = {"netFeatCoarse": model.FeatureExtractor(), "netCorr": model.CorrNeigh(7), "netFlowCoarse": model.NetFlowCoarse(7),
        "netMatch": model.NetMatchability(7)}
for k in nets:
    nets[k].cuda()
ckpt = torch.load(args.resumePth)
for k in ckpt:
    nets[k].load_state_dict(ckpt[k])
    nets[k].eval()
coarse = CoarseAlign(7, 1000, 0.05, "Homography", 320, segId=1, segFg=True, imageNet=True, scaleR=1.2)
coarse.setSource(src)
coarse.setTarget(tgt)
w, h = coarse.It.size
gx = torch.linspace(-1, 1, steps=w).view(1, 1, -1, 1).expand(1, h, w, 1)
gy = torch.linspace(-1, 1, steps=h).view(1, -1, 1, 1).expand(1, h, w, 1)
warper = tgm.HomographyWarper(h, w)
torch.manual_seed(1000)
H, inl = coarse.getCoarse(np.zeros((h, w)))
Ht = torch.from_numpy(H).unsqueeze(0).cuda()
coarse_flow = warper.warp_grid(Ht)
warped = F.grid_sample(coarse.IsTensor, coarse_flow)                   # torch's own op between the mirrored calls
f1 = F.normalize(nets["netFeatCoarse"](warped.cuda()))
f2 = F.normalize(nets["netFeatCoarse"](coarse.ItTensor))
vol = nets["netCorr"](f1, f2)
down = nets["netFlowCoarse"](vol, False)
grid = torch.cat((gx, gy), dim=3).cuda()
up = F.interpolate(down, size=(grid.size()[1], grid.size()[2]), mode="bilinear").permute(0, 2, 3, 1) + grid
flow = F.grid_sample(coarse_flow.permute(0, 3, 1, 2), up).permute(0, 2, 3, 1).contiguous()
fine = F.grid_sample(coarse.IsTensor, flow)
np.save(args.outdir + "H.npy", H)
np.save(args.outdir + "inlier.npy", inl)
np.save(args.outdir + "flow12.npy", flow.cpu().numpy())
np.save(args.outdir + "fine.npy", fine.cpu().numpy())
coarse.It.save(args.outdir + "resized_target.png")
'''


@pytest.mark.gpu
def test_dropin_runs_a_reference_style_driver_end_to_end(rf, tmp_path, monkeypatch):
    import PIL.Image as Image
    import torch
    from oracle import pair_oracle as PO
    from oracle import synth
    from ransac_flow_b200 import dropin
    from test_gpu_pair import oracle_net
    src, tgt, _ = synth.make_pair(21, 240, 320)
    Image.fromarray(src).save(tmp_path / "a.png")
    Image.fromarray(tgt).save(tmp_path / "b.png")
    rsd = synth.resnet50_conv4_state(0)
    torch.save(rsd, tmp_path / "resnet50.pth")
    net = oracle_net()
    torch.save({"netFeatCoarse": net["netFeatCoarse"], "netCorr": {}, "netFlowCoarse": net["netFlowCoarse"], "netMatch": net["netMatch"]},
               tmp_path / "ckpt.pth")
    drv_dir = tmp_path / "quick_start"
    drv_dir.mkdir()
    (drv_dir / "driver.py").write_text(DRIVER)
    out = str(tmp_path) + "/out_"
    monkeypatch.setenv("RF_RESNET50_WEIGHTS", str(tmp_path / "resnet50.pth"))
    saved = {k: sys.modules.get(k) for k in ("coarseAlignFeatMatch", "outil", "model", "kornia", "kornia.geometry")}
    argv, cwd, path = list(sys.argv), os.getcwd(), list(sys.path)
    monkeypatch.delenv("RF_ENGINE", raising=False)             # the launcher's default engine: f16x3 (fp32-grade tensor cores)
    try:
        dropin.main([str(drv_dir / "driver.py"), "--img1", str(tmp_path / "a.png"), "--img2", str(tmp_path / "b.png"),
                     "--resumePth", str(tmp_path / "ckpt.pth"), "--outdir", out])
    finally:
        assert rf.model.get_engine() == rf.ops.ENGINE_SPLIT
        dropin.select_engine("fp32")
        sys.argv, sys.path[:] = argv, path
        os.chdir(cwd)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    # the oracle on the same pair, fed the samples the driver's seeded torch.randint drew on the GPU
    oc = PO.CoarseAlignOracle(rsd, nbScale=7, nbIter=1000, tolerance=0.05, minSize=320, scaleR=1.2, variant="C")
    oc.setSource(Image.fromarray(src))
    oc.setTarget(Image.fromarray(tgt))
    oc.getCoarse(np.zeros((oc.It.size[1], oc.It.size[0])))          # to learn the match count
    torch.manual_seed(1000)
    oc.raw_samples = torch.randint(len(oc.match1), (1000, 4), device="cuda").cpu().numpy()
    ref = PO.align2images(oc, net, Image.fromarray(src), Image.fromarray(tgt))
    H = np.load(out + "H.npy")
    np.testing.assert_allclose(H, ref["bestPrm"], atol=1e-5)
    assert np.array_equal(np.load(out + "inlier.npy"), ref["inlierMask"])
    assert np.abs(np.load(out + "flow12.npy") - ref["flow12"].numpy()).max() < 1e-3
    assert np.abs(np.load(out + "fine.npy") - ref["img1_fine"].numpy()).max() < 5e-3
    assert Image.open(out + "resized_target.png").size == oc.It.size
