"""Drop-in for the reference's ``coarseAlignFeatMatch`` module: the ``CoarseAlign``
class in its three variants (SURVEY.md section 8b)

  * ``CoarseAlignA`` - evaluation/eval{Hpatch,Corr,KITTI}/coarseAlignFeatMatch.py:35-179
    (``setPair`` + ``getCoarse(Mt) -> H | None``),
  * ``CoarseAlignB`` - evaluation/evalYFCC/coarseAlignFeatMatch.py:35-196,
  * ``CoarseAlignC`` - quick_start/coarseAlignFeatMatch.py:26-173
    (``setSource`` / ``setTarget`` / ``getCoarse(Mt) -> (H, InlierMask)``),

with the reference's constructor signatures, public attributes (``Is``, ``It``,
``IsTensor``, ``ItTensor``, ``featt``, ``scaleList``) and None sentinels.  The 7-scale
source pyramid and the target go through ResNet-50 conv1..layer3 as ONE ragged
NHWC batch; matching and RANSAC are the fused kernels of the library.

ResNet-50 weights: ``models.resnet50(pretrained=True)`` needs a download in the
reference; here they come from ``resnet_state_dict=`` (a torchvision-style
state_dict), ``$RF_RESNET50_WEIGHTS`` (a .pth), or torchvision's own cache.
"""
import os

import numpy as np
import PIL.Image as Image
import torch

from . import model as rfmodel
from . import ops
from . import outil
from .model import FoldedConv
from .ops import Ragged
from .program import LayerProgram

RESNET50_LAYERS = (("layer1", 64, 3, 1), ("layer2", 128, 4, 2), ("layer3", 256, 6, 2))


class _BN:
    def __init__(self, sd, p, eps=1e-5):
        self.weight, self.bias = sd[p + ".weight"], sd[p + ".bias"]
        self.running_mean, self.running_var = sd[p + ".running_mean"], sd[p + ".running_var"]
        self.eps = eps


class ResNet50Conv4:
    """torchvision ResNet-50 conv1..layer3 (quick_start/coarseAlignFeatMatch.py:34-52; the MoCo
    variant model/resnet50.py:107-168 has the same trunk) on the library's conv kernels."""

    def __init__(self, state_dict, device="cuda"):
        self.device = torch.device(device)
        self._sd = {k: v.detach().to(device="cpu", dtype=torch.float32) for k, v in state_dict.items()       # folded on the host
                    if torch.is_tensor(v) and v.dtype.is_floating_point}
        self.program = self._build(32)            # fp32 activations: 'fp32' / 'tf32' engines
        self._program_f16 = None                  # fp16 activations ('f16' engine), built on first use
        self._program_split = None                # split activations ('f16x3' engine), built on first use
        self.out_channels = self.program.chan[-1]

    def _build(self, kalign, fuse_downsample=False):
        """``fuse_downsample`` (split engine): a block's conv3 and its down-sampling 1x1 run as one dual-input GEMM."""
        sd, dev = self._sd, self.device
        P = LayerProgram(3, device=dev)
        if kalign == 64 and os.environ.get("RF_STEM_FUSED", "1") != "0":
            x = P.stem7_fused(0, sd["conv1.weight"], _BN(sd, "bn1"))                 # fp16 engine: patches built in shared memory
        else:
            x = P.stem(0, sd["conv1.weight"], _BN(sd, "bn1"), 2, 3, kalign)          # 7x7/2 stem as im2col + 1x1 conv
        x = P.maxpool(x, 3, 2, 1)
        for layer, planes, blocks, stride in RESNET50_LAYERS:
            for b in range(blocks):
                p = "%s.%d" % (layer, b)
                s = stride if b == 0 else 1
                out = P.conv(x, FoldedConv(sd[p + ".conv1.weight"], _BN(sd, p + ".bn1"), 1, pad=0, device=dev), relu=True)
                out = P.conv(out, FoldedConv(sd[p + ".conv2.weight"], _BN(sd, p + ".bn2"), s, pad=1, device=dev), relu=True)
                r = x
                c3 = FoldedConv(sd[p + ".conv3.weight"], _BN(sd, p + ".bn3"), 1, pad=0, device=dev)
                if (p + ".downsample.0.weight") in sd:
                    ds = FoldedConv(sd[p + ".downsample.0.weight"], _BN(sd, p + ".downsample.1"), s, pad=0, device=dev)
                    if fuse_downsample:
                        x = P.conv_dual(out, x, FoldedConv.concat_k(c3, ds), s, relu=True)
                        continue
                    r = P.conv(x, ds, relu=False)
                x = P.conv(out, c3, relu=True, res=r)
        return P

    def __call__(self, x):
        """x: Ragged [P, 3] normalised images -> Ragged [P/256, 1024] (post-ReLU; fp16 rows under the 'f16' engine, split
        planes under 'f16x3', which ``ops.l2norm`` turns into fp32).  One library call for the whole trunk; the output buffer belongs to the
        program (valid until the next call with these sizes)."""
        eng = rfmodel.get_engine()
        if eng == ops.ENGINE_SPLIT:
            if self._program_split is None:
                # the fp16 program's topology with the weights read as hi / lo planes; conv3 + down-sampling branch fused
                self._program_split = self._build(64, fuse_downsample=True)
            out, ohw = self._program_split.run(x, eng)
        elif eng == ops.ENGINE_F16:
            if self._program_f16 is None:
                self._program_f16 = self._build(64)      # stem patches padded to a multiple of 64 halves
            out, ohw = self._program_f16.run(x, eng)
        else:
            out, ohw = self.program.run(x, eng)
        return Ragged(out, ohw)


def _load_resnet50_state(imageNet, resnet_state_dict):
    if resnet_state_dict is not None:
        return resnet_state_dict
    path = os.environ.get("RF_RESNET50_WEIGHTS")
    if path:
        sd = torch.load(path, map_location="cpu")
        if "model" in sd:           # MoCo checkpoint layout (coarseAlignFeatMatch.py:44-47)
            sd = {k.replace("module.", ""): v for k, v in sd["model"].items()}
        return sd
    if imageNet:
        import torchvision.models as models
        return models.resnet50(weights="IMAGENET1K_V1").state_dict()       # needs the torchvision cache / network
    raise RuntimeError("CoarseAlign: MoCo weights requested; give resnet_state_dict= or $RF_RESNET50_WEIGHTS")


def scale_list(nbScale, scaleR):
    if nbScale == 1:
        return [1]
    return np.linspace(scaleR, 1, nbScale // 2 + 1).tolist() + np.linspace(1, 1 / scaleR, nbScale // 2 + 1).tolist()[1:]


class _CoarseAlignBase:
    resize_mode = "min"

    def _setup(self, nbScale, nbIter, tolerance, transform, minSize, scaleR, imageNet, segNet, resnet_state_dict, verbose):
        if not torch.cuda.is_available():
            raise ops._lib.RFError("CoarseAlign needs a CUDA device: ransac_flow_b200 has no CPU path")
        self.nbIter = nbIter
        self.tolerance = tolerance
        self.net = ResNet50Conv4(_load_resnet50_state(imageNet, resnet_state_dict))
        if segNet:
            raise NotImplementedError("segNet sky masking is out of scope (SURVEY.md section 2 #9); pass segNet=False")
        if transform == "Affine":
            self.Transform = outil.Affine
            self.nbPoint = 3
        else:
            self.Transform = outil.Homography
            self.nbPoint = 4
        self.strideNet = 16
        self.minSize = minSize
        self.scaleList = scale_list(nbScale, scaleR)
        self.device_preproc = False       # True: LANCZOS pyramid on the GPU (bit-exact PIL emulation) instead of on the host
        if verbose:
            print(self.scaleList)

    # -- resizing (host PIL like the reference, or the bit-exact device resampler) -----------------
    def _target_size(self, w, h, minSize):
        if self.resize_mode == "min":
            ratio = min(w / float(minSize), h / float(minSize))
        else:
            ratio = max(w / float(minSize), h / float(minSize))
        new_w, new_h = int(round(w / ratio)), int(round(h / ratio))
        return new_w // self.strideNet * self.strideNet, new_h // self.strideNet * self.strideNet

    def _resize(self, I, minSize):
        new_w, new_h = self._target_size(I.size[0], I.size[1], minSize)
        return I.resize((new_w, new_h), resample=Image.LANCZOS)

    def ResizeMinSize(self, I, minSize):
        return self._resize(I, minSize)

    ResizeMaxSize = ResizeMinSize

    # -- features -------------------------------------------------------------------------------
    @staticmethod
    def _to_device_u8(I):
        a = np.array(I, dtype=np.uint8)          # writable copy
        t = torch.from_numpy(a)
        return t.pin_memory().cuda(non_blocking=True)

    def _features(self, images):
        """list of PIL images (or uint8 CUDA HxWx3 tensors) -> (Ragged normalised conv4 features, list of uint8 CUDA images)."""
        u8 = [im if torch.is_tensor(im) else self._to_device_u8(im) for im in images]
        hw = [(int(t.shape[0]), int(t.shape[1])) for t in u8]
        flat = torch.cat([t.reshape(-1, 3) for t in u8], dim=0) if len(u8) > 1 else u8[0].reshape(-1, 3)
        x = Ragged(ops.preproc_u8(flat, normalize=True), hw)
        f = self.net(x)
        if f.split and outil.corr_precision == 2:
            # engine 'f16x3' + fp16-split correlation: the normalisation writes the correlation's operand planes directly;
            # the fp32 views the reference exposes (featsMultiScale, featt) are rebuilt on first access (__getattr__)
            return Ragged(ops.l2norm_planes(f.data), f.hw), u8
        return Ragged(ops.l2norm(f.data), f.hw), u8

    def _pyramid(self, I_org, sizes):
        """Resize ``I_org`` to each (w, h) in ``sizes``: PIL on the host, or the device resampler."""
        if self.device_preproc:
            src = I_org if torch.is_tensor(I_org) else self._to_device_u8(I_org)
            return [ops.resize_lanczos_u8(src, w, h) for (w, h) in sizes]
        return [I_org.resize((w, h), resample=Image.LANCZOS) for (w, h) in sizes]

    @staticmethod
    def _size_of(I):
        return (int(I.shape[1]), int(I.shape[0])) if torch.is_tensor(I) else I.size

    @staticmethod
    def _as_pil(I):
        return I                              # kept as is; the ``Is`` / ``It`` properties convert lazily

    def _get_img(self, name):
        v = self.__dict__.get(name)
        if torch.is_tensor(v):                # device-resident resized image: materialise the PIL view on first use
            v = Image.fromarray(v.cpu().numpy())
            self.__dict__[name] = v
        return v

    Is = property(lambda self: self._get_img("_Is"), lambda self, v: self.__dict__.__setitem__("_Is", v))
    It = property(lambda self: self._get_img("_It"), lambda self, v: self.__dict__.__setitem__("_It", v))

    @property
    def target_size(self):
        """(w, h) of the resized target without forcing a device->host copy."""
        v = self.__dict__.get("_It")
        return (int(v.shape[1]), int(v.shape[0])) if torch.is_tensor(v) else v.size

    def _to_tensor01(self, u8):
        h, w = int(u8.shape[0]), int(u8.shape[1])
        return ops.preproc_u8(u8.reshape(-1, 3), normalize=False).view(1, h, w, 3).permute(0, 3, 1, 2)

    _LAZY = ("_feats_rows", "featsMultiScale", "_featt_rows", "featt")

    def __getattr__(self, name):
        """fp32 views of features held as fp16 hi / lo planes (engine 'f16x3'): rebuilt (exactly) on first access."""
        if name in _CoarseAlignBase._LAZY:
            d = self.__dict__
            if name in ("_feats_rows", "featsMultiScale") and "_src_planes" in d:
                d["_feats_rows"] = ops.from_split(d["_src_planes"])               # [NA, 1024] rows = feature vectors
                d["featsMultiScale"] = d["_feats_rows"].t()                       # (1024, NA) view, the reference's layout
                return d[name]
            if name in ("_featt_rows", "featt") and "_tgt_planes" in d:
                d["_featt_rows"] = ops.from_split(d["_tgt_planes"])
                d["featt"] = d["_featt_rows"].view(1, self.W2, self.H2, -1).permute(0, 3, 1, 2)
                return d[name]
        raise AttributeError(name)

    def _set_source_feats(self, feats, nS):
        o = feats.offsets()
        self._srcN = o[nS]
        for k in ("_feats_rows", "featsMultiScale", "_src_planes"):
            self.__dict__.pop(k, None)
        if feats.split:
            self._src_planes = feats.data[:, :o[nS]]                  # (hi, lo) planes of the [NA, 1024] rows
        else:
            self._feats_rows = feats.data[:o[nS]]                     # [NA, 1024] rows = feature vectors
            self.featsMultiScale = self._feats_rows.t()               # (1024, NA) view, the reference's layout
        Ws, Hs = [], []
        for i in range(nS):
            _, _, W, H = outil._wh(feats.hw[i][0], feats.hw[i][1], feats.data.device)      # outil.getWHTensor of scale i
            Ws.append(W)
            Hs.append(H)
        self.WMultiScale = torch.cat(Ws)
        self.HMultiScale = torch.cat(Hs)

    def _set_target_feats(self, feats, i):
        o = feats.offsets()
        self.W2, self.H2 = feats.hw[i]
        for k in ("_featt_rows", "featt", "_tgt_planes"):
            self.__dict__.pop(k, None)
        if feats.split:
            self._tgt_planes = feats.data[:, o[i]:o[i + 1]]
        else:
            self.featt = feats.image(i)                               # (1, 1024, h16, w16) view
            self._featt_rows = feats.data[o[i]:o[i + 1]]
        self.WtInt, self.HtInt, self.Wt, self.Ht = outil._wh(self.W2, self.H2, feats.data.device)   # getWHTensor(_Int) of featt

    def _mask16(self, Mt):
        """coarseAlignFeatMatch.py (A) :158-162: 1 - Mt, bilinear to the feature grid, > 0.5."""
        MtExtend = torch.from_numpy((1 - Mt).astype(np.float32)).cuda().unsqueeze(0).unsqueeze(0)
        MtTensor = ops.upsample_bilinear(MtExtend, (self.W2, self.H2))
        return (MtTensor > 0.5).squeeze()

    def skyFromSeg(self, path):
        raise NotImplementedError("segNet sky masking is out of scope (SURVEY.md section 2 #9)")


class CoarseAlignA(_CoarseAlignBase):
    """evaluation/evalHpatch/coarseAlignFeatMatch.py:35-179 (identical in evalCorr / evalKITTI)."""
    resize_mode = "min"

    def __init__(self, nbScale, nbIter, tolerance, transform, minSize, segId=2, segFg=False, scaleR=2, imageNet=True,
                 segNet=True, resnet_state_dict=None, verbose=True):
        self._setup(nbScale, nbIter, tolerance, transform, minSize, scaleR, imageNet, segNet, resnet_state_dict, verbose)

    def setPair(self, Is_org, It_org):
        with torch.no_grad():
            ws, hs = self._size_of(Is_org)
            sizes = [self._target_size(ws, hs, int(self.minSize * s)) for s in self.scaleList]
            IsList = self._pyramid(Is_org, sizes)
            wt, ht = self._size_of(It_org)
            ItR = self._pyramid(It_org, [self._target_size(wt, ht, self.minSize)])[0]
            imgs = IsList + [ItR]
            u8 = [im if torch.is_tensor(im) else self._to_device_u8(im) for im in imgs]
            nS = len(IsList)
            mid = len(self.scaleList) // 2
            self.Is, self.It = self._as_pil(IsList[mid]), self._as_pil(ItR)
            self.IsTensor = self._to_tensor01(u8[mid])
            self.ItTensor = self._to_tensor01(u8[nS])
            feats, _ = self._features(u8)                         # 7 scales + target: one ragged batch
            self._set_source_feats(feats, nS)
            self._set_target_feats(feats, nS)
            # mutual matching once per pair (:139-147), kept on the device; the matched-coordinate attributes the
            # reference caches (:140-147) are materialised lazily (they need the match count on the host)
            if feats.split:
                sp, tp = self._src_planes, self._tgt_planes
                self._idx1, self._idx2, self._count = ops.corr_mutual_nn_presplit(sp[0], sp[1], tp[0], tp[1])
            else:
                self._idx1, self._idx2, self._count = ops.corr_mutual_nn(self._feats_rows, self._featt_rows, outil.corr_precision)
            self._mm = None

    def _matched(self):
        if self._mm is None:
            n = int(self._count.item())
            i1, i2 = self._idx1[:n], self._idx2[:n]
            self._mm = dict(W1MutualMatch=self.WMultiScale[i1], H1MutualMatch=self.HMultiScale[i1], W2MutualMatch=self.Wt[i2],
                            H2MutualMatch=self.Ht[i2], W2MutualMatchInt=self.WtInt[i2], H2MutualMatchInt=self.HtInt[i2])
        return self._mm

    W1MutualMatch = property(lambda self: self._matched()["W1MutualMatch"])
    H1MutualMatch = property(lambda self: self._matched()["H1MutualMatch"])
    W2MutualMatch = property(lambda self: self._matched()["W2MutualMatch"])
    H2MutualMatch = property(lambda self: self._matched()["H2MutualMatch"])
    W2MutualMatchInt = property(lambda self: self._matched()["W2MutualMatchInt"])
    H2MutualMatchInt = property(lambda self: self._matched()["H2MutualMatchInt"])

    def getCoarse_device(self, Mt=None, samples=None):
        """Device-resident ``getCoarse``: no host synchronisation.  Returns (H [9], nbInlier [1], mask [NB], status [1],
        match_count [1]) as CUDA tensors; ``status`` follows RF_RANSAC_* (0 = OK; 1/3 = the reference returns None).
        The RANSAC samples are the reference's own stream: ``ops.philox_words`` draws the generator words
        ``torch.randint(M, (nbIter, 4), device='cuda')`` (utils/outil.py:120) would reduce modulo M, and the kernel reduces
        them with M read on the device - under ``torch.manual_seed(s)`` this path returns what ``getCoarse`` returns, also
        inside a replayed CUDA graph.  ``samples`` (optional, (nbIter, 4) int64 indices): injected sample table instead
        (parity tests drive both paths with the oracle's ``last_samples``)."""
        with torch.no_grad():
            valid16 = None
            if torch.is_tensor(Mt):                          # device-resident mask (480x640 float, 1 = masked)
                MtTensor = ops.upsample_bilinear((1 - Mt).reshape(1, 1, Mt.shape[-2], Mt.shape[-1]).float(), (self.W2, self.H2))
                valid16 = (MtTensor > 0.5).reshape(-1).to(torch.uint8).contiguous()
            elif Mt is not None and np.any(Mt):
                valid16 = self._mask16(Mt).reshape(-1).to(torch.uint8).contiguous()
            match1, match2, _, cnt = ops.build_matches(self._idx1, self._idx2, self._count, self.WMultiScale, self.HMultiScale,
                                                       self.Wt, self.Ht, valid16)
            self.match1, self.match2, self._match_count = match1, match2, cnt
            if samples is not None:
                raw, mode = torch.as_tensor(samples, dtype=torch.int64).to(match1.device).contiguous(), ops.SAMPLES_MOD
            else:
                raw, mode = ops.philox_words(self.nbIter, self.nbPoint, match1.device), ops.SAMPLES_PHILOX64
            H, nb, mask, status = ops.ransac_homography(match1, match2, raw, self.tolerance, 100, cnt, mode)
            return H, nb, mask, status, cnt

    def getCoarse(self, Mt):
        with torch.no_grad():
            MtTensor = self._mask16(Mt)
            valid16 = MtTensor.reshape(-1).to(torch.uint8).contiguous()
            match1, match2, _, cnt = ops.build_matches(self._idx1, self._idx2, self._count, self.WMultiScale, self.HMultiScale,
                                                       self.Wt, self.Ht, valid16)
            n = int(cnt.item())
            match1, match2 = match1[:n], match2[:n]
            self.match1, self.match2 = match1, match2
            if len(match1) < self.nbPoint:
                return None
            bestParam, _, indexInlier, _ = outil.RANSAC(self.nbIter, match1, match2, self.tolerance, self.nbPoint, self.Transform)
            if bestParam is None:
                return None
            return bestParam.astype(np.float32)


class CoarseAlignC(_CoarseAlignBase):
    """quick_start/coarseAlignFeatMatch.py:26-173."""
    resize_mode = "max"
    returns_mask = True

    def __init__(self, nbScale, nbIter, tolerance, transform, minSize, segId=1, segFg=True, imageNet=True, scaleR=2,
                 resnet_state_dict=None, verbose=True):
        self._setup(nbScale, nbIter, tolerance, transform, minSize, scaleR, imageNet, False, resnet_state_dict, verbose)

    def setSource(self, Is_org):
        with torch.no_grad():
            ws, hs = self._size_of(Is_org)
            IsList = self._pyramid(Is_org, [self._target_size(ws, hs, int(self.minSize * s)) for s in self.scaleList])
            feats, u8 = self._features(IsList)
            mid = len(self.scaleList) // 2
            self.Is = self._as_pil(IsList[mid])
            self.IsTensor = self._to_tensor01(u8[mid])
            self._set_source_feats(feats, len(IsList))

    def setTarget(self, It_org):
        with torch.no_grad():
            wt, ht = self._size_of(It_org)
            ItR = self._pyramid(It_org, [self._target_size(wt, ht, self.minSize)])[0]
            feats_raw, u8 = self._features_raw([ItR])
            self.It = self._as_pil(ItR)
            self.ItTensor = self._to_tensor01(u8[0])
            self._featt_raw = feats_raw                               # un-normalised conv4 (masking re-normalises rows)
            self._set_target_feats(Ragged(ops.l2norm(feats_raw.data), feats_raw.hw), 0)

    def _features_raw(self, images):
        u8 = [im if torch.is_tensor(im) else self._to_device_u8(im) for im in images]
        hw = [(int(t.shape[0]), int(t.shape[1])) for t in u8]
        flat = torch.cat([t.reshape(-1, 3) for t in u8], dim=0) if len(u8) > 1 else u8[0].reshape(-1, 3)
        f = self.net(Ragged(ops.preproc_u8(flat, normalize=True), hw))
        return Ragged(f.data.clone(), f.hw), u8        # the program owns its output buffer: keep a private copy

    def getCoarse(self, Mt):
        with torch.no_grad():
            MtTensor = self._mask16(Mt)
            # featt * mask (:143): masked cells become all-zero feature vectors, then re-match (:145)
            featt_rows = ops.l2norm(self._featt_raw.data, MtTensor.reshape(-1).to(torch.uint8).contiguous())
            idx1, idx2, count = ops.corr_mutual_nn(self._feats_rows, featt_rows, outil.corr_precision)
            match1, match2, kept, cnt = ops.build_matches(idx1, idx2, count, self.WMultiScale, self.HMultiScale, self.Wt, self.Ht, None)
            n = int(cnt.item())
            match1, match2, index2 = match1[:n], match2[:n], kept[:n]
            self.match1, self.match2 = match1, match2
            if len(match1) < self.nbPoint:
                return None, []
            bestParam, _, indexInlier, _ = outil.RANSAC(self.nbIter, match1, match2, self.tolerance, self.nbPoint, self.Transform)
            if bestParam is None:
                return None, []
            index2Inlier = index2.cpu().numpy()[indexInlier]
            h16, w16 = self.featt.size()[2], self.featt.size()[3]
            InlierMask = np.zeros((h16, w16), dtype=np.float32)
            Wt, Ht = self.Wt.cpu().numpy(), self.Ht.cpu().numpy()
            InlierMask[((Wt[index2Inlier] / 2 + 0.5) * h16).astype(np.int64), ((Ht[index2Inlier] / 2 + 0.5) * w16).astype(np.int64)] = 1
            return bestParam.astype(np.float32), InlierMask


class CoarseAlignB(CoarseAlignC):
    """evaluation/evalYFCC/coarseAlignFeatMatch.py:35-196: variant C's API with ResizeMinSize."""
    resize_mode = "min"

    def __init__(self, nbScale, nbIter, tolerance, transform, minSize, segId=1, segFg=True, use_cuda=True, imageNet=True,
                 segNet=True, scaleR=2, resnet_state_dict=None, verbose=True):
        if not use_cuda:
            raise ops._lib.RFError("use_cuda=False: ransac_flow_b200 has no CPU path")
        self._setup(nbScale, nbIter, tolerance, transform, minSize, scaleR, imageNet, segNet, resnet_state_dict, verbose)


CoarseAlign = CoarseAlignA
