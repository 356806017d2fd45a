"""The per-pair path above the modules: ``PredFlowMask`` and the multi-hypothesis driver
loop of the evaluation scripts, and ``getFlow_all`` / ``getFlow`` of the getResults scripts,
restated on the library's kernels (no file IO, no metrics: those stay in the drivers).

  PredFlowMask : evaluation/evalHpatch/evaluation.py:23-55, evaluation/evalCorr/evaluation.py:29-59
  align_pair   : evaluation/evalHpatch/evaluation.py:172-243
  getFlow_all  : evaluation/evalHpatch/getResults.py:16-63 (after the np.load calls)
  KITTI        : evaluation/evalKITTI/evaluation.py:49-100,216-344 (two-level flow, small connected components),
                 evaluation/evalKITTI/getResults.py:95-141 (two-level recomposition)
"""

import numpy as np
import torch

from . import _lib, model, ops
from .kornia_geometry import HomographyWarper
from .ops import Ragged


def base_grid(h, w, device="cuda"):
    """evaluation/evalHpatch/evaluation.py:187-189."""
    gy = torch.linspace(-1, 1, steps=h, device=device).view(1, -1, 1, 1).expand(1, h, w, 1)
    gx = torch.linspace(-1, 1, steps=w, device=device).view(1, 1, -1, 1).expand(1, h, w, 1)
    return torch.cat((gx, gy), dim=3).contiguous()


def fine_features(netFeatCoarse, img):
    """F.normalize(netFeatCoarse(img)) as a Ragged (rows = pixels)."""
    f = netFeatCoarse.forward_ragged(Ragged.from_nchw(img))
    return Ragged(ops.l2norm(f.data), f.hw)


def PredFlowMask_device(IsTensor, featt, flowCoarse, size, network, with_match21=False, align_corners=False, ItTensor=None, feat_box=None):
    """PredFlowMask without the device->host copies: returns CUDA tensors
    (flow12 (1,H,W,2), match (1,1,H,W), flowDown8 (1,2,h8,w8), matchDown8 (2,1,h8,w8) = [match12, match21]).
    ``featt = None`` with ``ItTensor``: the target's fine features are computed HERE, in one two-image batch with the warped
    source's (twice the tiles per FeatureExtractor launch: 8.1 waves on 148 SMs instead of 2 x 4.05, half the launches);
    ``feat_box`` (a dict) receives them for the next hypotheses."""
    with torch.no_grad():
        IsSample = ops.grid_sample(IsTensor, flowCoarse, align_corners)
        if featt is None:
            f = fine_features(network["netFeatCoarse"], torch.cat([IsSample, ItTensor], dim=0))
            n = f.data.shape[0] // 2
            fs, ft = Ragged(f.data[:n], f.hw[:1]), Ragged(f.data[n:], f.hw[1:])
            if feat_box is not None:
                feat_box["featt"] = ft
        else:
            fs = fine_features(network["netFeatCoarse"], IsSample)
            ft = featt if isinstance(featt, Ragged) else Ragged.from_nchw(featt)
        k = network["netCorr"].kernelSize
        ld = network["netFlowCoarse"].CORR_LD
        tc = model.fine_engine()            # 0 plain fp32, 1 TF32-rounded, 2 fp16, 4 split planes: the operand type of the heads
        if tc == ops.ENGINE_SPLIT:              # one launch: corr12 standalone + the two-image [corr12 ; corr21] tensor, split planes
            corr12, both = ops.corr_neigh_pair_split(ft, fs, k, ld)
        else:                                   # both volumes from one launch, already laid out as the two-image batch
            corr12, corr21, both = ops.corr_neigh_pair(ft, fs, k, ld, tc)
        # the two heads are independent: the flow head (one image: 152 tiles in its widest layer, i.e. one full wave + 4 tiles on 148
        # SMs) runs on the side stream and fills the tails of the matchability head's kernels (two images) and vice versa
        main, side = torch.cuda.current_stream(), _side_stream()
        if side != main:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                flowDown8 = network["netFlowCoarse"].forward_ragged(corr12)
            corr12.data.record_stream(side)
            mboth = network["netMatch"].forward_ragged(both)                # (2,1,h8,w8): match12, match21 in one batch
            main.wait_stream(side)
            flowDown8.record_stream(main)
        else:
            flowDown8 = network["netFlowCoarse"].forward_ragged(corr12)
            mboth = network["netMatch"].forward_ragged(both)                # (2,1,h8,w8): match12, match21 in one batch
        flow12, match, _ = ops.compose_fine(flowDown8, mboth[0:1], mboth[1:2] if with_match21 else None, flowCoarse,
                                            clamp=True, align_corners=align_corners)
        return flow12, match, flowDown8, mboth


def PredFlowMask(IsTensor, featt, flowCoarse, grid, network, with_match21=False, align_corners=False):
    """Same inputs/outputs as the reference function (evaluation/evalHpatch/evaluation.py:23-55; ``with_match21``:
    evaluation/evalCorr/evaluation.py:54).  ``featt`` may be the (1,256,h8,w8) tensor the reference passes or a Ragged
    from ``fine_features``.  ``grid`` is only used for its size (the base grid is regenerated inside the fused
    composition kernel)."""
    H, W = grid.size()[1], grid.size()[2]
    flow12, match, flowDown8, mboth = PredFlowMask_device(IsTensor, featt, flowCoarse, (H, W), network, with_match21, align_corners)
    out = torch.cat([match.reshape(-1), flowDown8.reshape(-1), mboth.reshape(-1)]).cpu().numpy()   # one D2H
    n0, n1 = H * W, flowDown8.numel()
    return (flow12, out[:n0].reshape(H, W), out[n0:n0 + n1].reshape(tuple(flowDown8.shape)),
            out[n0 + n1:].reshape(1, 2, flowDown8.shape[2], flowDown8.shape[3]))


_pinned = {}
_side = {}


def _side_stream():
    d = torch.cuda.current_device()
    if d not in _side:
        _side[d] = torch.cuda.Stream(device=d)
    return _side[d]


def _to_host(t):
    """One asynchronous D2H into a cached pinned buffer + a stream synchronise."""
    key = (t.numel(), t.dtype)
    if key not in _pinned:
        _pinned[key] = torch.empty(t.numel(), dtype=t.dtype).pin_memory()
    h = _pinned[key]
    h.copy_(t.reshape(-1), non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return h.numpy()


def _single_device(coarseModel, network, Is, It, with_match21, samples=None):
    """Device part of the single-hypothesis path: everything queued on the current stream, nothing read back."""
    coarseModel.setPair(Is, It)
    Itw, Ith = coarseModel.target_size
    Hd, nb, mask, status, cnt = coarseModel.getCoarse_device(None, samples)
    flowCoarse = ops.warp_grid(Hd.view(1, 3, 3), Ith, Itw)
    # target and warped source through the FeatureExtractor as one two-image batch (bit-identical features)
    flow12, match, f8, mboth = PredFlowMask_device(coarseModel.IsTensor, None, flowCoarse, (Ith, Itw), network, with_match21,
                                                   ItTensor=coarseModel.ItTensor)
    packed = torch.cat([status.float(), cnt.float(), nb.float(), Hd, match.reshape(-1), f8.reshape(-1), mboth.reshape(-1)])
    return packed, flow12, (Ith, Itw), tuple(f8.shape)


def _unpack_single(host, flow12, size, f8shape):
    Ith, Itw = size
    st, n0, n8 = int(host[0]), Ith * Itw, int(np.prod(f8shape))
    if st != 0:                                    # the reference's `if bestPara is None: break` (evaluation.py:215-216)
        if st == 2:
            raise TypeError("'NoneType' object is not subscriptable")     # utils/outil.py:162
        return dict(H=np.zeros((0,)), flowDown8=np.zeros((0,)), matchDown8=np.zeros((0,)), flow12=[], match=[],
                    nbInlier=0, nbMatch=int(host[1]))
    H = host[3:12].reshape(1, 3, 3).astype(np.float32)
    o = 12
    return dict(H=H, flowDown8=host[o + n0:o + n0 + n8].reshape(f8shape),
                matchDown8=host[o + n0 + n8:].reshape(1, 2, f8shape[2], f8shape[3]),
                flow12=[flow12], match=[host[o:o + n0].reshape(Ith, Itw)], nbInlier=int(host[2]), nbMatch=int(host[1]))


def align_pair_single(coarseModel, network, Is, It, with_match21=False, samples=None):
    """The single-hypothesis case of the evaluation loop (maxCoarse = 0, no background mask) with NO host
    synchronisation until the results are fetched: matching, RANSAC (device-side match count), warp, fine flow and
    composition are queued back to back, then one pinned D2H brings back status, H, the matchability map and the /8
    tensors.  Same outputs as ``align_pair``; under ``torch.manual_seed(s)`` also the same RANSAC samples (the reference's
    stream, ``ops.philox_words``).  ``samples``: an injected (nbIter, 4) index table instead."""
    packed, flow12, size, f8shape = _single_device(coarseModel, network, Is, It, with_match21, samples)
    return _unpack_single(_to_host(packed).copy(), flow12, size, f8shape)


class GraphedAligner:
    """``align_pair_single`` captured once in a CUDA graph per input size and replayed per pair: the ~140 kernel
    launches of a pair (pyramid, ResNet-50 trunk, matching, RANSAC, fine flow) cost one graph launch on the host.
    Inputs are copied into static device buffers (H2D when they are host tensors / arrays); the RANSAC samples are
    drawn inside the graph (torch's graph-safe Philox offsets), so successive replays use fresh samples."""

    def __init__(self, coarseModel, network, with_match21=False, warmup=2, max_graphs=8):
        self.coarse, self.net, self.m21, self.warmup = coarseModel, network, with_match21, warmup
        self.coarse.device_preproc = True
        self.graphs = {}                # insertion-ordered: least recently used first
        self.max_graphs = max_graphs    # datasets with many image sizes (HPatches, MegaDepth, YFCC): LRU-bounded graph memory
        self.replayed_kernels = 0       # library kernels executed through graph replays (they bypass rf_launch_count)
        self.rng = None                 # generator state the graphs draw their samples from (None: the default CUDA generator's)

    def _device(self, s_in, t_in):
        """The device work of one pair, queued on the current stream: (packed results, flow12 | None, (H, W), flowDown8 shape)."""
        return _single_device(self.coarse, self.net, s_in, t_in, self.m21)

    def _unpack(self, host, flow12, size, f8shape):
        return _unpack_single(host, flow12, size, f8shape)

    def _programs(self):
        """Every LayerProgram whose cached activation buffers a captured graph of this aligner points into."""
        progs = [p for p in (self.coarse.net.program, self.coarse.net._program_f16, self.coarse.net._program_split) if p is not None]
        for m in self.net.values():
            progs += list(getattr(m, "_fold", {}).values())
        return progs

    def _evict(self):
        """Drop the least recently used graph TOGETHER with the activation buffers only it refers to: the graph holds raw
        pointers into the layer programs' cached buffers, so neither may outlive the other (ADVICE r1: use-after-free)."""
        key = next(iter(self.graphs))
        torch.cuda.synchronize()
        rec = self.graphs.pop(key)
        live = set()
        for r in self.graphs.values():
            live |= r["prog_keys"]
        for prog in self._programs():
            for k in [k for k in prog._compiled if (id(prog), k) in rec["prog_keys"] and (id(prog), k) not in live]:
                del prog._compiled[k]
        del rec

    def _build(self, Is, It):
        if self.rng is None:
            return self._capture(Is, It)
        d = torch.cuda.current_device()
        gen = torch.cuda.default_generators[d]
        default_state = gen.graphsafe_get_state()
        gen.graphsafe_set_state(self.rng)            # the graph registers (and its replays advance) this state, not the default
        try:
            return self._capture(Is, It)
        finally:
            gen.graphsafe_set_state(default_state)

    def _capture(self, Is, It):
        dev = torch.device("cuda", torch.cuda.current_device())
        s_in = torch.empty(tuple(Is.shape), dtype=torch.uint8, device=dev)
        t_in = torch.empty(tuple(It.shape), dtype=torch.uint8, device=dev)
        s_in.copy_(Is)
        t_in.copy_(It)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(self.warmup):                       # eager runs: func attributes, TMA maps, caches, buffers
                self._device(s_in, t_in)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.cuda.graph(g):
            packed, flow12, size, f8shape = self._device(s_in, t_in)
        # the compiled program entries (activation buffers) this graph's kernels point into: every entry whose image-set
        # signature the warm-up / capture of THIS input size touched
        touched = {(id(p), k) for p in self._programs() for k in p._compiled if k in p.__dict__.get("_touched", ())}
        for p in self._programs():
            p.__dict__["_touched"] = set()
        return dict(n_kernels=_lib.launch_count() - n0, graph=g, s_in=s_in, t_in=t_in, packed=packed, flow12=flow12, size=size, f8shape=f8shape,
                    prog_keys=touched)

    def prepare(self, Is, It):
        """Capture (once) the graph for this pair of input sizes; returns its record."""
        if isinstance(Is, np.ndarray):
            Is, It = torch.from_numpy(Is), torch.from_numpy(It)
        key = (tuple(Is.shape), tuple(It.shape))
        if key not in self.graphs:
            while self.max_graphs and len(self.graphs) >= self.max_graphs:
                self._evict()
            for p in self._programs():
                p.__dict__["_touched"] = set()
            self.graphs[key] = self._build(Is, It)
        else:
            self.graphs[key] = self.graphs.pop(key)            # most recently used last
        return self.graphs[key]

    def enqueue(self, Is, It):
        """Queue one pair on the CURRENT stream without waiting for it: input copies (H2D when the images are pinned host
        tensors), one graph replay, one D2H of the packed results into this aligner's own pinned buffer.  Returns a
        ticket for ``fetch``.  The ticket's buffers are reused by the next ``enqueue`` with the same sizes."""
        if isinstance(Is, np.ndarray):
            Is, It = torch.from_numpy(Is), torch.from_numpy(It)
        c = self.prepare(Is, It)
        c["s_in"].copy_(Is, non_blocking=True)
        c["t_in"].copy_(It, non_blocking=True)
        c["graph"].replay()
        self.replayed_kernels += c["n_kernels"]
        if "host" not in c:
            c["host"] = torch.empty(c["packed"].numel(), dtype=c["packed"].dtype).pin_memory()
        c["host"].copy_(c["packed"].reshape(-1), non_blocking=True)
        done = torch.cuda.Event()
        done.record()
        return (c, done)

    def fetch(self, ticket, copy=True):
        """Wait for a ticket and unpack it (same dict as ``align_pair_single``).  ``flow12`` is the graph's static output
        buffer: it is cloned so that results collected over several replays stay valid (``copy=False`` returns the live
        buffer, overwritten by the next replay with these input sizes)."""
        c, done = ticket
        done.synchronize()
        f12 = c["flow12"]
        return self._unpack(c["host"].numpy().copy(), (f12.clone() if copy else f12) if f12 is not None else None, c["size"], c["f8shape"])

    def __call__(self, Is, It, copy=True):
        """Is, It: uint8 (H, W, 3) torch tensors (CUDA, or pinned host for an asynchronous H2D) or numpy arrays."""
        return self.fetch(self.enqueue(Is, It), copy)


def _multi_device(coarseModel, network, Is, It, maxCoarse, maskRegionTh, with_match21, samples=None):
    """The multi-hypothesis loop of evaluation/evalCorr/evaluation.py:211-243 with NO host control at all: every one of the
    ``maxCoarse + 1`` iterations is queued unconditionally; what the reference decides on the host - stop at the first failed
    RANSAC (:215-216), stop at the first hypothesis whose new-region matchability mean is below ``maskRegionTh`` (:226), update
    the mask (:236) - becomes a device-side ``alive`` flag that gates the mask update, and the host drops the hypotheses
    after the first dead one when it unpacks.  Accepted hypotheses are computed from exactly the state the reference's loop
    would have had; dead ones are wasted work (none when every hypothesis is accepted, the common case at maxCoarse = 10).
    One packed result tensor: per hypothesis [alive, status, nbMatch, nbInlier, H(9), flowDown8, matchDown8] - the tensors
    the drivers save (evaluation.py:244-260); the full-resolution maps stay on the device and are not returned."""
    box = {}
    coarseModel.setPair(Is, It)
    Itw, Ith = coarseModel.target_size
    dev = coarseModel.ItTensor.device
    Mask = torch.zeros((Ith, Itw), device=dev)
    alive = torch.ones((), device=dev, dtype=torch.bool)
    recs, featt, f8shape = [], None, None
    for k in range(maxCoarse + 1):
        fgMask = (Mask > 0.5).float()                                    # It_bg = 1 everywhere: (Mask + (1 - It_bg)) > 0.5
        Hd, nb, mask, status, cnt = coarseModel.getCoarse_device(fgMask if k > 0 else None, None if samples is None else samples[k])
        flowCoarse = ops.warp_grid(Hd.view(1, 3, 3), Ith, Itw)
        flow12, match, f8, mboth = PredFlowMask_device(coarseModel.IsTensor, featt, flowCoarse, (Ith, Itw), network, with_match21,
                                                       ItTensor=coarseModel.ItTensor, feat_box=box)
        if featt is None:
            featt = box["featt"]            # computed with the first hypothesis' warped source in one batch
        newreg = (match[0, 0] * (1 - fgMask)).mean()
        ok = (status[0] == 0) & ((newreg > maskRegionTh) if k > 0 else torch.ones((), device=dev, dtype=torch.bool))
        alive = alive & ok
        matchFine = match[0, 0] if k == 0 else match[0, 0] * (1 - fgMask)
        Mask = torch.where(alive, ((Mask + matchFine) >= 1.0).float(), Mask)
        recs.append(torch.cat([alive.float().reshape(1), status.float(), cnt.float(), nb.float(), Hd, f8.reshape(-1), mboth.reshape(-1)]))
        f8shape = tuple(f8.shape)
    return torch.cat(recs), None, (Ith, Itw), f8shape


def _unpack_multi(host, size, f8shape, nhyp):
    host = host.reshape(nhyp, -1)
    if host[0, 1] == 2 or any(host[i, 1] == 2 and host[:i, 0].all() for i in range(nhyp)):
        raise TypeError("'NoneType' object is not subscriptable")          # utils/outil.py:162
    n = 0
    while n < nhyp and host[n, 0] > 0.5:
        n += 1
    if n == 0:
        return dict(H=np.zeros((0,)), flowDown8=np.zeros((0,)), matchDown8=np.zeros((0,)), flow12=[], match=[], nbMatch=[], nbInlier=[])
    n8 = int(np.prod(f8shape))
    return dict(H=host[:n, 4:13].reshape(n, 3, 3).astype(np.float32),
                flowDown8=host[:n, 13:13 + n8].reshape((n,) + tuple(f8shape[1:])),
                matchDown8=host[:n, 13 + n8:13 + 2 * n8].reshape(n, 2, f8shape[2], f8shape[3]),
                flow12=[], match=[], nbMatch=[int(v) for v in host[:n, 2]], nbInlier=[int(v) for v in host[:n, 3]])


def align_pair_multi(coarseModel, network, Is, It, maxCoarse=10, maskRegionTh=0.01, with_match21=True, samples=None):
    """``align_pair_device`` without any host round trip inside the loop (see ``_multi_device``): one pinned D2H at the end.
    Returns H / flowDown8 / matchDown8 / nbMatch / nbInlier of the accepted hypotheses (what the drivers save)."""
    packed, _, size, f8shape = _multi_device(coarseModel, network, Is, It, maxCoarse, maskRegionTh, with_match21, samples)
    return _unpack_multi(_to_host(packed).copy(), size, f8shape, maxCoarse + 1)


class GraphedMultiAligner(GraphedAligner):
    """The whole multi-hypothesis pair (``align_pair_multi``: trunk, matching, ``maxCoarse + 1`` x (RANSAC, warp, fine flow,
    acceptance test, mask update)) as ONE CUDA graph per input size: ~0.6 k kernels per pair at maxCoarse = 10 with no host
    work between them.  BASELINE config 4 (evalCorr / evalYFCC semantics) is measured through it."""

    def __init__(self, coarseModel, network, maxCoarse=10, maskRegionTh=0.01, with_match21=True, warmup=2, max_graphs=4):
        super().__init__(coarseModel, network, with_match21=with_match21, warmup=warmup, max_graphs=max_graphs)
        self.maxCoarse, self.maskRegionTh = maxCoarse, maskRegionTh

    def _device(self, s_in, t_in):
        return _multi_device(self.coarse, self.net, s_in, t_in, self.maxCoarse, self.maskRegionTh, self.m21)

    def _unpack(self, host, flow12, size, f8shape):
        return _unpack_multi(host, size, f8shape, self.maxCoarse + 1)


class ConcurrentAligner:
    """``lanes`` independent GraphedAligners (each with its OWN CoarseAlign state, network activations, graph memory,
    pinned result buffer and stream) replayed side by side: pairs are independent (SURVEY 8e), and a single pair leaves
    SMs idle in its small layers (the /16 grids of the trunk's late layers, the 60 x 80 heads, RANSAC), which the other
    lanes' kernels fill.  ``make_models()`` must return a fresh ``(coarseModel, network)`` per lane (layer programs cache
    their activation buffers per module, so lanes cannot share modules).  Results are per pair and identical to what a
    single GraphedAligner returns for it."""

    def __init__(self, make_models, lanes=2, with_match21=False, make_aligner=None):
        """``make_aligner(coarseModel, network)`` (optional): the per-lane aligner, e.g. a ``GraphedMultiAligner``."""
        mk = make_aligner or (lambda c, n: GraphedAligner(c, n, with_match21=with_match21))
        self.lanes = [mk(*make_models()) for _ in range(lanes)]
        self.streams = [torch.cuda.Stream() for _ in range(lanes)]
        # a replay writes its generator state's seed / offset into device tensors on its own stream: lanes replayed side by
        # side must not share a state, or a lane's RANSAC draws with whichever offset another lane wrote last
        d = torch.cuda.current_device()
        default = torch.cuda.default_generators[d]
        for a in self.lanes:
            a.rng = default.clone_state()
        self.manual_seed(default.initial_seed())

    def manual_seed(self, seed):
        """Seed lane k's generator with ``seed + k`` (distinct sample streams; ``torch.manual_seed`` does not reach them)."""
        for k, a in enumerate(self.lanes):
            a.rng.manual_seed(seed + k)

    @property
    def replayed_kernels(self):
        return sum(a.replayed_kernels for a in self.lanes)

    def prepare(self, Is, It):
        for a in self.lanes:                      # graph capture is serial
            a.prepare(Is, It)
        torch.cuda.synchronize()

    def enqueue(self, pairs):
        """pairs: up to ``lanes`` (Is, It) tuples -> tickets; lane k runs on its own stream, ordered after the work
        already queued on the current stream."""
        assert len(pairs) <= len(self.lanes)
        main = torch.cuda.current_stream()
        tickets = []
        for a, s, (Is, It) in zip(self.lanes, self.streams, pairs):
            a.prepare(Is, It)
            s.wait_stream(main)
            with torch.cuda.stream(s):
                tickets.append(a.enqueue(Is, It))
        for s in self.streams[:len(pairs)]:
            main.wait_stream(s)                   # later work on the current stream (e.g. the next batch) follows all lanes
        return tickets

    def fetch(self, tickets, copy=True):
        return [a.fetch(t, copy) for a, t in zip(self.lanes, tickets)]

    def __call__(self, pairs, copy=True):
        return self.fetch(self.enqueue(pairs), copy)

    def run(self, pairs, copy=True):
        """Any number of pairs through the lanes WITHOUT a barrier between rounds: lane k is refilled as soon as its previous
        pair has been fetched, so the lanes drift apart instead of starting every round in lock-step (their tails and launch
        gaps then overlap each other's work).  Results in the order of ``pairs``.  With ``copy=False`` a result's ``flow12`` is
        valid only until its lane is refilled."""
        main = torch.cuda.current_stream()
        L = len(self.lanes)
        for s in self.streams:
            s.wait_stream(main)
        tickets, owner, out = [None] * L, [None] * L, [None] * len(pairs)
        for i, (Is, It) in enumerate(pairs):
            k = i % L
            if tickets[k] is not None:
                out[owner[k]] = self.lanes[k].fetch(tickets[k], copy)
            with torch.cuda.stream(self.streams[k]):
                tickets[k], owner[k] = self.lanes[k].enqueue(Is, It), i
        for k in range(L):
            if tickets[k] is not None:
                out[owner[k]] = self.lanes[k].fetch(tickets[k], copy)
        for s in self.streams:
            main.wait_stream(s)
        return out


def align_pair(coarseModel, network, Is, It, maxCoarse=0, maskRegionTh=0.01, with_match21=False, It_bg=None):
    """One pair through the evaluation loop (evaluation/evalHpatch/evaluation.py:172-243).
    Returns dict(H (nH,3,3), flowDown8 (nH,2,h8,w8), matchDown8 (nH,2,h8,w8), flow12 [..], match [..])."""
    coarseModel.setPair(Is, It)
    Itw, Ith = coarseModel.target_size
    if It_bg is None:
        It_bg = np.ones((Ith, Itw), dtype=np.float32)
    featt = fine_features(network["netFeatCoarse"], coarseModel.ItTensor)
    grid = torch.empty((1, Ith, Itw, 2), device="meta")                    # size carrier only
    warper = HomographyWarper(Ith, Itw)
    Mask = np.zeros((Ith, Itw), dtype=np.float32)
    Hs, flows8, matches8, flows, matches = [], [], [], [], []
    nbCoarse = 0
    while nbCoarse <= maxCoarse:
        fgMask = ((Mask + (1 - It_bg)) > 0.5).astype(np.float32)
        bestPara = coarseModel.getCoarse(fgMask)
        if bestPara is None:
            break
        bestParaT = torch.from_numpy(bestPara).unsqueeze(0).cuda()
        flowCoarse = warper.warp_grid(bestParaT)
        flowFine, matchFine, f8, m8 = PredFlowMask(coarseModel.IsTensor, featt, flowCoarse, grid, network, with_match21)
        if (matchFine * (1 - fgMask)).mean() > maskRegionTh or nbCoarse == 0:
            Hs.append(bestPara[None])
            flows8.append(f8)
            matches8.append(m8)
            flows.append(flowFine)
            matches.append(matchFine)
            nbCoarse += 1
            matchFine = matchFine if len(matches8) == 0 else matchFine * (1 - fgMask)
            Mask = ((Mask + matchFine) >= 1.0).astype(np.float32)
        else:
            break
    cat = lambda l: np.concatenate(l, axis=0) if l else np.zeros((0,))
    return dict(H=cat(Hs), flowDown8=cat(flows8), matchDown8=cat(matches8), flow12=flows, match=matches)


def align_pair_device(coarseModel, network, Is, It, maxCoarse=0, maskRegionTh=0.01, with_match21=False, It_bg=None, samples=None):
    """The multi-hypothesis loop of evaluation/evalHpatch/evaluation.py:211-243 with the masks kept on the device:
    per hypothesis only the two scalars the host needs to steer the loop (RANSAC status, new-region matchability mean)
    cross the bus instead of the full-resolution matchability map, and the accepted results are fetched once at the
    end.  Same outputs as ``align_pair`` (plus ``nbMatch`` per hypothesis), and under a seed the same RANSAC samples per
    hypothesis.  ``samples``: optional list of injected (nbIter, 4) index tables, one per ``getCoarse`` call."""
    coarseModel.setPair(Is, It)
    Itw, Ith = coarseModel.target_size
    dev = coarseModel.ItTensor.device
    bg = torch.ones((Ith, Itw), device=dev) if It_bg is None else torch.as_tensor(It_bg, dtype=torch.float32, device=dev)
    featt = fine_features(network["netFeatCoarse"], coarseModel.ItTensor)
    Mask = torch.zeros((Ith, Itw), device=dev)
    acc = []
    nbCoarse = ncall = 0
    while nbCoarse <= maxCoarse:
        fgMask = ((Mask + (1 - bg)) > 0.5).float()
        Hd, nb, mask, status, cnt = coarseModel.getCoarse_device(fgMask if nbCoarse > 0 or It_bg is not None else None,
                                                                 None if samples is None else samples[ncall])
        ncall += 1
        # the fine stage is queued before the status is known (no host round trip between RANSAC and the networks); a failed
        # RANSAC leaves H = 0, whose warp grid is NaN: harmless (the results are dropped below) and finite work
        flowCoarse = ops.warp_grid(Hd.view(1, 3, 3), Ith, Itw)
        flow12, match, f8, mboth = PredFlowMask_device(coarseModel.IsTensor, featt, flowCoarse, (Ith, Itw), network, with_match21)
        newreg = (match[0, 0] * (1 - fgMask)).mean()
        ctl = _to_host(torch.cat([status.float(), newreg.reshape(1), cnt.float()])).copy()        # 12 bytes per hypothesis
        st = int(ctl[0])
        if st == 2:
            raise TypeError("'NoneType' object is not subscriptable")     # utils/outil.py:162
        if st != 0:
            break                                                          # bestPara is None (evaluation.py:215-216)
        if float(ctl[1]) > maskRegionTh or nbCoarse == 0:
            acc.append((Hd, f8, mboth, flow12, match, int(ctl[2])))
            matchFine = match[0, 0] if nbCoarse == 0 else match[0, 0] * (1 - fgMask)
            nbCoarse += 1
            Mask = ((Mask + matchFine) >= 1.0).float()
        else:
            break
    if not acc:
        return dict(H=np.zeros((0,)), flowDown8=np.zeros((0,)), matchDown8=np.zeros((0,)), flow12=[], match=[], nbMatch=[])
    packed = torch.cat([torch.cat([a[0], a[1].reshape(-1), a[2].reshape(-1), a[4].reshape(-1)]) for a in acc])
    host = _to_host(packed).copy().reshape(len(acc), -1)
    n8 = acc[0][1].numel()
    f8shape = tuple(acc[0][1].shape)
    return dict(H=host[:, :9].reshape(-1, 3, 3).astype(np.float32),
                flowDown8=host[:, 9:9 + n8].reshape((len(acc),) + f8shape[1:]),
                matchDown8=host[:, 9 + n8:9 + 2 * n8].reshape(len(acc), 2, f8shape[2], f8shape[3]),
                flow12=[a[3] for a in acc], match=[host[i, 9 + 2 * n8:].reshape(Ith, Itw) for i in range(len(acc))],
                nbMatch=[a[5] for a in acc])


def align2images(coarseModel, network, img1, img2, align_corners=False):
    """quick_start/align2images.py:53-97 without the matplotlib / file output: coarse homography from the variant-C
    CoarseAlign, coarse warp, fine flow (no clamp, align2images.py:91-94) and the finely aligned source.
    Note the reference calls ``netCorr(feat_source, feat_target)`` here (align2images.py:89, SURVEY A.3 #9)."""
    with torch.no_grad():
        coarseModel.setSource(img1)
        coarseModel.setTarget(img2)
        w, h = coarseModel.target_size
        bestPrm, inlierMask = coarseModel.getCoarse(np.zeros((h, w)))
        if bestPrm is None:
            return None
        Hd = torch.from_numpy(bestPrm).unsqueeze(0).cuda()
        flowCoarse = HomographyWarper(h, w).warp_grid(Hd)
        img1_coarse = ops.grid_sample(coarseModel.IsTensor, flowCoarse, align_corners)
        feat1 = fine_features(network["netFeatCoarse"], img1_coarse)
        feat2 = fine_features(network["netFeatCoarse"], coarseModel.ItTensor)
        k = network["netCorr"].kernelSize
        if model.fine_engine() == ops.ENGINE_SPLIT:
            corr12, _ = ops.corr_neigh_pair_split(feat1, feat2, k, network["netFlowCoarse"].CORR_LD, want_both=False)
        else:
            corr12 = ops.corr_neigh(feat1, feat2, k, network["netFlowCoarse"].CORR_LD, model.fine_engine())
        flowDown = network["netFlowCoarse"].forward_ragged(corr12)
        flow12, _, _ = ops.compose_fine(flowDown, None, None, flowCoarse, clamp=False, align_corners=align_corners, want_match=False)
        img1_fine = ops.grid_sample(coarseModel.IsTensor, flow12, align_corners)
        return dict(bestPrm=bestPrm, inlierMask=inlierMask, flowCoarse=flowCoarse, img1_coarse=img1_coarse, flowDown=flowDown,
                    flow12=flow12, img1_fine=img1_fine)


# ------------------------------------------------------------------------------------------------------------------
# KITTI: two-level fine flow (evaluation/evalKITTI/evaluation.py) and its recomposition (evalKITTI/getResults.py)
# ------------------------------------------------------------------------------------------------------------------
def PredFlowMask_kitti_device(IsSample, ItSample, flowCoarse, size, network, align_corners=False):
    """evaluation/evalKITTI/evaluation.py:49-81 without the device->host copy: both images' fine features are computed
    here (one ragged batch of two images), the matchability is always ``match12 * grid_sample(match21) * inside``, and
    ``flowCoarse`` (1,Hc,Wc,2) may live on another grid than the ``size`` = (H, W) outputs (the second level, :296-302).
    Returns CUDA tensors (flow12 (1,H,W,2), match (1,1,H,W), flowDown8 (1,2,h8,w8), matchDown8 (1,2,h8,w8))."""
    with torch.no_grad():
        f = fine_features(network["netFeatCoarse"], torch.cat([IsSample, ItSample], dim=0))
        n = f.data.shape[0] // 2
        fs, ft = Ragged(f.data[:n], f.hw[:1]), Ragged(f.data[n:], f.hw[1:])
        k, ld, tc = network["netCorr"].kernelSize, network["netFlowCoarse"].CORR_LD, model.fine_engine()
        if tc == ops.ENGINE_SPLIT:
            corr12, both = ops.corr_neigh_pair_split(ft, fs, k, ld)
        else:
            corr12, _, both = ops.corr_neigh_pair(ft, fs, k, ld, tc)
        flowDown8 = network["netFlowCoarse"].forward_ragged(corr12)
        mboth = network["netMatch"].forward_ragged(both)                    # (2,1,h8,w8): match12, match21
        flow12, match, _ = ops.compose_fine(flowDown8, mboth[0:1], mboth[1:2], flowCoarse, clamp=True, align_corners=align_corners,
                                            size=size)
        return flow12, match, flowDown8, mboth.permute(1, 0, 2, 3).contiguous()


def PredFlowMask_kitti(IsSample, ItSample, flowCoarse, grid, network):
    """Same inputs / outputs as evaluation/evalKITTI/evaluation.py:49-81 (``match`` as a numpy (H, W) array, the /8
    tensors on the device)."""
    flow12, match, f8, m8 = PredFlowMask_kitti_device(IsSample, ItSample, flowCoarse, (grid.size()[1], grid.size()[2]), network)
    return flow12, match[0, 0].cpu().numpy(), f8, m8


def remove_small_cc(matchFine, match_th, cc_th):
    """evaluation/evalKITTI/evaluation.py:85-100 for a numpy (H, W) map, on the device (connected components by union-find)."""
    m = torch.from_numpy(np.ascontiguousarray(matchFine, dtype=np.float32)).cuda()
    return ops.remove_small_cc(m, match_th, cc_th).cpu().numpy()


def align_pair_kitti(coarseModel, network, Is, It, fineSize=650, cc_th=0.01, maskRegionTh=0.005, maxH=None):
    """One pair through evaluation/evalKITTI/evaluation.py:216-344 (no segNet, no file output): per hypothesis the coarse
    homography from ``coarseModel`` (variant A at ``coarseSize``), the first fine level on the half-size target, the
    second level on the ``fineSize`` target sampled on the ORIGINAL image's grid, small connected components of the
    matchability removed on the device, and the reference's mask update on the host.  ``Is`` / ``It``: PIL images.
    ``maxH`` caps the reference's ``while True``.  Returns the four arrays the script saves (H (nH,3,3) 'Homograpy',
    flow_d2 'Finetune_D2', mask 'Finetune_Mask', flow 'Finetune') plus the per-hypothesis full-resolution maps."""
    from . import outil
    strideNet = 8
    to_t = lambda I: coarseModel._to_tensor01(coarseModel._to_device_u8(I))          # transforms.ToTensor()(I)[None].cuda()
    It_resize = outil.resizeImg(It, strideNet, fineSize)
    It_d2 = outil.resizeImg(It, strideNet, fineSize // 2)
    w_org, h_org = It.size
    tensor_s = to_t(Is)
    (w_r, h_r), tensor_resize = It_resize.size, to_t(It_resize)
    (w_d2, h_d2), tensor_d2 = It_d2.size, to_t(It_d2)
    coarseModel.setPair(Is, It)
    It_bg = np.ones((h_org, w_org), dtype=np.float32)
    Mask = np.zeros((h_org, w_org), dtype=np.float32)
    Hs, D2, Msk, Fin, maps = [], [], [], [], []
    nbCoarse = 0
    while maxH is None or nbCoarse < maxH:
        fgMask = ((Mask + (1 - It_bg)) > 0.5).astype(np.float32)
        bestPara = coarseModel.getCoarse(fgMask)
        if bestPara is None:
            break
        with torch.no_grad():
            bp = torch.from_numpy(bestPara).unsqueeze(0).cuda()
            homography_d2 = ops.warp_grid(bp, h_d2, w_d2)
            homography_resize = ops.warp_grid(bp, h_r, w_r)
            IsSample_d2 = ops.grid_sample(tensor_s, homography_d2)
            _, _, flowFine_d2, _ = PredFlowMask_kitti_device(IsSample_d2, tensor_d2, homography_d2, (h_d2, w_d2), network)
            flowCoarse, _, _ = ops.compose_fine(flowFine_d2, None, None, homography_resize, clamp=True, want_match=False)     # :291-294
            IsSample = ops.grid_sample(tensor_s, flowCoarse)
            flowFine_org, match_org, f8, m8 = PredFlowMask_kitti_device(IsSample, tensor_resize, flowCoarse, (h_org, w_org), network)
            ops.remove_small_cc(match_org, 0.99, cc_th)                                                                        # :311
            matchFine = match_org[0, 0].cpu().numpy()
        if ((matchFine > 0.9999) * (1 - fgMask)).mean() > maskRegionTh or nbCoarse == 0:
            Hs.append(bestPara[None])
            D2.append(flowFine_d2.cpu().numpy())
            Msk.append(m8.cpu().numpy())
            Fin.append(f8.cpu().numpy())
            maps.append((flowFine_org, matchFine.copy()))
            nbCoarse += 1
            matchFine = matchFine * (1 - fgMask)              # :324 (len(Finetune_Mask) is never 0 here)
            Mask = ((Mask + matchFine) > 0.9999).astype(np.float32)
        else:
            break
    cat = lambda l: np.concatenate(l, axis=0) if l else np.zeros((0,))
    return dict(H=cat(Hs), flow_d2=cat(D2), mask=cat(Msk), flow=cat(Fin), maps=maps, size=(h_org, w_org))


def getFlow_all_kitti(param, flowd2, flow, match, outH, outW, th=1.0, cc_th=0.01, multiH=True, interpolate=False):
    """evaluation/evalKITTI/getResults.py:95-141 after its np.load calls: param (nH,3,3) 'Homograpy', flowd2 (nH,2,.,.)
    'Finetune_D2', flow (nH,2,.,.) 'Finetune', match (nH,2,.,.) 'Finetune_Mask' -> (flowGlobal (1,outH,outW,2), binary match
    map), both CUDA.  The two levels are composed with the fused kernel, small connected components are removed on the
    device, the first-hypothesis-wins merge is elementwise torch.  ``interpolate``: the EDT hole filling of :87-93
    (``ops.fill_nearest_matched``: exact nearest matched pixel; between equidistant ones the choice may differ from scipy's)."""
    param = torch.as_tensor(param, dtype=torch.float32).cuda()
    flowd2 = torch.as_tensor(flowd2, dtype=torch.float32).cuda()
    flow = torch.as_tensor(flow, dtype=torch.float32).cuda()
    match = torch.as_tensor(match, dtype=torch.float32).cuda()
    homography_org = ops.warp_grid(param, outH, outW)
    fl, ms = [], []
    for i in range(flow.shape[0]):
        fd2, _, _ = ops.compose_fine(flowd2[i:i + 1], None, None, homography_org[i:i + 1], clamp=True, want_match=False)     # :104-107
        f12, m, _ = ops.compose_fine(flow[i:i + 1], match[i:i + 1, 0:1], match[i:i + 1, 1:2], fd2, clamp=True)              # :110-123
        fl.append(f12)
        ms.append(m)
    m = ops.remove_small_cc(torch.cat(ms, dim=0).contiguous(), 0.99, cc_th).permute(0, 2, 3, 1)
    f = torch.clamp(torch.cat(fl, dim=0), min=-1, max=1)
    flowGlobal = f[:1].clone()
    mb = m[:1] >= th
    if multiH:
        for i in range(1, len(m)):
            tmp = (m.narrow(0, i, 1) >= th) * (~mb)
            mb = mb + tmp
            tmp = tmp.expand_as(flowGlobal)
            flowGlobal[tmp] = f.narrow(0, i, 1)[tmp]
    if interpolate:
        flowGlobal = ops.fill_nearest_matched(flowGlobal, mb)
    return flowGlobal, mb


def merge_first_wins(f, m, th, multiH=True):
    """The first-hypothesis-wins merge every getResults script ends with (evaluation/evalCorr/getResults.py:121-134):
    f (nH,H,W,2) clamped flows, m (nH,H,W,1) matchabilities -> (flowGlobal (1,H,W,2), matchGlobal (1,H,W,1), binary map).
    Elementwise torch on the tensors' device."""
    flowGlobal, matchGlobal = f[:1].clone(), m[:1].clone()
    mb = m[:1] >= th
    if multiH:
        for i in range(1, len(m)):
            tmp = (m.narrow(0, i, 1) >= th) * (~mb)
            matchGlobal[tmp] = m.narrow(0, i, 1)[tmp]
            mb = mb + tmp
            tmp = tmp.expand_as(flowGlobal)
            flowGlobal[tmp] = f.narrow(0, i, 1)[tmp]
    return flowGlobal, matchGlobal, mb


def getFlow_corr(flow, param, match, th=0.95, multiH=True):
    """evaluation/evalCorr/getResults.py:78-134 ``getFlow`` (= evalYFCC/getResults.py:150-190 ``_getFlow``) after its np.load
    calls: flow (nH,2,h8,w8), param (nH,3,3), match (nH,2,h8,w8) -> (flowGlobal (1,8h8,8w8,2), matchGlobal (1,8h8,8w8,1)), CUDA:
    x8 upsampling, ``match12 * grid_sample(match21) * inside`` from the fused composition kernel, then ``merge_first_wins``."""
    flow = torch.as_tensor(flow, dtype=torch.float32).cuda()
    param = torch.as_tensor(param, dtype=torch.float32).cuda()
    match = torch.as_tensor(match, dtype=torch.float32).cuda()
    H, W = int(flow.shape[2]) * 8, int(flow.shape[3]) * 8
    coarse = ops.warp_grid(param, H, W)
    fl, ms = [], []
    for i in range(flow.shape[0]):
        f12, m, _ = ops.compose_fine(flow[i:i + 1], match[i:i + 1, 0:1], match[i:i + 1, 1:2], coarse[i:i + 1], clamp=True)
        fl.append(f12)
        ms.append(m)
    f = torch.clamp(torch.cat(fl, dim=0), min=-1, max=1)
    m = torch.cat(ms, dim=0).permute(0, 2, 3, 1)
    flowGlobal, matchGlobal, _ = merge_first_wins(f, m, th, multiH)
    return flowGlobal, matchGlobal


def getFlow_all(flow, param, match, outH, outW, th=0.95, multiH=True, with_match21=False):
    """evaluation/evalHpatch/getResults.py:16-63 on device tensors: flow (nH,2,h8,w8), param (nH,3,3),
    match (nH,2,h8,w8) -> flowGlobal (1,outH,outW,2).  The reference runs this on CPU tensors; the
    composition here is the fused kernel, the first-hypothesis-wins merge is elementwise torch."""
    flow = torch.as_tensor(flow, dtype=torch.float32).cuda()
    param = torch.as_tensor(param, dtype=torch.float32).cuda()
    match = torch.as_tensor(match, dtype=torch.float32).cuda()
    coarse = ops.warp_grid(param, outH, outW)
    fl, ms = [], []
    for i in range(flow.shape[0]):
        f12, m, _ = ops.compose_fine(flow[i:i + 1], match[i:i + 1, 0:1], match[i:i + 1, 1:2] if with_match21 else None,
                                     coarse[i:i + 1], clamp=True)
        fl.append(f12)
        ms.append(m)
    f = torch.clamp(torch.cat(fl, dim=0), min=-1, max=1)
    m = torch.cat(ms, dim=0).permute(0, 2, 3, 1)
    flowGlobal = f[:1].clone()
    if multiH:
        mb = m[:1] >= th
        for i in range(1, len(m)):
            tmp = (m.narrow(0, i, 1) >= th) * (~mb)
            mb = mb + tmp
            tmp = tmp.expand_as(flowGlobal)
            flowGlobal[tmp] = f.narrow(0, i, 1)[tmp]
    return flowGlobal
