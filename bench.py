#!/usr/bin/env python
"""bench.py - image-pairs/sec on synthetic pairs (BASELINE.json configs 2-5; default config 2 = 480x640).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 2|3|4|5]
                    [--engine f16x3|fp32|f16|tf32] [--lanes L] [--pairs-per-step P] [--dump-outputs DIR]

One "step" = P independent pairs per GPU (default 32, `config.pairs_per_gpu_per_step`), each through the whole hot path
(variant-A CoarseAlign.setPair -> getCoarse -> warp_grid -> PredFlowMask).  Config 2: nbScale 7, scaleR 2, nbIter 1000, one
hypothesis; L pairs at a time run as L CUDA graphs on L streams (pipeline.ConcurrentAligner).  Config 3 adds the
getFlow_all recomposition at minSize 240 (evalHpatch/getResults.py), config 4 the multi-hypothesis loop with maxCoarse = 10
and the evalCorr matchability (device-resident masks), config 5 the KITTI two-level flow on 376x1241 pairs capped at 5
hypotheses.  Prints ONE JSON line (rank 0).  `value` = pairs/s with the uint8 images already in HBM; `e2e` = the same
through the public API from pinned HOST images (H2D of the inputs + D2H of the results inside the timed region).  The default
engine `f16x3` is the fp32-grade tensor-core engine (fp16 hi / lo split operands, 3 MMAs per MAC); `parity` reports how far
that engine is from the CPU oracle on pair 0 of the workload (computed outside the timed region from the file the
cpu_baseline child wrote).  `--impl reference` times the CPU oracle (oracle/pair_oracle.py: the reference's own PyTorch-CPU
algorithm, all host threads) on the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    2: "config2: synthetic 480x640 pairs, variant-A CoarseAlign nbScale=7 scaleR=2 nbIter=1000 tol=0.05, 1 hypothesis, PredFlowMask",
    3: "config3: HPatches-shaped synthetic 480x640 pairs, config-2 path + getFlow_all recomposition at minSize 240 (evalHpatch/getResults.py:171,191-194)",
    4: "config4: MegaDepth/YFCC-shaped synthetic 480x640 pairs, multi-hypothesis loop maxCoarse=10, match12*grid_sample(match21) (evalCorr/evaluation.py:211-243)",
    5: "config5: KITTI-shaped synthetic 376x1241 pairs, coarseSize 800 nbScale=3 scaleR=1.2, two-level fine flow, up to 5 hypotheses (evalKITTI/evaluation.py:270-336)",
}
WORKLOAD = WORKLOADS[2]
METRIC = "image-pairs/sec at 480x640, nbIter=1k RANSAC"
NA, NB, CFEAT = 13065, 1200, 1024
PARITY_RAW_SEED = 1000            # the raw sample table both arms reduce modulo their match count for the parity pair
DTYPES = {"fp32": "f32", "tf32": "tf32",
          "f16x3": "f32-grade: fp16 hi/lo split operands and activations (22 significand bits), 3 tcgen05 MMAs per MAC, fp32 accumulate; fp16-split correlation; fp32/fp64 RANSAC",
          "f16": "f16 (reduced precision fast mode: conv operands and activations fp16, fp32 accumulate; TF32 output convs of the heads; fp16-split correlation; fp32/fp64 RANSAC)",
          "f16-trunk": "f16 trunk + tf32 fine-flow nets (reduced precision)"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"), src="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, src="fallback")


class ClockSampler:
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md's clocks line).  Sampled in-process through
    NVML - the library nvidia-smi itself reads - every 100 ms: spawning `nvidia-smi -lms 100` next to the bench perturbed the
    first timed region (every other 32-pair step took 143 instead of 123 ms while nvidia-smi was starting up on the 8-GPU
    box); the subprocess form is kept as the fallback when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.nvml, self.handle, self.stop_flag, self.thread, self.max_mhz = None, None, False, None, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:                                  # CUDA_VISIBLE_DEVICES may renumber the GPUs: resolve through the UUID
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid if not uuid.startswith("GPU-") else uuid).encode())
        except Exception:  # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, h

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.max_mhz = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:  # noqa: BLE001
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _poll(self):
        n = self.nvml
        bits = [n.nvmlClocksThrottleReasonHwSlowdown, n.nvmlClocksThrottleReasonHwThermalSlowdown,
                n.nvmlClocksThrottleReasonSwThermalSlowdown, n.nvmlClocksThrottleReasonSwPowerCap]
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append([mhz] + [bool(r & b) for b in bits])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.1)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            sm = [r[0] for r in self.rows]
            reasons = [nm for j, nm in enumerate(self.NAMES) if any(r[1 + j] for r in self.rows)]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm),
                    "source": "NVML in-process, 100 ms"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = [n for j, n in enumerate(self.NAMES) if any(len(r) >= 7 and r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


def ncu_facts(precision, v2):
    """What the committed `ncu --set full` capture of the correlation kernel says (profiles/*.json, one launch at config 2):
    DRAM bytes read + written, duration and tensor-pipe activity of the dominant launch.  {} when there is no capture."""
    try:
        pf = {1: "r1_corr_ncu.json", 2: "r2_ncu_full_kernels.json" if v2 else "r1_corr_f16_ncu.json"}[int(precision)]
        prof = json.load(open(os.path.join(ROOT, "profiles", pf)))
        l = [l for l in prof["launches"] if "tc_kernel" in l["kernel"] or "tc_corr_pipe" in l["kernel"]][0]
        dur = l["gpu__time_duration.sum"]
        us = float(dur["value"]) * {"ns": 1e-3, "us": 1.0, "ms": 1e3, "nsecond": 1e-3, "usecond": 1.0, "msecond": 1e3}.get(dur["unit"], 1.0)
        return {"file": "profiles/" + pf, "traffic": l["dram_traffic_bytes"], "kernel_us": us,
                "tensor_pct": float(l["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"]["value"])}
    except Exception:  # noqa: BLE001
        return {}


def roofline_record(prec, v2, corr_ms, ransac_ms, n_matches, pk, presplit=False):
    """The `roofline` object of the JSON line for the kernel BASELINE.json names (correlation + mutual NN, plus RANSAC as
    us/call): algorithmic flops / bytes of config 2 (SURVEY 8d) over the call's measured time, against the measured peaks.
    Pure arithmetic (tests/test_abi_and_host.py runs it without a GPU)."""
    flops = 2.0 * NA * NB * CFEAT
    abytes = 4.0 * CFEAT * (NA + NB) + 16.0 * n_matches
    tf = flops / (corr_ms * 1e-3) / 1e12
    tensor_peak = pk["bf16_tflops"]
    ncu = ncu_facts(prec, v2)              # DRAM traffic etc. of the dominant launch, from the committed ncu --set full capture
    kname = {0: "corr_argmax_kernel (fp32 SIMT)", 1: "tc_kernel<128,MODE_CORR> (3xTF32 tcgen05)",
             2: ("tc_corr_pipe_kernel (persistent, two TMEM accumulator pairs; " if v2 else "tc_kernel<128,MODE_CORR,f16> (")
                + "fp16 split tcgen05: hi*hi + (hi*lo + lo*hi) * 2^-11)"}[prec]
    # tensor work actually issued per algorithmic MAC: 3 MMAs either way; kind::tf32 runs at half the bf16/f16 rate
    rate = {0: None, 1: tensor_peak / 2, 2: tensor_peak}[prec]
    call = ("rf_corr_mutual_nn_presplit = key memset + %s + column-driven compaction (operand planes written by rf_l2norm_split_nhwc)" if presplit
            else "rf_corr_mutual_nn = %s + split/compaction helpers")
    return {"kernel": call % kname,
            "bound": "tensor", "achieved": tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": tf / tensor_peak, "traffic": ncu.get("traffic"),
            "peak_source": pk["src"] + " bf16 dense GEMM (burst); fp32-grade scores need 3 tensor MMAs per algorithmic MAC (split operands), "
                           "so the executed tensor fraction is 3 x frac for the fp16 split (6 x for 3xTF32, whose MMAs run at half rate)",
            "executed_tensor_frac": (3 * tf) / rate if rate else None,
            "ms_per_launch": corr_ms, "algorithmic_gflop": flops / 1e9, "algorithmic_mb": abytes / 1e6,
            "hbm_gbs_achieved": abytes / (corr_ms * 1e-3) / 1e9, "hbm_frac": abytes / (corr_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
            # the dominant kernel alone, from the committed capture (the live number above times the whole 3-launch call)
            "ncu_capture": ncu.get("file"), "kernel_us_ncu": ncu.get("kernel_us"), "tensor_pipe_active_pct_ncu": ncu.get("tensor_pct"),
            "executed_tensor_frac_kernel_ncu": (3 * flops / (ncu["kernel_us"] * 1e-6) / 1e12 / rate) if (rate and ncu.get("kernel_us")) else None,
            "ransac_us_per_call": 1e3 * ransac_ms, "ransac_matches": n_matches,
            "corr_plus_ransac_gbs": (abytes + 61e3) / ((corr_ms + ransac_ms) * 1e-3) / 1e9}


def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except Exception:  # noqa: BLE001
            pass
    return max(1, n)


def pair_size(config):
    return (376, 1241) if config == 5 else (480, 640)


def make_pairs(n, config=2):
    import synthdata as synth                        # workload generator (repo root); nothing under oracle/ on the B200 arm
    h, w = pair_size(config)
    return [synth.make_pair(i, h, w)[:2] for i in range(n)]


def raw_sample_table(nbIter=1000):
    import synthdata as synth
    return synth.draw_samples(PARITY_RAW_SEED, 2 ** 31 - 1, nbIter)


def states():
    import synthdata as synth
    return (synth.resnet50_conv4_state(0), synth.feature_extractor_state(0), synth.net_flow_coarse_state(1),
            synth.net_matchability_state(2))


DUMP_SAMPLE = 1 << 16          # elements kept of a larger output array (a seeded sample): a step's dump stays far below 64 MB
DUMP_MAX_BYTES = 64 << 20


def _dump_leaves(name, v):
    """(name, value) for every array-like leaf of a result: dict keys and list positions join the name with '_'."""
    if isinstance(v, dict):
        for k, x in v.items():
            yield from _dump_leaves("%s_%s" % (name, k), x)
    elif isinstance(v, (list, tuple)) and not all(isinstance(x, (int, float, np.number)) for x in v):
        for j, x in enumerate(v):
            yield from _dump_leaves("%s_%d" % (name, j), x)
    else:
        yield name, v


def dump_outputs(outs, d):
    """Write the per-pair results of one step as d/pair<r>_<key>.npy: integers and float64 data as float64, the rest as float32;
    an array of more than DUMP_SAMPLE elements as the same seeded sample of its flat elements in every run.  A CUDA tensor is
    written only for the last result that holds its storage: the graphed aligners return flow12 as the graph's output buffer
    (copy=False), which the lane's next pair overwrites."""
    import torch
    leaves = [leaf for r, out in enumerate(outs) for leaf in _dump_leaves("pair%02d" % r, out)]
    owner = {v.data_ptr(): name for name, v in leaves if isinstance(v, torch.Tensor) and v.is_cuda}
    arrays = {}
    for name, v in leaves:
        if isinstance(v, torch.Tensor):
            if v.is_cuda and owner[v.data_ptr()] != name:
                continue
            v = v.detach().cpu().numpy()
        a = np.asarray(v)
        a = a.astype(np.float64 if a.dtype.kind in "iu" or a.dtype == np.float64 else np.float32)
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.RandomState(a.size).choice(a.size, DUMP_SAMPLE, replace=False))]
        arrays[name] = a
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %.1f MB (limit %d MB); use fewer --pairs-per-step" % (total / 1e6, DUMP_MAX_BYTES >> 20))
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


# ----------------------------------------------------------------------------- reference arm (CPU oracle)
def run_reference(args, rank, world):
    """The reference's own algorithm on the host cores (oracle/pair_oracle.py, torch-CPU fp32).  With --dump-parity FILE it
    also runs pair 0 of the workload once more with the shared raw sample table and writes everything a parity check needs
    (index lists, score matrix, matches, H, inlier mask, flows) to FILE: the B200 arm reads that FILE, never the oracle."""
    if rank != 0:
        return
    import PIL.Image as Image
    import torch
    from oracle import pair_oracle as PO
    from oracle import warp_oracle as WO
    cores = int(os.environ.get("RF_CPU_THREADS", "0")) or min(usable_cores(), 64)
    torch.set_num_threads(cores)
    rsd, fe, nf, nm = states()
    net = {"netFeatCoarse": fe, "netFlowCoarse": nf, "netMatch": nm}
    cfg = args.config
    pairs = make_pairs(2, cfg)
    if cfg == 5:
        oc = PO.CoarseAlignOracle(rsd, nbScale=3, nbIter=1000, tolerance=0.05, minSize=800, scaleR=1.2, variant="A", seed=1000)
    else:
        oc = PO.CoarseAlignOracle(rsd, nbScale=7, nbIter=1000, tolerance=0.05, minSize=480, scaleR=2, variant="A", seed=1000)

    def step(i):
        s, t = pairs[i % len(pairs)]
        Is, It = Image.fromarray(s), Image.fromarray(t)
        if cfg == 5:
            return PO.align_pair_kitti(oc, net, Is, It, maxH=5)
        if cfg == 4:
            return PO.align_pair(oc, net, Is, It, maxCoarse=10, with_match21=True)
        out = PO.align_pair(oc, net, Is, It, maxCoarse=0)
        if cfg == 3:
            out["flowGlobal"] = WO.get_flow_all(out["flowDown8"], out["H"], out["matchDown8"], 240, 240, th=0.95, multiH=True)[0]
        return out
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    dt = time.perf_counter() - t0
    v = args.steps / dt
    if args.dump_parity and cfg in (2, 3):
        from oracle import outil_oracle as OO
        oc.raw_samples = raw_sample_table()
        dump = {}
        for pi in (0, 1):                                         # pairs 0 and 1 of the workload
            s0, t0_ = pairs[pi]
            ref = PO.align_pair(oc, net, Image.fromarray(s0), Image.fromarray(t0_), maxCoarse=0)
            featt = oc.featt.contiguous().view(oc.featt.shape[1], -1).numpy()
            score = oc.featsMultiScale.numpy().T @ featt
            _, nbInl, isInl, _ = OO.RANSAC_from_samples(oc.match1, oc.match2, oc.last_samples, 0.05)
            for key, arr in dict(index1=oc.index1, index2=oc.index2, score=score, match1=oc.match1, match2=oc.match2, samples=oc.last_samples,
                             H=ref["H"], nbInlier=np.int64(nbInl), isInlier=np.asarray(isInl, dtype=bool), flowDown8=ref["flowDown8"],
                                 matchDown8=ref["matchDown8"], flow12=ref["flow12"][0].numpy(), match=ref["match"][0]).items():
                dump["%s_%d" % (key, pi)] = arr
        np.savez(args.dump_parity, **dump)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOADS[cfg]},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": "%d whole pairs through oracle/pair_oracle.py (torch-CPU fp32, %d threads)" % (args.steps, torch.get_num_threads())},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def parity_report(rf, torch, ref, coarse, net, pair, engine, label="pair 0"):
    """How far the timed engine is from the CPU oracle on one pair of the workload (outside the timed region).  `ref` = the
    arrays the cpu_baseline child wrote for that pair.  (a) match set and tie proofs, (b) the oracle's matches + samples through the RANSAC kernel,
    (c) the oracle's H through the fine stage, (d) end to end with the shared sample table."""
    import PIL.Image as Image
    raw = raw_sample_table()
    s, t = pair
    out = rf.pipeline.align_pair_single(coarse, net, s, t, samples=raw)
    n = int(coarse._count.item())
    got = set(zip(coarse._idx1[:n].cpu().tolist(), coarse._idx2[:n].cpu().tolist()))
    exp = set(zip(ref["index1"].tolist(), ref["index2"].tolist()))
    score = ref["score"]
    dev = float((coarse._feats_rows.double() @ coarse._featt_rows.double().t() - torch.from_numpy(score).cuda().double()).abs().max())
    rowmax, colmax = score.max(1), score.max(0)
    s2r, s2c = np.partition(score, -2, axis=1)[:, -2], np.partition(score, -2, axis=0)[-2]
    margins = [float(min(rowmax[i] - s2r[i], colmax[j] - s2c[j])) if (i, j) in exp else float(max(rowmax[i] - score[i, j], colmax[j] - score[i, j]))
               for (i, j) in sorted(got ^ exp)]
    # (b) the oracle's match list and sample table through the RANSAC kernel
    m1, m2 = torch.from_numpy(ref["match1"]).cuda(), torch.from_numpy(ref["match2"]).cuda()
    Hd, nb, mask, status = rf.ops.ransac_homography(m1, m2, torch.from_numpy(ref["samples"]).cuda(), 0.05)
    # (c) the oracle's H through warp_grid + PredFlowMask
    Itw, Ith = coarse.target_size
    featt = rf.pipeline.fine_features(net["netFeatCoarse"], coarse.ItTensor)
    fc = rf.ops.warp_grid(torch.from_numpy(ref["H"]).cuda(), Ith, Itw)
    f12, match, f8, mb = rf.pipeline.PredFlowMask_device(coarse.IsTensor, featt, fc, (Ith, Itw), net)
    same = len(got ^ exp) == 0
    rec = {
        "engine": engine, "pair": label + " of the workload, shared raw sample table % match count, oracle = oracle/pair_oracle.py (CPU fp32)",
        "matches_oracle": len(exp), "matches_b200": len(got), "match_symdiff": len(got ^ exp),
        "max_abs_score_dev": dev, "symdiff_worst_margin": max(margins, default=0.0),
        "symdiff_all_proven_ties": bool(all(m <= 2 * dev + 3e-6 for m in margins)),      # 3e-6: the fp16-split correlation kernel's own arithmetic
        "stage_ransac_on_oracle_matches": {"status": int(status.item()), "nb_inlier_equal": bool(int(nb.item()) == int(ref["nbInlier"])),
                                           "inlier_mask_equal": bool(np.array_equal(mask.cpu().numpy().astype(bool), ref["isInlier"])),
                                           "max_abs_H": float(np.abs(Hd.cpu().numpy().reshape(3, 3) - ref["H"][0]).max())},
        "stage_fine_on_oracle_H": {"max_abs_flowDown8": float(np.abs(f8.cpu().numpy() - ref["flowDown8"]).max()),
                                   "max_abs_matchDown8": float(np.abs(mb.cpu().numpy().reshape(ref["matchDown8"].shape) - ref["matchDown8"]).max()),
                                   "max_abs_flow12": float(np.abs(f12.cpu().numpy() - ref["flow12"]).max())},
        "end_to_end": {"max_abs_H": float(np.abs(out["H"] - ref["H"]).max()) if len(out["H"]) else None,
                       "max_abs_flowDown8": float(np.abs(out["flowDown8"] - ref["flowDown8"]).max()) if len(out["H"]) else None,
                       "max_abs_flow12": float(np.abs(out["flow12"][0].cpu().numpy() - ref["flow12"]).max()) if len(out["H"]) else None,
                       "note": "meaningful as parity only when match_symdiff == 0: the samples index the match list, so one tie re-labels every hypothesis (the reference's own CPU and GPU runs differ the same way)" if not same else "match lists identical"},
    }
    fine = rec["stage_fine_on_oracle_H"]
    rec["within_north_star"] = bool(rec["symdiff_all_proven_ties"] and rec["stage_ransac_on_oracle_matches"]["inlier_mask_equal"]
                                    and max(fine.values()) < 1e-3 and (not same or rec["end_to_end"]["max_abs_flow12"] < 1e-3))
    return rec


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args, rank, world, local):
    import PIL.Image as Image
    import torch
    import torch.distributed as dist
    import ransac_flow_b200 as rf
    from ransac_flow_b200 import shard
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = args.config
    rf.model.set_engine(args.engine)
    rf.outil.corr_precision = {"fp32": 0, "tf32": 1}.get(args.engine, 2)      # exact fp32 / 3xTF32 / fp16 split
    rsd, fe_sd, nf_sd, nm_sd = states()
    H_img, W_img = pair_size(cfg)

    def make_models():
        """A fresh (CoarseAlign, networks) set: same weights, own activation buffers / pair state."""
        net = {"netFeatCoarse": rf.model.FeatureExtractor(), "netCorr": rf.model.CorrNeigh(7),
               "netFlowCoarse": rf.model.NetFlowCoarse(7), "netMatch": rf.model.NetMatchability(7)}
        net["netFeatCoarse"].load_state_dict(fe_sd)
        net["netFlowCoarse"].load_state_dict(nf_sd)
        net["netMatch"].load_state_dict(nm_sd)
        for m in net.values():
            m.cuda()
            m.eval()
        if cfg == 5:
            c = rf.CoarseAlignA(3, 1000, 0.05, "Homography", 800, 2, False, 1.2, True, False, resnet_state_dict=rsd, verbose=False)
        else:
            c = rf.CoarseAlignA(7, 1000, 0.05, "Homography", 480, 2, False, 2, True, False, resnet_state_dict=rsd, verbose=False)
        c.device_preproc = True
        return c, net
    coarse, net = make_models()
    graphed = args.graph and cfg in (2, 3, 4)          # config 5 steers its hypothesis loop from the host (12 bytes per hypothesis)
    lanes = max(1, args.lanes) if graphed else 1
    P = max(lanes, (args.pairs_per_step // lanes) * lanes) if graphed else max(1, args.pairs_per_step)
    pairs = make_pairs(4, cfg)
    host = [(torch.from_numpy(s).pin_memory(), torch.from_numpy(t).pin_memory()) for s, t in pairs]
    resident = [(s.to(dev), t.to(dev)) for s, t in host]
    pil = [(Image.fromarray(s), Image.fromarray(t)) for s, t in pairs]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    if cfg == 4:      # evalCorr / evalYFCC semantics: maxCoarse = 10, match12 * grid_sample(match21); the whole loop is one CUDA graph
        mk = lambda c, n: rf.pipeline.GraphedMultiAligner(c, n, maxCoarse=10, maskRegionTh=0.01, with_match21=True)
    else:
        mk = lambda c, n: rf.pipeline.GraphedAligner(c, n)
    aligner = mk(coarse, net) if (graphed and lanes == 1) else None
    multi = rf.pipeline.ConcurrentAligner(make_models, lanes, make_aligner=mk) if lanes > 1 else None
    if multi is not None:
        multi.prepare(*resident[0])

    def replayed():
        return (aligner.replayed_kernels if aligner is not None else 0) + (multi.replayed_kernels if multi is not None else 0)

    def one_pair(i, from_host):
        """Configs 4 / 5 (and --no-graph): one pair through the eager API."""
        s, t = (host if from_host else resident)[i % len(resident)]
        if cfg == 5:
            Is, It = pil[i % len(pil)]               # align_pair_kitti takes PIL images (resizeImg on the host, like the script)
            torch.manual_seed(1000)                  # evalKITTI/evaluation.py:182
            return rf.pipeline.align_pair_kitti(coarse, net, Is, It, maxH=5)
        if from_host:
            s, t = s.to(dev, non_blocking=True), t.to(dev, non_blocking=True)
        torch.manual_seed(1000)
        if cfg == 4:
            return rf.pipeline.align_pair_device(coarse, net, s, t, maxCoarse=10, with_match21=True)
        return rf.pipeline.align_pair_single(coarse, net, s, t)

    def step(i, from_host):
        """One step = P pairs: returns the list of per-pair results."""
        src = host if from_host else resident                                       # pinned host (H2D inside) or HBM-resident
        outs = []
        if multi is not None:                                                       # lanes graphs side by side, each lane refilled as it completes
            outs = multi.run([src[(i * P + r) % len(src)] for r in range(P)], copy=False)
        elif aligner is not None:
            for r in range(P):
                outs.append(aligner(*src[(i * P + r) % len(src)], copy=False))      # one CUDA-graph launch + one pinned D2H
        else:
            for r in range(P):
                outs.append(one_pair(i * P + r, from_host))
        if cfg == 3:                                                                # evalHpatch/getResults.py: recomposition at minSize 240
            for o in outs:
                if len(o["H"]):
                    o["flowGlobal"] = rf.pipeline.getFlow_all(o["flowDown8"], o["H"], o["matchDown8"], 240, 240, th=0.95, multiH=True)
        flush.zero_()                                                               # L2 flush between steps
        return outs

    def timed(from_host, K, W):
        for i in range(W):
            step(i, from_host)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        # the graphs draw their RANSAC samples from CUDA generator states whose offsets the time-bounded pre-warm leaves wherever
        # it stopped: reseeding makes the timed steps see the same samples in every run
        torch.cuda.manual_seed(1000)
        if multi is not None:
            multi.manual_seed(1000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = rf._lib.launch_count() + replayed()
        e0.record()
        recs = []
        tstamps = [time.perf_counter()]
        for i in range(K):
            outs = step(i, from_host)
            tstamps.append(time.perf_counter())
            for k, out in enumerate(outs):
                recs.append(shard.pack_record(rank + world * (i * P + k), out["H"][0] if len(out["H"]) else None,
                                              status=0 if len(out["H"]) else 1))
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()                                                          # ranks drift apart (each GPU sits at its own power-capped
        g0 = time.perf_counter()                                                    # clock): the gather's own time, not the wait for the slowest
        allr = shard.gather_records(recs, K * P * world, world, dev)                # the one collective: per-pair records
        e1.record()
        torch.cuda.synchronize()
        gather_ms = 1e3 * (time.perf_counter() - g0)
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if os.environ.get("RF_BENCH_STEP_TIMES") and rank == 0:
            print("step ms (host clock, from_host=%s): %s; gather %.1f" % (from_host, " ".join("%.1f" % (1e3 * (b - a)) for a, b in zip(tstamps, tstamps[1:])), gather_ms), file=sys.stderr)
        launches = rf._lib.launch_count() + replayed() - l0
        if world > 1:
            tmax = torch.tensor([ms], device=dev)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ms = float(tmax.item())
        return ms, launches, outs, allr, gather_ms

    # set-up, untimed and before the W warm-up steps of the contract: a couple of seconds of the real load (clocks, power state,
    # allocator).  Observation (profiles/README.md): with device-resident inputs every other 32-pair step takes ~139 instead of
    # ~123 ms (per-step host timestamps), whatever the pre-warm (2 s, 6 s, a discarded dry-run region) and however the clocks are
    # sampled, while the pinned-host-input region of the same process is flat: the resident path copies each pair device-to-device
    # into the graph's static input buffers on the lane's stream, the host path uses the copy engines.  `value` is therefore ~4 %
    # conservative against `e2e`.
    # (the clock sampler starts first: nvidia-smi's own start-up perturbs the GPU for about a second)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if graphed:
        t_pre = time.perf_counter()
        i_pre = 0
        while time.perf_counter() - t_pre < float(os.environ.get("RF_PREWARM_SECONDS", "2.0")):
            step(i_pre, False)
            i_pre += 1
        torch.cuda.synchronize()
    ms_dev, launches, outs, _, _ = timed(False, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(outs, args.dump_outputs)                     # before the next region's replays overwrite the graphs' buffers
    del outs                                                      # the e2e region allocates its results in the memory these held
    ms_e2e, _, outs, allr, gather_ms = timed(True, args.steps, max(1, args.warmup // 2))
    out = outs[-1]
    clocks = sampler.stop() if rank == 0 else None
    assert allr.shape[0] == args.steps * P * world
    if os.environ.get("RF_BENCH_REPEAT_RESIDENT") and rank == 0 and world == 1:      # experiment: order dependence of the two timed regions
        ms2 = timed(False, args.steps, 2)[0]
        ms3 = timed(True, args.steps, 2)[0]
        print("repeat: resident %.1f pairs/s (first %.1f), host %.1f pairs/s (first %.1f)" % (
            P * args.steps / (ms2 * 1e-3), P * args.steps / (ms_dev * 1e-3), P * args.steps / (ms3 * 1e-3), P * args.steps / (ms_e2e * 1e-3)), file=sys.stderr)
    if rank != 0:
        return                                       # the per-kernel sections below are rank 0's (no collective inside)
    nH_mean = float(np.mean([len(o["H"]) for o in [out]]))

    stages = roofline = None
    if cfg in (2, 3):
        # ---- where a pair's GPU time goes: the device path stage by stage (eager launches, CUDA events, median of 7 pairs) ----
        def stage_breakdown():
            names = ["pyramid+preproc+resnet50_conv4(8 imgs)+l2norm", "corr+mutual_nn", "fine_features(target)", "build_matches+ransac",
                     "warp_grid+PredFlowMask"]
            acc = []
            reps, skip = 7, 3                     # the first eager passes of these model objects build TMA maps / layer programs
            for rep in range(reps + skip):
                s_, t_ = resident[rep % len(resident)]
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
                saved, saved_p = rf.ops.corr_mutual_nn, rf.ops.corr_mutual_nn_presplit
                marks = {}

                def hook(fn):                                            # setPair ends with the correlation: split it out
                    def wrapped(*a, **k):
                        marks["pre"] = torch.cuda.Event(enable_timing=True)
                        marks["pre"].record()
                        return fn(*a, **k)
                    return wrapped
                rf.ops.corr_mutual_nn, rf.ops.corr_mutual_nn_presplit = hook(saved), hook(saved_p)
                try:
                    evs[0].record()
                    coarse.setPair(s_, t_)
                finally:
                    rf.ops.corr_mutual_nn, rf.ops.corr_mutual_nn_presplit = saved, saved_p
                evs[2].record()
                Itw, Ith = coarse.target_size
                featt = rf.pipeline.fine_features(net["netFeatCoarse"], coarse.ItTensor)
                evs[3].record()
                Hd, nb, mask, status, cnt = coarse.getCoarse_device(None)
                evs[4].record()
                fc = rf.ops.warp_grid(Hd.view(1, 3, 3), Ith, Itw)
                rf.pipeline.PredFlowMask_device(coarse.IsTensor, featt, fc, (Ith, Itw), net)
                evs[5].record()
                torch.cuda.synchronize()
                if rep < skip:
                    continue
                acc.append([evs[0].elapsed_time(marks["pre"]), marks["pre"].elapsed_time(evs[2]), evs[2].elapsed_time(evs[3]),
                            evs[3].elapsed_time(evs[4]), evs[4].elapsed_time(evs[5])])
            med = np.median(np.array(acc), axis=0)    # median: an eager pass now and then pays a cudaMalloc / host hiccup
            return {n: round(float(v), 4) for n, v in zip(names, med)}
        stages = stage_breakdown()

        # ---- roofline of the kernel BASELINE names (corr + mutual-NN), timed alone with CUDA events ----
        presplit = "_src_planes" in coarse.__dict__      # engine f16x3: the normalisation wrote the correlation's hi / lo planes
        if presplit:
            sp, tp = coarse._src_planes, coarse._tgt_planes
            corr_call = lambda: rf.ops.corr_mutual_nn_presplit(sp[0], sp[1], tp[0], tp[1])
        else:
            fa, ft = coarse._feats_rows, coarse._featt_rows
            corr_call = lambda: rf.ops.corr_mutual_nn(fa, ft, rf.outil.corr_precision)
        st = torch.cuda.current_stream()
        reps = 20
        for _ in range(3):
            corr_call()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ev:
            flush.zero_()
            a.record(st)
            corr_call()
            b.record(st)
        torch.cuda.synchronize()
        corr_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
        # RANSAC alone (latency-bound: reported as us/call)
        nm = int(coarse._match_count.item())             # matches of the pair `coarse` holds (set by stage_breakdown)
        m1, m2 = coarse.match1[:nm].contiguous(), coarse.match2[:nm].contiguous()
        smp = torch.randint(len(m1), (1000, 4), device=dev)
        for _ in range(3):
            rf.ops.ransac_homography(m1, m2, smp, 0.05)
        for a, b in ev:
            a.record(st)
            rf.ops.ransac_homography(m1, m2, smp, 0.05)
            b.record(st)
        torch.cuda.synchronize()
        ransac_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
        prec = rf.outil.corr_precision
        v2 = prec == 2 and rf._lib.lib.rf_corr_mutual_nn_launches(2) == 3
        roofline = roofline_record(prec, v2, corr_ms, ransac_ms, int(len(m1)), peaks(), presplit)

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same workload on the host cores, run as
    # `bench.py --impl reference` in a child process so that it can be cut off.  The child also writes the oracle's
    # outputs for pair 0 to a file; `parity` compares the timed engine with that file (outside every timed region) ----
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import tempfile
        dump = os.path.join(tempfile.mkdtemp(prefix="rf_parity_"), "pair0.npz")
        try:
            nref = {2: 3, 3: 3, 4: 1, 5: 1}[cfg]
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(nref), "--warmup", "1",
                                "--config", str(cfg), "--dump-parity", dump], capture_output=True, text=True, timeout=420)
            ref = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
            cpu = ref["cpu_baseline"]
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": "pairs/s", "cores": usable_cores(), "kind": "port",
                   "sample": "CPU oracle did not finish in 420 s (%s)" % type(e).__name__}
        if cfg in (2, 3) and os.path.exists(dump):
            try:
                allref = dict(np.load(dump))
                sub = lambda pi: {k[:-2]: v for k, v in allref.items() if k.endswith("_%d" % pi)}
                parity = parity_report(rf, torch, sub(0), coarse, net, resident[0], args.engine, "pair 0")
                parity["pair1"] = parity_report(rf, torch, sub(1), coarse, net, resident[1], args.engine, "pair 1")
                parity["within_north_star"] = bool(parity["within_north_star"] and parity["pair1"]["within_north_star"])
            except Exception as e:  # noqa: BLE001
                parity = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0 and roofline is not None:
        # the whole pair against the chip: 655 GFLOP of convolutions + correlation per pair (SURVEY 8d), x3 MMAs on the split
        # engine; ~8.4 GB of algorithmic HBM traffic per pair at 4 B per activation element, every layer reading its inputs and writing
        # its output once (the fused conv3 + down-sampling GEMMs of the split engine move 1.1 GB less: profiles/r2_split_floor_analysis.txt)
        pps = P * args.steps / (ms_dev * 1e-3)                      # this GPU's pairs/s
        mma = 3.0 if args.engine == "f16x3" else 1.0
        gb = 8.4 if args.engine in ("f16x3", "fp32", "tf32") else 4.3
        pk = peaks()
        roofline["whole_pair"] = {"algorithmic_gflop_per_pair": 655.0 + 32.1, "algorithmic_tflops": (655.0 + 32.1) * pps / 1e3,
                                  "tensor_frac_algorithmic": (655.0 + 32.1) * pps / 1e3 / pk["bf16_tflops"],
                                  "tensor_frac_executed": mma * (655.0 + 32.1) * pps / 1e3 / pk["bf16_tflops"],
                                  "algorithmic_hbm_gb_per_pair": gb, "hbm_frac": gb * pps / pk["hbm_gbs"]}
    if rank == 0:
        hw8 = (H_img // 8) * (W_img // 8)
        d2h = int(H_img * W_img * 4 + 4 * hw8 * 4 + 9 * 4 + 64) if cfg in (2, 3) else (int(11 * (13 + 4 * hw8) * 4) if (cfg == 4 and graphed) else None)
        line = {
            "metric": METRIC, "value": world * P * args.steps / (ms_dev * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPES[args.engine], "data": "synthetic",
            "config": {"workload": WORKLOADS[cfg], "engine": args.engine, "pairs_per_gpu_per_step": P, "pairs_in_flight": lanes,
                       "parallelism": "pairs sharded i %% %d" % world,
                       "l2": "256 MiB buffer written between steps (L2 flush); activations per pair also exceed the 126 MB L2",
                       "preprocessing": "LANCZOS pyramid on the GPU (bit-exact PIL emulation)" if cfg != 5 else "coarse pyramid on the GPU; the two fine-level resizes with PIL on the host like the script",
                       "launch": ("one CUDA graph per pair" + (", %d independent pairs in flight on %d streams" % (lanes, lanes) if lanes > 1 else ""))
                                 + (" (the whole maxCoarse = 10 loop inside the graph: acceptance test and mask update on the device)" if cfg == 4 else "")
                                 if graphed else "stream launches, hypothesis loop steered from the host (12 bytes per hypothesis)"},
            "e2e": {"value": world * P * args.steps / (ms_e2e * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": P * 2 * H_img * W_img * 3,
                    "d2h_bytes_per_step": (P * d2h) if d2h else None},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "stages_ms": stages,
            "all_gather_ms": round(gather_ms, 3), "hypotheses_last_pair": nH_mean,
        }
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("RF_CONFIG", "2")), choices=[2, 3, 4, 5], help="BASELINE.json configs[N-1]")
    ap.add_argument("--engine", default=os.environ.get("RF_ENGINE", "f16x3"), choices=["f16x3", "fp32", "tf32", "f16", "f16-trunk"],
                    help="f16x3 (default): fp32-grade tcgen05 engine, fp16 hi/lo split operands, 3 MMAs per MAC; fp32: exact-FMA SIMT engine; "
                         "f16 / tf32 / f16-trunk: reduced-precision fast modes (10-bit operands)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("RF_LANES", "4")),
                    help="independent pairs in flight per GPU (each with its own CUDA graph, models' activation buffers and stream)")
    ap.add_argument("--pairs-per-step", type=int, default=int(os.environ.get("RF_PAIRS_PER_STEP", "0")),
                    help="pairs per GPU and step (default 32 for configs 2 / 3, 8 for config 4, 4 for config 5)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch the kernels of a pair one by one instead of replaying a CUDA graph")
    ap.add_argument("--dump-parity", default=None, help="(reference arm) write the oracle's outputs for pair 0 to this .npz")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the results of the last timed step (the region `value` times) to DIR/<name>.npy; same arguments, same inputs")
    args = ap.parse_args()
    if args.pairs_per_step <= 0:
        args.pairs_per_step = {2: 32, 3: 32, 4: 8, 5: 4}[args.config]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    # stdout carries exactly ONE line, the JSON record: whatever the libraries print meanwhile (NCCL writes its version / INFO lines
    # to file descriptor 1 when NCCL_DEBUG asks for them) goes to stderr
    sys.stdout.flush()
    fd_out = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(fd_out, "w")
    if world > 1:
        from ransac_flow_b200 import shard
        rank, world, local = shard.init_from_env("nccl")
    run_b200(args, rank, world, local)
    sys.stdout.flush()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
