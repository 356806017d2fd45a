"""CPU-side checks: the C-ABI library loads and exports every symbol include/ransacflow_b200.h
declares, the host-side mirrors keep the reference's API surface, and compute calls fail loudly
without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import pair_oracle as PO
from oracle import synth


def header_symbols():
    src = open(os.path.join(ROOT, "include", "ransacflow_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rf_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(rf):
    lib = ctypes.CDLL(rf._lib.LIB_PATH)
    syms = header_symbols()
    assert len(syms) >= 24
    for s in syms:
        assert hasattr(lib, s), "missing export " + s
    assert set(syms) == set(rf._lib.SIGNATURES), "ctypes table and header disagree"
    assert rf._lib.lib.rf_version() >= 100


def test_workspace_queries_are_host_only(rf):
    assert rf._lib.lib.rf_ransac_workspace(1000) >= 1000 * (4 + 36)
    assert rf._lib.lib.rf_corr_mutual_nn_workspace(13065, 1200, 1024, 0) >= (13065 + 1200) * 8


def test_corr_kernel_sequence_query(rf):
    """rf_corr_mutual_nn_launches is host-only: 4 launches for the fp32 kernel, 6 for the 3xTF32 kernel with separate
    helpers, 3 for precision 2 (fused split / zeroing, persistent kernel, fused mutual test + compaction)."""
    L = rf._lib.lib
    assert (L.rf_corr_mutual_nn_launches(0), L.rf_corr_mutual_nn_launches(1), L.rf_corr_mutual_nn_launches(2)) == (4, 6, 3)


def test_lanczos_coefficients_match_pil(rf):
    """rf_lanczos_coeffs_host is host arithmetic: check it through a numpy emulation of the 8bpc
    resampler against PIL itself (bit exact)."""
    import PIL.Image as Image
    rs = np.random.RandomState(0)
    img = rs.randint(0, 256, (37, 53, 3)).astype(np.uint8)
    for (ow, oh) in [(96, 64), (20, 11), (53, 80)]:
        cur = img
        for axis, (insz, outsz) in ((1, (img.shape[1], ow)), (0, (img.shape[0], oh))):
            if insz == outsz:
                continue
            ks = ctypes.c_int(0)
            assert rf._lib.lib.rf_lanczos_coeffs_host(insz, outsz, None, None, 0, ctypes.byref(ks)) == 0
            b = np.zeros(2 * outsz, np.int32)
            kk = np.zeros(ks.value * outsz, np.int32)
            assert rf._lib.lib.rf_lanczos_coeffs_host(insz, outsz, b.ctypes.data_as(ctypes.c_void_p),
                                                      kk.ctypes.data_as(ctypes.c_void_p), kk.size, ctypes.byref(ks)) == 0
            kk = kk.reshape(outsz, ks.value)
            src = np.moveaxis(cur, axis, 0).astype(np.int64)
            out = np.zeros((outsz,) + src.shape[1:], np.int64)
            for o in range(outsz):
                lo, n = b[2 * o], b[2 * o + 1]
                acc = (1 << 21) + np.tensordot(kk[o, :n].astype(np.int64), src[lo:lo + n], axes=(0, 0))
                out[o] = np.clip(acc >> 22, 0, 255)
            cur = np.moveaxis(out.astype(np.uint8), 0, axis)
        ref = np.asarray(Image.fromarray(img).resize((ow, oh), resample=Image.LANCZOS))
        assert np.array_equal(cur, ref)


def test_state_dict_keys_match_reference_layout(rf):
    fe = rf.model.FeatureExtractor()
    assert set(fe.state_dict().keys()) == set(synth.feature_extractor_state(0).keys())
    fe.load_state_dict(synth.feature_extractor_state(0))            # strict
    nf, nm, nc = rf.model.NetFlowCoarse(7), rf.model.NetMatchability(7), rf.model.CorrNeigh(7)
    assert set(nf.state_dict().keys()) == set(synth.net_flow_coarse_state(1).keys())
    assert set(nm.state_dict().keys()) == set(synth.net_matchability_state(2).keys())
    assert len(nc.state_dict()) == 0
    nf.load_state_dict(synth.net_flow_coarse_state(1))
    nm.load_state_dict(synth.net_matchability_state(2))


def test_scale_list_and_sizes_match_oracle(rf):
    from importlib import import_module
    ca = import_module("ransac_flow_b200.coarseAlignFeatMatch")
    for n, r in [(7, 2), (3, 1.2), (5, 1.5), (1, 2)]:
        assert ca.scale_list(n, r) == PO.scale_list(n, r)
    a = ca.CoarseAlignA.__new__(ca.CoarseAlignA)
    a.strideNet = 16
    c = ca.CoarseAlignC.__new__(ca.CoarseAlignC)
    c.strideNet = 16
    for (w, h, ms) in [(640, 480, 480), (1241, 376, 800), (447, 315, 400), (720, 480, 960)]:
        assert a._target_size(w, h, ms) == PO.resized_size(w, h, ms, 16, "min")
        assert c._target_size(w, h, ms) == PO.resized_size(w, h, ms, 16, "max")
    # SURVEY A.5: 480x640, scaleR 2 -> NA = 13065
    sizes = [a._target_size(640, 480, int(480 * s)) for s in ca.scale_list(7, 2)]
    assert sum((w // 16) * (h // 16) for w, h in sizes) == 13065


def test_host_helpers_match_reference(rf):
    """The two helpers of ``outil`` that are host arithmetic in the product too: getWHTensor(_Int) (exact IEEE division on
    the host, cached) against the reference's golden output, and resizeImg (PIL) against the oracle's restatement."""
    import PIL.Image as Image
    g = np.load(os.path.join(ROOT, "tests", "golden", "wh_tensor.npz"))
    feat = torch.zeros(1, 4, int(g["h"]), int(g["w"]))
    W, H = rf.outil.getWHTensor(feat)
    Wi, Hi = rf.outil.getWHTensor_Int(feat)
    assert np.array_equal(W.numpy(), g["W"]) and np.array_equal(H.numpy(), g["H"])
    assert np.array_equal(Wi.numpy(), g["Wi"]) and np.array_equal(Hi.numpy(), g["Hi"])
    rs = np.random.RandomState(0)
    for (w, h, stride, ms) in [(1241, 376, 8, 650), (1241, 376, 8, 325), (640, 480, 16, 400), (123, 457, 8, 96)]:
        I = Image.fromarray(rs.randint(0, 256, (h, w, 3)).astype(np.uint8))
        a, b = rf.outil.resizeImg(I, stride, ms), PO.resize_img(I, stride, ms)
        assert a.size == b.size and a.size[0] % stride == 0 and a.size[1] % stride == 0
        assert np.array_equal(np.asarray(a), np.asarray(b))


def test_no_cpu_fallback(rf):
    x = torch.zeros(4, 8)
    with pytest.raises(rf._lib.RFError):
        rf.ops.l2norm(x)
    with pytest.raises(rf._lib.RFError):
        rf.outil.mutualMatching(torch.zeros(8, 4), torch.zeros(8, 4))
    with pytest.raises(rf._lib.RFError):
        rf.model.FeatureExtractor().eval()(torch.zeros(1, 3, 16, 16))
    with pytest.raises(rf._lib.RFError):
        rf.kornia_geometry.HomographyWarper(4, 4).warp_grid(torch.eye(3)[None])
    if not torch.cuda.is_available():
        with pytest.raises(rf._lib.RFError):
            rf.CoarseAlignA(7, 1000, 0.05, "Homography", 480, segNet=False, resnet_state_dict={})


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "ransac-flow_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_bench_product_arm_never_touches_oracle():
    """bench.py may execute oracle/ only on its CPU-baseline / --impl reference leg: every `oracle` import must sit inside
    run_reference(); the B200 arm gets its synthetic inputs from synthdata.py (no reference arithmetic)."""
    import ast
    tree = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    for fn in [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef)]:
        for node in ast.walk(fn):
            mods = []
            if isinstance(node, ast.Import):
                mods = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                mods = [node.module or ""]
            if any(m.split(".")[0] == "oracle" for m in mods):
                assert fn.name == "run_reference", "oracle imported in bench.%s" % fn.name
    top = [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
    assert not any("oracle" in ast.dump(n) for n in top)
    src = open(os.path.join(ROOT, "synthdata.py")).read()
    assert "import oracle" not in src and "from oracle" not in src and "ransac_flow_b200" not in src


def test_bench_roofline_record_is_complete():
    """bench.py's `roofline` object (pure arithmetic over the measured times): the keys the bench contract names, algorithmic work
    of config 2 (SURVEY 8d: 32.1 GFLOP, 58.4 MB) and the facts of the committed ncu capture."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    pk = dict(hbm_gbs=6575.1, bf16_tflops=1703.4, bf16_tflops_sustained=1450.6, src="measured")
    r = bench.roofline_record(2, True, 0.112, 0.039, 662, pk)
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(r["algorithmic_gflop"] - 2 * 13065 * 1200 * 1024 / 1e9) < 1e-9 and abs(r["algorithmic_mb"] - 58.44) < 0.01
    assert abs(r["achieved"] - 32.108544 / 0.112) < 1e-6 and abs(r["executed_tensor_frac"] - 3 * r["frac"]) < 1e-12
    assert r["traffic"] == bench.ncu_facts(2, True)["traffic"] and 55e6 < r["traffic"] < 70e6          # ~ the algorithmic bytes
    assert r["ncu_capture"] == "profiles/r2_ncu_full_kernels.json" and 0.5 < r["executed_tensor_frac_kernel_ncu"] < 1.0
    assert bench.roofline_record(0, False, 1.0, 0.04, 10, pk)["executed_tensor_frac"] is None and bench.ncu_facts(0, False) == {}
    assert abs(bench.roofline_record(1, False, 0.24, 0.04, 10, pk)["executed_tensor_frac"] - 6 * (32.108544 / 0.24) / 1703.4) < 1e-9


def test_bench_dump_outputs_names_dtypes_and_sample(tmp_path):
    """bench.py --dump-outputs: one float .npy per result leaf, large arrays as the same seeded sample every time, and no dump
    over 64 MB."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rs = np.random.RandomState(0)
    big = rs.rand(480, 640).astype(np.float32)
    outs = [dict(H=rs.rand(1, 3, 3), flowDown8=rs.rand(1, 2, 60, 80).astype(np.float32), match=[big], nbInlier=17, size=(480, 640),
                 maps=[(big > 0.5, np.arange(3))]) for _ in range(2)]
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(outs, str(d))
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted("pair%02d_%s.npy" % (r, k) for r in range(2)
                           for k in ("H", "flowDown8", "match_0", "nbInlier", "size", "maps_0_0", "maps_0_1"))
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
    assert np.array_equal(np.load(tmp_path / "a" / "pair00_H.npy"), outs[0]["H"])
    assert np.load(tmp_path / "a" / "pair01_nbInlier.npy") == 17 and np.load(tmp_path / "a" / "pair00_size.npy").dtype == np.float64
    m = np.load(tmp_path / "a" / "pair00_match_0.npy")
    assert m.shape == (bench.DUMP_SAMPLE,) and np.isin(m, big).all()
    with pytest.raises(SystemExit):
        bench.dump_outputs([dict(match=[big])] * (bench.DUMP_MAX_BYTES // (4 * bench.DUMP_SAMPLE) + 1), str(tmp_path / "c"))
    assert not (tmp_path / "c").exists()


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU oracle timed on the host cores; rank 0 only under torchrun) prints ONE JSON line with
    the contract's keys; a non-zero rank prints nothing and exits 0."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, RF_CPU_THREADS="8")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["steps"] == 1
    assert d["metric"].startswith("image-pairs/sec at 480x640") and d["config"]["workload"].startswith("config2")
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) < 1e-6 * d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 8 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    r1 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                        capture_output=True, text=True, timeout=120, env=dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_dropin_installs_the_reference_module_names(rf, tmp_path):
    """The names the reference's drivers import by bare name resolve to this package (SURVEY 8b)."""
    import runpy
    import sys
    from ransac_flow_b200 import dropin
    saved = {k: sys.modules.get(k) for k in ("coarseAlignFeatMatch", "outil", "model", "kornia", "kornia.geometry")}
    try:
        for script, cls in (("x/quick_start/a.py", rf.CoarseAlignC), ("x/evaluation/evalYFCC/evaluation.py", rf.CoarseAlignB),
                            ("x/evaluation/evalHpatch/evaluation.py", rf.CoarseAlignA)):
            dropin.install(dropin.variant_for(script))
            drv = tmp_path / "drv.py"
            drv.write_text("from coarseAlignFeatMatch import CoarseAlign\nimport outil\nimport model as model\n"
                           "import kornia.geometry as tgm\nW = tgm.HomographyWarper(4, 4)\n"
                           "names = (outil.RANSAC, outil.Homography, outil.mutualMatching, outil.getWHTensor, model.FeatureExtractor,\n"
                           "         model.CorrNeigh, model.NetFlowCoarse, model.NetMatchability, model.predFlowCoarse)\n")
            ns = runpy.run_path(str(drv))
            assert ns["CoarseAlign"] is cls and ns["outil"] is rf.outil and ns["model"] is rf.model
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
