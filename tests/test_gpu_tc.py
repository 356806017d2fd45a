"""tcgen05 engine: TF32 implicit-GEMM convolution and 3xTF32 correlation vs fp32 references."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import outil_oracle as OO
from test_gpu_matching import check_same
from test_gpu_ops import ragged

pytestmark = pytest.mark.gpu
TF32_TOL = 4e-3          # two TF32-truncated operands (2^-10 each), fp32 accumulation


@pytest.mark.parametrize("cin,cout,k,sizes", [
    (64, 49, 3, [(6, 8)]), (128, 1, 3, [(6, 8), (6, 8)]), (64, 512, 3, [(60, 80)]),
    (64, 64, 3, [(24, 32), (9, 7)]), (64, 64, 1, [(16, 16)]), (64, 256, 1, [(13, 17), (6, 5), (1, 1)]),
    (128, 128, 3, [(16, 16), (16, 16)]), (256, 64, 1, [(30, 40)]), (1024, 256, 1, [(15, 20), (30, 40)]),
    (256, 256, 3, [(15, 20), (33, 25)]), (256, 1024, 1, [(20, 15), (40, 30)]), (512, 128, 1, [(60, 80)]),
    (64, 48, 3, [(12, 20)]), (128, 16, 3, [(6, 8)]), (32, 32, 3, [(128, 3), (3, 128)])])
@pytest.mark.parametrize("relu,res,stride", [(True, True, 1), (False, False, 1), (True, False, 2)])
def test_conv2d_tf32(rf, cin, cout, k, sizes, relu, res, stride):
    g = torch.Generator().manual_seed(cin + cout * 3 + k)
    xs = [torch.randn(1, cin, h, w, generator=g) for h, w in sizes]
    w = torch.randn(cout, cin, k, k, generator=g) / np.sqrt(cin * k * k)
    bias = torch.randn(cout, generator=g)
    refs = [F.conv2d(x, w, bias, stride=stride, padding=k // 2) for x in xs]
    rs = [torch.randn(r.shape, generator=g) for r in refs] if res else None
    if res:
        refs = [a + b for a, b in zip(refs, rs)]
    if relu:
        refs = [F.relu(r) for r in refs]
    wp = w.permute(2, 3, 1, 0).reshape(k * k * cin, cout).contiguous().cuda()
    wtc = w.permute(0, 2, 3, 1).reshape(cout, k * k * cin).contiguous().cuda()
    y = rf.ops.conv2d(ragged(rf, xs), wp, bias.cuda(), cout, k, stride, k // 2, relu, ragged(rf, rs) if res else None,
                      rf.ops.ENGINE_TF32, wtc)
    torch.cuda.synchronize()
    for i, r in enumerate(refs):
        got = y.image(i).cpu()
        assert tuple(got.shape) == tuple(r.shape)
        err = (got - r).abs().max().item()
        assert err <= TF32_TOL * max(1.0, r.abs().max().item()), (err, r.abs().max().item())


F16_TOL = 2e-3           # fp16 output rounding (2^-11 relative) + fp32 accumulation order


@pytest.mark.parametrize("cin,cout,k,sizes", [
    (64, 64, 3, [(24, 32), (9, 7)]), (64, 64, 3, [(120, 160), (60, 80), (33, 47)]), (64, 64, 1, [(16, 16)]),
    (64, 256, 1, [(13, 17), (6, 5), (1, 1)]), (128, 128, 3, [(16, 16), (16, 16)]), (256, 64, 1, [(30, 40)]),
    (1024, 256, 1, [(15, 20), (30, 40)]), (256, 256, 3, [(15, 20), (33, 25)]), (256, 1024, 1, [(20, 15), (40, 30)]),
    (512, 128, 1, [(60, 80)]), (192, 64, 1, [(37, 53)]), (64, 48, 3, [(12, 20)]), (128, 8, 3, [(6, 8)]), (512, 2048, 1, [(9, 5)])])
@pytest.mark.parametrize("relu,res,stride", [(True, True, 1), (False, False, 1), (True, False, 2)])
def test_conv2d_f16(rf, cin, cout, k, sizes, relu, res, stride):
    """Engine 2: fp16 activations and weights through tcgen05 kind::f16, fp32 accumulation, fp16 output.  The
    reference is an fp32 convolution of the same fp16-rounded operands."""
    g = torch.Generator().manual_seed(cin + cout * 3 + k)
    xs = [torch.randn(1, cin, h, w, generator=g).half() for h, w in sizes]
    w = (torch.randn(cout, cin, k, k, generator=g) / np.sqrt(cin * k * k)).half()
    bias = torch.randn(cout, generator=g)
    refs = [F.conv2d(x.float(), w.float(), bias, stride=stride, padding=k // 2) for x in xs]
    rs = [torch.randn(r.shape, generator=g).half() for r in refs] if res else None
    if res:
        refs = [a + b.float() for a, b in zip(refs, rs)]
    if relu:
        refs = [F.relu(r) for r in refs]
    wtc = w.permute(0, 2, 3, 1).reshape(cout, k * k * cin).contiguous().cuda()
    y = rf.ops.conv2d(ragged(rf, xs), None, bias.cuda(), cout, k, stride, k // 2, relu, ragged(rf, rs) if res else None,
                      rf.ops.ENGINE_F16, wtc)
    torch.cuda.synchronize()
    assert y.data.dtype == torch.float16
    for i, r in enumerate(refs):
        got = y.image(i).float().cpu()
        assert tuple(got.shape) == tuple(r.shape)
        err = (got - r).abs().max().item()
        assert err <= F16_TOL * max(1.0, r.abs().max().item()), (err, r.abs().max().item())


@pytest.mark.parametrize("env", [{}, {"RF_TC_RESPF": "1"}])
@pytest.mark.parametrize("cin,cout,k,stride,res,sizes", [
    (64, 256, 1, 1, True, [(120, 160), (60, 80), (33, 47)]), (256, 64, 1, 1, False, [(120, 160), (31, 17)]),
    (512, 1024, 1, 2, False, [(60, 80), (30, 44)]), (128, 128, 3, 2, False, [(64, 96), (37, 41)]),
    (256, 1024, 1, 1, True, [(30, 40), (60, 80), (15, 20)]), (128, 512, 1, 1, True, [(9, 7)]),
    (256, 64, 1, 1, False, [(240, 320)])])                                  # 600 tiles: tc_pipe_kernel<64>
def test_conv2d_f16_kernel_variants(rf, monkeypatch, env, cin, cout, k, stride, res, sizes):
    """fp16 tap-streaming convolutions on both sides of the kernel selection: the pipelined persistent kernel (two
    epilogue groups, producer-issued residual prefetch; >= 4 K blocks and >= 2 tiles per SM) and the one-tile kernel,
    also with its residual prefetch (RF_TC_RESPF, read per call).  All must agree with the fp32 reference."""
    for kk, v in env.items():
        monkeypatch.setenv(kk, v)
    g = torch.Generator().manual_seed(cin + cout + k + stride)
    xs = [torch.randn(1, cin, h, w, generator=g).half() for h, w in sizes]
    w = (torch.randn(cout, cin, k, k, generator=g) / np.sqrt(cin * k * k)).half()
    bias = torch.randn(cout, generator=g)
    refs = [F.conv2d(x.float(), w.float(), bias, stride=stride, padding=k // 2) for x in xs]
    rs = [torch.randn(r.shape, generator=g).half() for r in refs] if res else None
    if res:
        refs = [a + b.float() for a, b in zip(refs, rs)]
    refs = [F.relu(r) for r in refs]
    wtc = w.permute(0, 2, 3, 1).reshape(cout, k * k * cin).contiguous().cuda()
    y = rf.ops.conv2d(ragged(rf, xs), None, bias.cuda(), cout, k, stride, k // 2, True, ragged(rf, rs) if res else None,
                      rf.ops.ENGINE_F16, wtc)
    torch.cuda.synchronize()
    for i, r in enumerate(refs):
        err = (y.image(i).float().cpu() - r).abs().max().item()
        assert err <= F16_TOL * max(1.0, r.abs().max().item()), (env, err, r.abs().max().item())


def test_f16_engine_saturates_and_rejects_unsupported_shapes(rf):
    x = torch.full((1, 64, 4, 4), 200.0).half()
    w = torch.full((8, 64, 1, 1), 100.0).half()
    y = rf.ops.conv2d(ragged(rf, [x]), None, None, 8, 1, 1, 0, False, None, rf.ops.ENGINE_F16, w.reshape(8, 64).cuda())
    assert torch.isfinite(y.data.float()).all() and float(y.data.float().max()) == 65504.0
    with pytest.raises(rf._lib.RFError):     # Cin % 64 != 0: no fp16 path and no silent fallback
        rf.ops.conv2d(ragged(rf, [x[:, :32]]), None, None, 8, 1, 1, 0, False, None, rf.ops.ENGINE_F16, w.reshape(8, 64)[:, :32].contiguous().cuda())


def test_tf32_engine_falls_back_to_fp32_kernels_for_unsupported_shapes(rf):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 3, 16, 16, generator=g)                       # 3-channel stem: not a TMA-able operand
    w = torch.randn(64, 3, 7, 7, generator=g) / 12
    ref = F.conv2d(x, w, stride=2, padding=3)
    wp = w.permute(2, 3, 1, 0).reshape(147, 64).contiguous().cuda()
    wtc = w.permute(0, 2, 3, 1).reshape(64, 147).contiguous().cuda()
    y = rf.ops.conv2d(ragged(rf, [x]), wp, None, 64, 7, 2, 3, False, None, rf.ops.ENGINE_TF32, wtc)
    assert (y.image(0).cpu() - ref).abs().max().item() < 2e-5        # exact-fp32 SIMT path


@pytest.mark.parametrize("C,NA,NB,seed", [(1024, 13065, 1200, 0), (1024, 2107, 300, 1), (64, 129, 127, 2), (256, 1, 1, 4),
                                           (1024, 300, 1200, 5), (32, 500, 260, 6)])
@pytest.mark.parametrize("precision", [1, 2])
def test_corr_3xtf32_matches_fp32_argmax(rf, C, NA, NB, seed, precision):
    """precision 1 = 3xTF32, 2 = fp16 split (hi + lo * 2^-11, two TMEM accumulators): both carry 22 significand bits."""
    if precision == 2 and C % 64:
        pytest.skip("fp16 split needs C % 64 == 0")
    rs = np.random.RandomState(seed)
    A = np.abs(rs.randn(C, NA)).astype(np.float32)
    B = np.abs(rs.randn(C, NB)).astype(np.float32)
    n = min(NA, NB) // 2
    B[:, :n] = A[:, rs.permutation(NA)[:n]] + 0.1 * np.abs(rs.randn(C, n)).astype(np.float32)
    A /= np.linalg.norm(A, axis=0, keepdims=True)
    B /= np.linalg.norm(B, axis=0, keepdims=True)
    if NB > 2:
        B[:, 1] = 0
    o1, o2, score = OO.mutualMatching(A, B, return_score=True)
    rf.outil.corr_precision = precision
    try:
        i1, i2 = rf.outil.mutualMatching(torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda())
    finally:
        rf.outil.corr_precision = 0
    nd = check_same(i1.cpu().numpy(), i2.cpu().numpy(), o1, o2, score)
    print("precision %d vs fp32 oracle: %d matches, %d differing (ambiguous) pairs" % (precision, len(o1), nd))
    # and against the library's own exact-fp32 kernel
    j1, j2 = rf.outil.mutualMatching(torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda())
    check_same(i1.cpu().numpy(), i2.cpu().numpy(), j1.cpu().numpy(), j2.cpu().numpy(), score)


def test_corr_kitti_shape_both_engines_agree(rf):
    """BASELINE config 5 shape (KITTI at coarseSize 800): NA = 25747, NB = 8250, C = 1024 (435 GFLOP, 850 MB score
    matrix in the reference).  The 3xTF32 tensor-core kernel and the exact-fp32 kernel must produce the same pairs."""
    g = torch.Generator().manual_seed(0)
    A = torch.nn.functional.normalize(torch.rand(25747, 1024, generator=g), dim=1).cuda()
    B = torch.nn.functional.normalize(torch.rand(8250, 1024, generator=g), dim=1).cuda()
    B[:3000] = torch.nn.functional.normalize(A[torch.randperm(25747, generator=g)[:3000].cuda()] + 0.05 * torch.rand(3000, 1024, device="cuda"), dim=1)
    j1, j2, n2 = rf.ops.corr_mutual_nn(A, B, 0)
    n2 = int(n2.item())
    b = set(zip(j1[:n2].tolist(), j2[:n2].tolist()))
    for precision in (1, 2):
        i1, i2, n1 = rf.ops.corr_mutual_nn(A, B, precision)
        n1 = int(n1.item())
        a = set(zip(i1[:n1].tolist(), i2[:n1].tolist()))
        print("KITTI-shaped correlation, precision %d: %d / %d pairs, %d differ" % (precision, n1, n2, len(a ^ b)))
        assert n1 >= 3000 and len(a ^ b) <= 2          # arg-max ties below fp32 accumulation noise only


@pytest.mark.parametrize("C,NA,NB,seed", [(1024, 13065, 1200, 0), (1024, 2107, 300, 1), (64, 129, 127, 2), (256, 1, 1, 4),
                                           (1024, 300, 1200, 5), (128, 5000, 130, 6), (64, 128, 128, 7), (192, 40000, 257, 8)])
def test_corr_persistent_kernel_sequence(rf, C, NA, NB, seed):
    """Precision 2 runs three launches: fused split / key zeroing, the persistent correlation kernel (two TMEM accumulator
    pairs, arg-max epilogue overlapped with the next tile's MMAs), fused mutual test + compaction.  Its pairs come in row
    order and agree with the fp32 oracle and with the library's exact-fp32 kernel up to arg-max ties below fp32
    accumulation noise."""
    rs = np.random.RandomState(seed)
    A = np.abs(rs.randn(C, NA)).astype(np.float32)
    B = np.abs(rs.randn(C, NB)).astype(np.float32)
    n = min(NA, NB) // 2
    B[:, :n] = A[:, rs.permutation(NA)[:n]] + 0.1 * np.abs(rs.randn(C, n)).astype(np.float32)
    A /= np.linalg.norm(A, axis=0, keepdims=True)
    B /= np.linalg.norm(B, axis=0, keepdims=True)
    if NB > 2:
        B[:, 1] = 0                              # masked target cell: never matches
    fa, fb = torch.from_numpy(A.T.copy()).cuda(), torch.from_numpy(B.T.copy()).cuda()
    assert rf._lib.lib.rf_corr_mutual_nn_launches(2) == 3
    for rep in range(2):                         # twice: the workspace keys must be re-zeroed by the call itself
        i1, i2, cnt = rf.ops.corr_mutual_nn(fa, fb, 2)
    k = int(cnt.item())
    got = (i1[:k].cpu().numpy(), i2[:k].cpu().numpy())
    assert np.all(np.diff(got[0]) > 0)
    o1, o2, score = OO.mutualMatching(A, B, return_score=True)
    check_same(got[0], got[1], o1, o2, score)
    j1, j2, n0 = rf.ops.corr_mutual_nn(fa, fb, 0)
    n0 = int(n0.item())
    check_same(got[0], got[1], j1[:n0].cpu().numpy(), j2[:n0].cpu().numpy(), score)


@pytest.mark.parametrize("C,NA,NB,seed", [(1024, 13065, 1200, 0), (1024, 2107, 300, 1), (64, 129, 127, 2), (256, 1, 1, 4), (1024, 300, 1200, 5),
                                           (1024, 25747, 8250, 7), (64, 60000, 300, 8)])
def test_corr_presplit_operands_and_column_compaction_identical(rf, C, NA, NB, seed):
    """rf_corr_mutual_nn_presplit (operand planes written by rf_l2norm_split_nhwc, key memset, persistent kernel, compaction)
    == rf_corr_mutual_nn at precision 2 (split launch, persistent kernel, compaction): identical index lists.  The
    compaction is column-driven while NA row flags fit in shared memory (NA <= 51200) and row-driven beyond; the largest
    shape takes the row-driven kernel in both calls and is also checked against the fp32 oracle."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.cat([torch.randn(NA + NB, C, generator=g).abs()]).cuda()
    raw[NA:NA + min(NA, NB) // 2] = raw[torch.randperm(NA, generator=g)[:min(NA, NB) // 2].cuda()] + 0.05 * raw[NA:NA + min(NA, NB) // 2]
    if NB > 2:
        raw[NA + 1] = 0                                           # an all-zero (masked) target row never matches
    planes = rf.ops.l2norm_planes(rf.ops.to_split(raw))           # [2, NA + NB, C]
    rows = rf.ops.from_split(planes)                              # the fp32 values those planes stand for
    ref = rf.ops.corr_mutual_nn(rows[:NA].contiguous(), rows[NA:].contiguous(), 2)
    nref = int(ref[2].item())
    for _ in range(2):                                            # twice: the keys are re-zeroed per call
        got = rf.ops.corr_mutual_nn_presplit(planes[0, :NA], planes[1, :NA], planes[0, NA:], planes[1, NA:])
        n = int(got[2].item())
        assert n == nref and torch.equal(got[0][:n], ref[0][:n]) and torch.equal(got[1][:n], ref[1][:n])
    again = rf.ops.corr_mutual_nn(rows[:NA].contiguous(), rows[NA:].contiguous(), 2)
    assert int(again[2].item()) == nref and torch.equal(again[0][:n], ref[0][:n])
    if NA * 4 > 200 * 1024:
        A, B = rows[:NA].T.cpu().numpy().copy(), rows[NA:].T.cpu().numpy().copy()
        o1, o2, score = OO.mutualMatching(A, B, return_score=True)
        check_same(got[0][:n].cpu().numpy(), got[1][:n].cpu().numpy(), o1, o2, score)
    assert nref >= 1 and (NB <= 2 or not bool((ref[1][:nref] == 1).any()))
