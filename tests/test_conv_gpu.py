"""GPU parity of the tcgen05 implicit-GEMM convolution (forward, data gradient, weight gradient)
against torch.nn.functional.conv2d in fp32 on the same bf16-rounded operands.
Tolerance: bf16 inputs, fp32 accumulation -> relative error ~1e-2 on bf16 outputs (north_star)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from iswm_b200 import _lib, ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rel_err(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def _mk(B, Cin, H, W, Cout, k, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((B, Cin, H, W), generator=g).to(torch.bfloat16)
    w = (torch.randn((Cout, Cin, k, k), generator=g) * (2.0 / (Cin * k * k)) ** 0.5)
    return x, w


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _assert_healthy():
    torch.cuda.synchronize()
    code = ops.abort_code()
    assert code == 0, f"tensor-core kernel timed out on an mbarrier (code {code})"


CASES = [
    # B, Cin, H, W, Cout, k, dilation
    (2, 64, 16, 16, 64, 1, 1),
    (2, 256, 16, 16, 64, 1, 1),
    (1, 64, 32, 32, 256, 1, 1),
    (2, 64, 16, 16, 64, 3, 1),
    (2, 128, 32, 32, 128, 3, 1),
    (2, 512, 8, 8, 512, 3, 2),
    (1, 2048, 8, 8, 256, 3, 6),
    (1, 2048, 8, 8, 256, 3, 12),
    (2, 304, 16, 16, 256, 3, 1),
    (2, 256, 13, 13, 48, 1, 1),
    (2, 256, 9, 11, 2, 1, 1),
    (3, 64, 25, 25, 128, 3, 1),
    (2, 1024, 8, 8, 2048, 1, 1),
    # large dilations with taps that land INSIDE the image (OS16 rate 18, OS8 rates 24 / 36 of network/modeling.py:27-33);
    # a wrong tap offset cannot hide behind the zero padding here
    (1, 128, 48, 48, 64, 3, 18),
    (1, 128, 80, 80, 64, 3, 24),
    (1, 128, 80, 80, 64, 3, 36),
    (2, 64, 50, 77, 64, 3, 36),
    (1, 192, 40, 40, 256, 3, 12),
]


@pytest.mark.parametrize("B,Cin,H,W,Cout,k,dil", CASES)
def test_conv_fwd_raw_and_stats(B, Cin, H, W, Cout, k, dil):
    x, w = _mk(B, Cin, H, W, Cout, k)
    xd = _nhwc(x).to(DEV)
    wp = ops.pack_weight_fwd(w.to(DEV))
    out_ld = ((Cout + 7) // 8) * 8
    out = torch.zeros((B, H, W, out_ld), dtype=torch.bfloat16, device=DEV)
    stats = torch.zeros(2 * Cout, dtype=torch.float64, device=DEV)
    d = ops.make_conv_desc(B, H, W, Cin, Cin, B, H, W, Cout, out_ld, ops.conv_taps(k, dil), flags=_lib.EPI_STATS)
    ops.conv_igemm(d, xd, wp, out, stats=stats)
    _assert_healthy()
    ref = F.conv2d(x.float(), w.to(torch.bfloat16).float(), padding=dil * (k // 2), dilation=dil)
    got = out[..., :Cout].float().cpu().permute(0, 3, 1, 2)
    assert _rel_err(got, ref) < 1e-2
    s = stats.float().cpu()
    # the statistics are fp32 sums of the bf16 values the kernel STORED (what BatchNorm reads back)
    np.testing.assert_allclose(s[:Cout].numpy(), got.sum((0, 2, 3)).numpy(), rtol=1e-4, atol=2e-3)
    np.testing.assert_allclose(s[Cout:].numpy(), (got * got).sum((0, 2, 3)).numpy(), rtol=1e-4, atol=2e-3)
    # and stay within bf16 rounding noise of the unrounded sums
    np.testing.assert_allclose(s[:Cout].numpy(), ref.sum((0, 2, 3)).numpy(), rtol=2e-2, atol=0.5)


def test_conv_fwd_affine_relu_residual_f32():
    B, Cin, H, W, Cout = 2, 128, 16, 16, 256
    x, w = _mk(B, Cin, H, W, Cout, 1, seed=3)
    g = torch.Generator().manual_seed(4)
    scale = torch.rand(Cout, generator=g) + 0.5
    shift = torch.randn(Cout, generator=g)
    res = torch.randn((B, Cout, H, W), generator=g).to(torch.bfloat16)
    ref = F.relu(F.conv2d(x.float(), w.to(torch.bfloat16).float()) * scale[None, :, None, None] + shift[None, :, None, None] + res.float())
    xd, wp = _nhwc(x).to(DEV), ops.pack_weight_fwd(w.to(DEV))
    for f32 in (False, True):
        out = torch.zeros((B, H, W, Cout), dtype=torch.float32 if f32 else torch.bfloat16, device=DEV)
        flags = _lib.EPI_AFFINE | _lib.EPI_RELU | _lib.EPI_RESIDUAL | (_lib.EPI_OUT_F32 if f32 else 0)
        d = ops.make_conv_desc(B, H, W, Cin, Cin, B, H, W, Cout, Cout, ops.conv_taps(1, 1), flags=flags, res_ld=Cout)
        ops.conv_igemm(d, xd, wp, out, scale=scale.to(DEV), shift=shift.to(DEV), res=_nhwc(res).to(DEV))
        _assert_healthy()
        got = out.float().cpu().permute(0, 3, 1, 2)
        assert _rel_err(got, ref) < (2e-3 if f32 else 1e-2)


def test_conv_fwd_channel_slices():
    """input read from, and output written into, channel slices of wider buffers (concat in place)."""
    B, H, W = 2, 16, 16
    x, w = _mk(B, 64, H, W, 48, 1, seed=5)
    big_in = torch.randn((B, H, W, 128)).to(torch.bfloat16).to(DEV)
    big_in[..., 64:128] = _nhwc(x).to(DEV)
    big_out = torch.full((B, H, W, 304), 7.0, dtype=torch.bfloat16, device=DEV)
    d = ops.make_conv_desc(B, H, W, 64, 128, B, H, W, 48, 304, ops.conv_taps(1, 1))
    ops.conv_igemm(d, big_in[..., 64:], ops.pack_weight_fwd(w.to(DEV)), big_out[..., 8:])
    _assert_healthy()
    ref = F.conv2d(x.float(), w.to(torch.bfloat16).float())
    assert _rel_err(big_out[..., 8:56].float().cpu().permute(0, 3, 1, 2), ref) < 1e-2
    assert float(big_out[..., :8].float().min()) == 7.0 and float(big_out[..., 56:].float().min()) == 7.0


def test_conv_stride2_via_phases():
    B, Cin, H, W, Cout = 2, 128, 16, 16, 128
    x, w = _mk(B, Cin, H, W, Cout, 3, seed=6)
    ref = F.conv2d(x.float(), w.to(torch.bfloat16).float(), stride=2, padding=1)
    xn = _nhwc(x)
    phases = torch.stack([xn[:, p::2, q::2, :] for p in (0, 1) for q in (0, 1)], 0).contiguous().to(DEV)  # [4,B,H/2,W/2,C]
    Ho, Wo = H // 2, W // 2
    out = torch.zeros((B, Ho, Wo, Cout), dtype=torch.bfloat16, device=DEV)
    d = ops.make_conv_desc(B, Ho, Wo, Cin, Cin, 4 * B, Ho, Wo, Cout, Cout, ops.conv_taps_s2_3x3())
    ops.conv_igemm(d, phases, ops.pack_weight_fwd(w.to(DEV)), out)
    _assert_healthy()
    assert _rel_err(out.float().cpu().permute(0, 3, 1, 2), ref) < 1e-2


@pytest.mark.parametrize("B,Cin,H,W,Cout,k,dil", [(2, 64, 16, 16, 128, 3, 1), (1, 256, 8, 8, 512, 3, 2), (2, 256, 16, 16, 64, 1, 1), (2, 256, 9, 11, 2, 1, 1),
                                                   (1, 128, 48, 48, 64, 3, 18), (1, 128, 80, 80, 64, 3, 24), (1, 128, 80, 80, 64, 3, 36),
                                                   (2, 64, 50, 77, 64, 3, 36),
                                                   # 304 gradient channels (the decoder's first 3x3): 2 x 160-column tiles, the narrow last chunk of
                                                   # each tile written with plain stores; odd spatial size -> rows outside the image
                                                   (2, 304, 16, 16, 256, 3, 1), (1, 304, 13, 21, 64, 1, 1), (1, 328, 9, 9, 64, 1, 1)])
def test_conv_dgrad(B, Cin, H, W, Cout, k, dil):
    x, w = _mk(B, Cin, H, W, Cout, k, seed=7)
    g = torch.Generator().manual_seed(8)
    dy = torch.randn((B, Cout, H, W), generator=g).to(torch.bfloat16)
    xr = x.float().requires_grad_(True)
    F.conv2d(xr, w.to(torch.bfloat16).float(), padding=dil * (k // 2), dilation=dil).backward(dy.float())
    dy_ld = ((Cout + 7) // 8) * 8
    dyd = torch.zeros((B, H, W, dy_ld), dtype=torch.bfloat16, device=DEV)
    dyd[..., :Cout] = _nhwc(dy).to(DEV)
    wd = ops.pack_weight_dgrad(w.to(DEV))
    dx = torch.zeros((B, H, W, Cin), dtype=torch.bfloat16, device=DEV)
    taps = [(-a, -b, 0) for (a, b, _) in ops.conv_taps(k, dil)]
    d = ops.make_conv_desc(B, H, W, Cout, dy_ld, B, H, W, Cin, Cin, taps)
    ops.conv_igemm(d, dyd, wd, dx)
    _assert_healthy()
    assert _rel_err(dx.float().cpu().permute(0, 3, 1, 2), xr.grad) < 1e-2


@pytest.mark.parametrize("B,Cin,H,W,Cout,k,dil", [(2, 64, 16, 16, 64, 1, 1), (2, 64, 16, 16, 128, 3, 1), (1, 512, 8, 8, 256, 3, 2),
                                                   (2, 304, 16, 16, 256, 3, 1), (2, 256, 9, 11, 2, 1, 1), (4, 2048, 8, 8, 256, 3, 6),
                                                   (2, 256, 32, 32, 48, 1, 1),
                                                   (1, 128, 48, 48, 64, 3, 18), (1, 128, 80, 80, 64, 3, 24), (1, 128, 80, 80, 64, 3, 36),
                                                   (2, 64, 50, 77, 64, 3, 36),
                                                   # column-chunk tiles of the (tap, 64-channel slice) axis: partial slices in the middle of a
                                                   # tile (Cin = 96: 18 chunks), at its end (Cin = 160, 304), 27 chunks (Cin = 192), a 6-chunk
                                                   # 384-column tile as two MMAs (Cin = 128), Cout above one M tile
                                                   (2, 96, 12, 12, 64, 3, 1), (2, 160, 16, 16, 64, 1, 1), (2, 192, 16, 16, 320, 3, 1),
                                                   (2, 128, 16, 16, 128, 3, 1), (1, 304, 24, 24, 256, 3, 1), (2, 40, 10, 10, 72, 3, 1)])
def test_conv_wgrad(B, Cin, H, W, Cout, k, dil):
    x, w = _mk(B, Cin, H, W, Cout, k, seed=9)
    g = torch.Generator().manual_seed(10)
    dy = torch.randn((B, Cout, H, W), generator=g).to(torch.bfloat16)
    wr = w.clone().requires_grad_(True)
    F.conv2d(x.float(), wr, padding=dil * (k // 2), dilation=dil).backward(dy.float())
    dy_ld = ((Cout + 7) // 8) * 8
    dyd = torch.zeros((B, H, W, dy_ld), dtype=torch.bfloat16, device=DEV)
    dyd[..., :Cout] = _nhwc(dy).to(DEV)
    dw = torch.zeros((Cout, k * k, Cin), dtype=torch.float32, device=DEV)
    d = ops.make_conv_desc(B, H, W, Cin, Cin, B, H, W, Cout, dy_ld, ops.conv_taps(k, dil))
    ops.conv_wgrad(d, _nhwc(x).to(DEV), dyd, dw)
    _assert_healthy()
    grad = torch.empty((Cout, Cin, k, k), dtype=torch.float32, device=DEV)
    ops.unpack_wgrad(dw, grad)
    torch.cuda.synchronize()
    assert _rel_err(grad.cpu(), wr.grad) < 5e-3


@pytest.mark.parametrize("Cout,Cin,RS", [(3, 8, 9), (64, 64, 9), (5, 304, 9), (7, 1111, 9), (2, 2048, 9), (4, 16, 4), (6, 24, 1)])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_unpack_wgrad_exact(Cout, Cin, RS, beta):
    """[Cout][tap][Cin] accumulator -> OIHW gradient (tiled shared-memory transpose for k x k, generic otherwise): a pure
    permutation, so bit-exact; beta = 1 accumulates."""
    g = torch.Generator().manual_seed(Cout * 131 + Cin)
    dw = torch.randn((Cout, RS, Cin), generator=g)
    base = torch.randn((Cout, Cin, RS), generator=g)
    out = base.clone().to(DEV)
    from iswm_b200 import _lib
    _lib.check(_lib.lib().iswm_unpack_wgrad(dw.to(DEV).data_ptr(), Cout, Cin, RS, Cin, RS * Cin, beta, out.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream), "unpack_wgrad")
    want = dw.permute(0, 2, 1) + (base if beta else 0)
    assert torch.equal(out.cpu(), want)


@pytest.mark.parametrize("B,H,W,Cf,Cb,rates", [(2, 24, 24, 128, 64, (6, 12, 18)), (1, 40, 40, 256, 64, (12, 24, 36)), (2, 9, 11, 128, 128, (6, 12, 18))])
def test_aspp_bwd_k_concatenated_dgrad(B, H, W, Cf, Cb, rates):
    """iswm_aspp_bwd: ONE data-gradient GEMM over the 1x1 branch and the three dilated 3x3 branches of ASPP
    (network/_deeplab.py:143-172), K = 28 taps x Cb, against torch autograd of the four convolutions summed; also the
    accumulate form and the concatenated operand written by the batched packer (mode 1, row_ld = 28)."""
    g = torch.Generator().manual_seed(31)
    feat = torch.randn((B, Cf, H, W), generator=g).to(torch.bfloat16)
    ws = [torch.randn((Cb, Cf, 1, 1), generator=g) * (2.0 / Cf) ** 0.5] + [torch.randn((Cb, Cf, 3, 3), generator=g) * (2.0 / (9 * Cf)) ** 0.5 for _ in rates]
    dys = [torch.randn((B, Cb, H, W), generator=g).to(torch.bfloat16) for _ in range(4)]
    fr = feat.float().requires_grad_(True)
    outs = [F.conv2d(fr, ws[0].to(torch.bfloat16).float())] + [F.conv2d(fr, ws[i + 1].to(torch.bfloat16).float(), padding=r, dilation=r) for i, r in enumerate(rates)]
    torch.autograd.backward(outs, [d.float() for d in dys])
    # concatenated operand through the batched packer
    wd = [w.to(DEV) for w in ws]
    wcat = torch.zeros(Cf * 28 * Cb, dtype=torch.bfloat16, device=DEV)
    jobs, off = [], 0
    for w in wd:
        rs = w.shape[2] * w.shape[3]
        jobs.append((w.data_ptr(), wcat.data_ptr() + 2 * off * Cb, Cb, Cf, rs, Cb, 28, 1))
        off += rs
    arr, nblk = _lib.fill_pack_jobs(jobs)
    jd = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone().to(DEV)
    _lib.check(_lib.lib().iswm_pack_weights_batched(jd.data_ptr(), len(jobs), nblk, torch.cuda.current_stream().cuda_stream), "pack")
    # the slice of each branch equals its stand-alone dgrad packing
    cat = wcat.view(Cf, 28, Cb)
    off = 0
    for w in wd:
        rs = w.shape[2] * w.shape[3]
        assert torch.equal(cat[:, off:off + rs, :].contiguous().view(-1), ops.pack_weight_dgrad(w))
        off += rs
    dycat = torch.cat([_nhwc(d) for d in dys], dim=-1).contiguous().to(DEV)
    dfeat = torch.zeros((B, H, W, Cf), dtype=torch.bfloat16, device=DEV)
    ops.aspp_bwd(dycat, wcat, rates, dfeat)
    _assert_healthy()
    assert _rel_err(dfeat.float().cpu().permute(0, 3, 1, 2), fr.grad) < 1e-2
    base = torch.randn((B, H, W, Cf), generator=g).to(torch.bfloat16)
    acc = base.clone().to(DEV)
    ops.aspp_bwd(dycat, wcat, rates, acc, accumulate=True)
    _assert_healthy()
    assert _rel_err(acc.float().cpu().permute(0, 3, 1, 2), fr.grad + base.float().permute(0, 3, 1, 2)) < 1e-2


@pytest.mark.parametrize("B,Cin,H,W,Cout", [(2, 128, 16, 16, 128), (2, 64, 17, 13, 128), (1, 256, 9, 9, 64)])
@pytest.mark.parametrize("accumulate", [False, True])
def test_stride2_3x3_dgrad_by_parity_phases(B, Cin, H, W, Cout, accumulate):
    """Data gradient of a 3x3 / stride 2 / pad 1 convolution (network/backbone/resnet.py:27-30, first block of layers 2-3) as four
    small convolutions, one per parity phase of dx, each over a SUBSET of the packed weight taps with a strided output view
    (iswm_conv_desc.wtap / out_ws / out_hs / out_bs): 1 + 2 + 2 + 4 taps, no zero-stuffed tensor. Odd sizes included."""
    x, w = _mk(B, Cin, H, W, Cout, 3, seed=17)
    g = torch.Generator().manual_seed(18)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    dy = torch.randn((B, Cout, Ho, Wo), generator=g).to(torch.bfloat16)
    xr = x.float().requires_grad_(True)
    F.conv2d(xr, w.to(torch.bfloat16).float(), stride=2, padding=1).backward(dy.float())
    dyd = _nhwc(dy).to(DEV)
    wd = ops.pack_weight_dgrad(w.to(DEV))
    base = torch.randn((B, H, W, Cin), generator=g).to(torch.bfloat16)
    dx = base.clone().to(DEV) if accumulate else torch.full((B, H, W, Cin), 7.0, dtype=torch.bfloat16, device=DEV)
    for pu in (0, 1):
        rs = [(1, 0)] if pu == 0 else [(0, 1), (2, 0)]
        for pv in (0, 1):
            ss = [(1, 0)] if pv == 0 else [(0, 1), (2, 0)]
            Hp, Wp = (H - pu + 1) // 2, (W - pv + 1) // 2
            taps = [(di, dj, 0) for (r, di) in rs for (s, dj) in ss]
            wt = [r * 3 + s for (r, di) in rs for (s, dj) in ss]
            d = ops.make_conv_desc(B, Ho, Wo, Cout, Cout, B, Hp, Wp, Cin, Cin, taps, _lib.EPI_RESIDUAL if accumulate else 0, Cin if accumulate else 0,
                                   wtaps=wt, out_strides=(2 * Cin, 2 * W * Cin, H * W * Cin), w_ntaps=9)
            view = dx.view(-1)[(pu * W + pv) * Cin:]
            ops.conv_igemm(d, dyd, wd, view, res=view if accumulate else None)
    _assert_healthy()
    want = xr.grad + (base.float().permute(0, 3, 1, 2) if accumulate else 0)
    assert _rel_err(dx.float().cpu().permute(0, 3, 1, 2), want) < 1e-2


@pytest.mark.parametrize("Cout,rep", [(64, 8), (48, 8), (128, 3), (256, 2)])
def test_conv_stats_replicas_sum_to_the_single_accumulator(Cout, rep):
    """iswm_conv_desc.stats_replicas: CTA i adds its per-channel sums into copy i % replicas of the fp64 accumulator; the copies
    summed in fp64 give the fp32 statistics of the single-copy run bit for bit (what iswm_bn_train_apply reads)."""
    B, Cin, H, W = 4, 64, 40, 40
    x, w = _mk(B, Cin, H, W, Cout, 3, seed=31)
    xd, wp = _nhwc(x).to(DEV), ops.pack_weight_fwd(w.to(DEV))
    out_ld = ((Cout + 7) // 8) * 8
    res = []
    for r in (1, rep):
        out = torch.zeros((B, H, W, out_ld), dtype=torch.bfloat16, device=DEV)
        stats = torch.zeros(2 * Cout * r, dtype=torch.float64, device=DEV)
        d = ops.make_conv_desc(B, H, W, Cin, Cin, B, H, W, Cout, out_ld, ops.conv_taps(3, 1), flags=_lib.EPI_STATS)
        d.stats_replicas = r
        ops.conv_igemm(d, xd, wp, out, stats=stats)
        _assert_healthy()
        res.append((out.clone(), stats.view(r, 2 * Cout)))
    assert torch.equal(res[0][0], res[1][0])
    assert float(res[1][1].abs().sum(1).min()) > 0            # every copy received something (50 tiles over `rep` copies)
    assert torch.equal(res[0][1].sum(0).float(), res[1][1].sum(0).float())


@pytest.mark.parametrize("B,Cin,H,W,Cout,k", [(2, 128, 16, 16, 128, 3), (1, 64, 24, 40, 64, 3), (2, 256, 16, 16, 512, 1), (3, 64, 8, 8, 96, 1), (1, 128, 130, 128, 64, 3)])
def test_stride2_convs_read_the_parity_phases_in_place(B, Cin, H, W, Cout, k):
    """iswm_conv_desc.in_phase_view: the stride-2 3x3 (resnet.py:104 with stride 2) and the stride-2 1x1 downsample (:183) read
    the dense input through a 5-D tensor map {(column parity, channel), w, row parity, h, image} - no phase_split / subsample2
    copy - in the forward convolution and in the weight gradient. Against F.conv2d and its autograd weight gradient."""
    x, w = _mk(B, Cin, H, W, Cout, k, seed=51)
    g = torch.Generator().manual_seed(52)
    Ho, Wo = H // 2, W // 2
    dy = torch.randn((B, Cout, Ho, Wo), generator=g).to(torch.bfloat16)
    wr = w.to(torch.bfloat16).float().requires_grad_(True)
    y = F.conv2d(x.float(), wr, stride=2, padding=k // 2)
    y.backward(dy.float())
    xd = _nhwc(x).to(DEV)
    taps = ops.conv_taps(1, 1) if k == 1 else ops.conv_taps_s2_3x3()
    out = torch.zeros((B, Ho, Wo, Cout), dtype=torch.bfloat16, device=DEV)
    d = ops.make_conv_desc(B, Ho, Wo, Cin, Cin, B, Ho, Wo, Cout, Cout, taps, phase_view=True)
    ops.conv_igemm(d, xd, ops.pack_weight_fwd(w.to(DEV)), out)
    _assert_healthy()
    assert _rel_err(out.float().cpu().permute(0, 3, 1, 2), y.detach()) < 1e-2
    dw = torch.zeros((Cout, k * k, Cin), dtype=torch.float32, device=DEV)
    ops.conv_wgrad(d, xd, _nhwc(dy).to(DEV), dw)
    _assert_healthy()
    grad = torch.empty((Cout, Cin, k, k), dtype=torch.float32, device=DEV)
    ops.unpack_wgrad(dw, grad)
    torch.cuda.synchronize()
    assert _rel_err(grad.cpu(), wr.grad) < 5e-3


def test_grouped_weight_gradients_equal_the_single_launches():
    """iswm_conv_wgrad_grouped: one launch for a layer's worth of convolutions (work units dealt to the CTAs on the host) against
    one iswm_conv_wgrad per convolution: 1x1 / 3x3 / dilated, Cin tails, Cout below and above one M tile, a stride-2 job reading
    its input as parity phases in place, and more jobs than one launch holds (26 > 24). fp32 split order differs: 1e-5."""
    g = torch.Generator().manual_seed(61)
    shapes = [(2, 256, 16, 16, 64, 1, 1, False), (2, 64, 16, 16, 64, 3, 1, False), (2, 64, 16, 16, 256, 1, 1, False),
              (1, 128, 24, 24, 128, 3, 2, False), (2, 96, 12, 12, 72, 3, 1, False), (2, 304, 16, 16, 256, 3, 1, False),
              (2, 128, 16, 16, 128, 3, 1, True), (2, 256, 16, 16, 512, 1, 1, True), (3, 1024, 8, 8, 256, 1, 1, False)]
    shapes = shapes * 3                                         # 27 jobs -> two launches
    jobs, singles = [], []
    for (B, Cin, H, W, Cout, k, dil, s2) in shapes:
        x = torch.randn((B, H, W, Cin), generator=g).to(torch.bfloat16).to(DEV)
        if s2:
            Ho, Wo = H // 2, W // 2
            taps = ops.conv_taps(1, 1) if k == 1 else ops.conv_taps_s2_3x3()
            d = ops.make_conv_desc(B, Ho, Wo, Cin, Cin, B, Ho, Wo, Cout, Cout, taps, phase_view=True)
        else:
            Ho, Wo = H, W
            d = ops.make_conv_desc(B, H, W, Cin, Cin, B, H, W, Cout, Cout, ops.conv_taps(k, dil))
        dy = torch.randn((B, Ho, Wo, Cout), generator=g).to(torch.bfloat16).to(DEV)
        dw_g = torch.zeros((Cout, k * k, Cin), dtype=torch.float32, device=DEV)
        dw_s = torch.zeros_like(dw_g)
        jobs.append((d, x, dy, dw_g))
        singles.append((d, x, dy, dw_s))
    for (d, x, dy, dw) in singles:
        ops.conv_wgrad(d, x, dy, dw)
    ops.conv_wgrad_grouped(jobs)
    ops.conv_wgrad_grouped(jobs)                                # accumulates: twice the gradient
    _assert_healthy()
    for i, ((_, _, _, a), (_, _, _, b)) in enumerate(zip(jobs, singles)):
        scale = float(b.abs().max()) + 1e-6
        assert float((a - 2.0 * b).abs().max()) <= 2e-5 * scale * 2, (i, shapes[i])
