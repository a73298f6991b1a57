"""GPU parity of the HBM-bound glue kernels against stock torch ops in fp32 on the same
bf16-rounded inputs (tolerances: one bf16 rounding of the output, 2^-8 relative)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from iswm_b200 import _lib
from iswm_b200._lib import check

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
L = _lib.lib


def st():
    return torch.cuda.current_stream().cuda_stream


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def nchw(x):
    return x.permute(0, 3, 1, 2).contiguous()


def close(a, b, rtol=1e-2, atol=1e-2):
    np.testing.assert_allclose(a.float().cpu().numpy(), b.float().cpu().numpy(), rtol=rtol, atol=atol)


def rnd(shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(torch.bfloat16)


@pytest.mark.parametrize("B,C,H,W,relu,with_res", [(2, 64, 9, 7, True, False), (3, 48, 8, 8, True, True), (2, 256, 5, 5, False, False), (2, 2048, 4, 4, True, True),
                                                    (4, 64, 96, 96, True, False), (4, 256, 48, 48, True, True), (2, 1024, 9, 11, True, False),
                                                    (3, 304, 7, 5, True, True), (2, 512, 16, 16, False, True)])
def test_bn_train_apply_and_two_launch_backward(B, C, H, W, relu, with_res):
    x = rnd((B, C, H, W), 1, 2.0)
    res = rnd((B, C, H, W), 2) if with_res else None
    g = torch.Generator().manual_seed(3)
    gamma = torch.rand(C, generator=g) + 0.5
    beta = torch.randn(C, generator=g) * 0.2
    rm, rv = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    dout = rnd((B, C, H, W), 4)
    # torch reference
    xr = x.float().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    rm_ref, rv_ref = rm.clone(), rv.clone()
    y = F.batch_norm(xr, rm_ref, rv_ref, gr, br, True, 0.1, 1e-5)
    resr = res.float().requires_grad_(True) if with_res else None
    if with_res:
        y = y + resr
    if relu:
        y = F.relu(y)
    y.backward(dout.float())
    # ours
    M = B * H * W
    xd = nhwc(x).to(DEV)
    stats = torch.stack([x.double().sum((0, 2, 3)), (x.double() ** 2).sum((0, 2, 3))]).reshape(-1).to(DEV)
    out = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    save = torch.empty(2 * C, dtype=torch.float32, device=DEV)
    rmd, rvd = rm.to(DEV), rv.to(DEV)
    nbt = torch.zeros((), dtype=torch.long, device=DEV)
    gd, bd = gamma.to(DEV), beta.to(DEV)
    resd = nhwc(res).to(DEV) if with_res else None
    check(L().iswm_bn_train_apply(xd.data_ptr(), C, stats.data_ptr(), 1, M, C, gd.data_ptr(), bd.data_ptr(), 1e-5, 0.1, rmd.data_ptr(), rvd.data_ptr(),
                                  nbt.data_ptr(), save.data_ptr(), save[C:].data_ptr(), None if resd is None else resd.data_ptr(), C,
                                  1 if relu else 0, 0.0, 0, None, out.data_ptr(), C, None, st()))
    close(nchw(out), y.detach(), 1e-2, 2e-2)
    close(rmd, rm_ref, 1e-4, 1e-5)
    close(rvd, rv_ref, 1e-3, 1e-4)
    assert nbt.item() == 1
    dd = nhwc(dout).to(DEV)
    sums = torch.zeros(2 * C, dtype=torch.float64, device=DEV)
    # units without a residual recompute the ReLU mask from x (act = NULL); residual units read the block output
    act_ptr = out.data_ptr() if with_res else None
    check(L().iswm_bn_bwd_reduce(dd.data_ptr(), C, xd.data_ptr(), C, act_ptr, C, M, C, save.data_ptr(), save[C:].data_ptr(),
                                 gd.data_ptr(), bd.data_ptr(), 1 if relu else 0, 0.0, 0, None, sums.data_ptr(), st()))
    if relu and not with_res:                       # both mask sources must agree bit for bit
        sums2 = torch.zeros(2 * C, dtype=torch.float64, device=DEV)
        check(L().iswm_bn_bwd_reduce(dd.data_ptr(), C, xd.data_ptr(), C, out.data_ptr(), C, M, C, save.data_ptr(), save[C:].data_ptr(),
                                     gd.data_ptr(), bd.data_ptr(), 1, 0.0, 0, None, sums2.data_ptr(), st()))
        assert torch.equal(sums.float(), sums2.float())   # fp64 accumulators: atomics order is invisible in fp32
    dx = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    dz = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    dg = torch.zeros(C, dtype=torch.float32, device=DEV)
    db = torch.zeros(C, dtype=torch.float32, device=DEV)
    check(L().iswm_bn_bwd_apply(dd.data_ptr(), C, xd.data_ptr(), C, act_ptr, C, M, C, gd.data_ptr(), bd.data_ptr(), save.data_ptr(), save[C:].data_ptr(),
                                sums.data_ptr(), 1 if relu else 0, 0.0, 0, None, dx.data_ptr(), C, dz.data_ptr(), C, dg.data_ptr(), db.data_ptr(), st()))
    scale = float(xr.grad.abs().max())
    close(nchw(dx), xr.grad, 2e-2, 2e-2 * scale)
    close(dg, gr.grad, 2e-2, 5e-2)
    close(db, br.grad, 2e-2, 5e-2)
    if with_res:
        close(nchw(dz), resr.grad, 1e-2, 1e-2)
    if relu and with_res:
        # packed ReLU sign bits (one byte per 8 channels) instead of the activation: identical sums and gradients
        bits = torch.zeros((M, C // 8), dtype=torch.uint8, device=DEV)
        out_b = torch.empty_like(out)
        check(L().iswm_bn_train_apply(xd.data_ptr(), C, stats.data_ptr(), 1, M, C, gd.data_ptr(), bd.data_ptr(), 1e-5, 0.1, None, None, None,
                                      save.data_ptr(), save[C:].data_ptr(), resd.data_ptr(), C, 1, 0.0, 0, None, out_b.data_ptr(), C, bits.data_ptr(), st()))
        assert torch.equal(out_b, out)
        want = (out.float().reshape(M, C // 8, 8) > 0).to(torch.int32) * (2 ** torch.arange(8, device=DEV, dtype=torch.int32))
        assert torch.equal(bits.to(torch.int32), want.sum(-1))
        sums_b = torch.zeros(2 * C, dtype=torch.float64, device=DEV)
        check(L().iswm_bn_bwd_reduce(dd.data_ptr(), C, xd.data_ptr(), C, bits.data_ptr(), 0, M, C, save.data_ptr(), save[C:].data_ptr(),
                                     gd.data_ptr(), bd.data_ptr(), 2, 0.0, 0, None, sums_b.data_ptr(), st()))
        assert torch.equal(sums_b.float(), sums.float())
        dx_b = torch.empty_like(dx); dz_b = torch.empty_like(dz)
        dg_b = torch.zeros(C, dtype=torch.float32, device=DEV); db_b = torch.zeros(C, dtype=torch.float32, device=DEV)
        check(L().iswm_bn_bwd_apply(dd.data_ptr(), C, xd.data_ptr(), C, bits.data_ptr(), 0, M, C, gd.data_ptr(), bd.data_ptr(), save.data_ptr(), save[C:].data_ptr(),
                                    sums.data_ptr(), 2, 0.0, 0, None, dx_b.data_ptr(), C, dz_b.data_ptr(), C, dg_b.data_ptr(), db_b.data_ptr(), st()))
        assert torch.equal(dx_b, dx) and torch.equal(dz_b, dz) and torch.equal(dg_b, dg) and torch.equal(db_b, db)


def test_maxpool_fwd_bwd():
    B, C, H, W = 2, 64, 13, 18
    x = rnd((B, C, H, W), 5)
    xr = x.float().requires_grad_(True)
    y = F.max_pool2d(xr, 3, 2, 1)
    dout = rnd(tuple(y.shape), 6)
    y.backward(dout.float())
    Ho, Wo = y.shape[2:]
    out = torch.empty((B, Ho, Wo, C), dtype=torch.bfloat16, device=DEV)
    idx = torch.empty((B, Ho, Wo, C), dtype=torch.uint8, device=DEV)
    xd = nhwc(x).to(DEV)
    check(L().iswm_maxpool_fwd(xd.data_ptr(), B, H, W, C, Ho, Wo, out.data_ptr(), idx.data_ptr(), st()))
    assert torch.equal(nchw(out).float().cpu(), y.detach())
    dx = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_maxpool_bwd(nhwc(dout).to(DEV).data_ptr(), idx.data_ptr(), B, H, W, C, Ho, Wo, dx.data_ptr(), st()))
    close(nchw(dx), xr.grad, 1e-2, 1e-2)


@pytest.mark.parametrize("Hi,Wi,Ho,Wo", [(4, 4, 16, 16), (13, 13, 50, 50), (8, 6, 17, 23), (1, 1, 5, 5), (7, 5, 25, 17), (32, 32, 128, 128)])
def test_bilinear_fwd_bwd(Hi, Wi, Ho, Wo):
    B, C = 2, 16
    x = rnd((B, C, Hi, Wi), 7)
    xr = x.float().requires_grad_(True)
    y = F.interpolate(xr, size=(Ho, Wo), mode="bilinear", align_corners=False)
    dout = rnd((B, C, Ho, Wo), 8)
    y.backward(dout.float())
    out = torch.full((B, Ho, Wo, 24), 3.0, dtype=torch.bfloat16, device=DEV)
    xd = nhwc(x).to(DEV)
    check(L().iswm_bilinear_fwd(xd.data_ptr(), C, B, Hi, Wi, C, Ho, Wo, out[..., 8:].data_ptr(), 24, st()))
    close(nchw(out[..., 8:]), y.detach(), 1e-2, 1e-2)
    assert float(out[..., :8].float().min()) == 3.0
    dx = torch.empty((B, Hi, Wi, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_bilinear_bwd(nhwc(dout).to(DEV).data_ptr(), C, B, Hi, Wi, C, Ho, Wo, dx.data_ptr(), C, st()))
    close(nchw(dx), xr.grad, 1e-2, 2e-2 * float(xr.grad.abs().max()))


@pytest.mark.parametrize("Hi,Wi,Ho,Wo,C", [(16, 16, 64, 64, 2), (13, 11, 50, 41, 3), (25, 17, 97, 65, 2), (7, 9, 7, 9, 5), (3, 5, 31, 77, 7)])
def test_logits_up_fwd_bwd(Hi, Wi, Ho, Wo, C):
    B = 2
    g = torch.Generator().manual_seed(9)
    x = torch.randn((B, C, Hi, Wi), generator=g)
    xr = x.clone().requires_grad_(True)
    y = F.interpolate(xr, size=(Ho, Wo), mode="bilinear", align_corners=False)
    dout = torch.randn((B, C, Ho, Wo), generator=g)
    y.backward(dout)
    out = torch.empty((B, C, Ho, Wo), dtype=torch.float32, device=DEV)
    check(L().iswm_logits_up_fwd(nhwc(x).to(DEV).data_ptr(), B, Hi, Wi, C, Ho, Wo, out.data_ptr(), st()))
    close(out, y.detach(), 1e-5, 1e-5)
    dx = torch.empty((B, Hi, Wi, 8), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_logits_up_bwd(dout.to(DEV).data_ptr(), B, Hi, Wi, C, Ho, Wo, dx.data_ptr(), 8, None, st()))
    close(nchw(dx[..., :C]), xr.grad, 1e-2, 1e-2 * float(xr.grad.abs().max()))
    assert torch.count_nonzero(dx[..., C:]).item() == 0
    # the same sweep with the classifier bias gradient riding along (accumulated into a non-zero start)
    dx2 = torch.empty_like(dx)
    bias2 = torch.full((C,), 0.5, dtype=torch.float32, device=DEV)
    check(L().iswm_logits_up_bwd(dout.to(DEV).data_ptr(), B, Hi, Wi, C, Ho, Wo, dx2.data_ptr(), 8, bias2.data_ptr(), st()))
    assert torch.equal(dx2, dx)
    close(bias2 - 0.5, dout.sum((0, 2, 3)), 1e-4, 1e-3)
    bias = torch.zeros(C, dtype=torch.float32, device=DEV)
    check(L().iswm_bias_grad_nchw(dout.to(DEV).data_ptr(), B, C, Ho * Wo, bias.data_ptr(), st()))
    close(bias, dout.sum((0, 2, 3)), 1e-4, 1e-3)


def test_gap_broadcast_sum():
    B, C, H, W = 3, 2048, 5, 7
    x = rnd((B, C, H, W), 10)
    xd = nhwc(x).to(DEV)
    out = torch.empty((B, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_gap_fwd(xd.data_ptr(), C, B, H * W, C, out.data_ptr(), st()))
    close(out, x.float().mean((2, 3)), 1e-2, 1e-2)
    s = torch.empty((B, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_sum_hw(xd.data_ptr(), C, B, H * W, C, s.data_ptr(), st()))
    close(s, x.float().sum((2, 3)), 1e-2, 5e-2)
    v = rnd((B, 256), 11).to(DEV)
    cat = torch.zeros((B, H, W, 1280), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_broadcast_hw(v.data_ptr(), B, H * W, 256, cat[..., 1024:].data_ptr(), 1280, st()))
    assert torch.equal(cat[..., 1024:], v[:, None, None, :].expand(B, H, W, 256))
    assert torch.count_nonzero(cat[..., :1024]).item() == 0
    dx = torch.ones((B, H, W, 256), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_gap_bwd_add(v.data_ptr(), B, H * W, 256, dx.data_ptr(), 256, st()))
    close(dx, 1.0 + v.float()[:, None, None, :].expand(B, H, W, 256) / (H * W), 1e-2, 1e-2)


@pytest.mark.parametrize("H,W", [(8, 8), (9, 7)])
def test_stride2_helpers(H, W):
    B, C = 2, 16
    x = rnd((B, C, H, W), 12)
    xn = nhwc(x).to(DEV)
    Hp, Wp = (H + 1) // 2, (W + 1) // 2
    ph = torch.empty((4, B, Hp, Wp, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_phase_split(xn.data_ptr(), C, B, H, W, C, ph.data_ptr(), st()))
    for p in (0, 1):
        for q in (0, 1):
            ref = torch.zeros((B, Hp, Wp, C), dtype=torch.bfloat16, device=DEV)
            sub = xn[:, p::2, q::2, :]
            ref[:, :sub.shape[1], :sub.shape[2]] = sub
            assert torch.equal(ph[p * 2 + q], ref)
    ss = torch.empty((B, Hp, Wp, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_subsample2(xn.data_ptr(), C, B, H, W, C, ss.data_ptr(), st()))
    assert torch.equal(ss, xn[:, ::2, ::2, :])
    z = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_zero_stuff2(ss.data_ptr(), B, Hp, Wp, C, H, W, z.data_ptr(), st()))
    ref = torch.zeros_like(z)
    ref[:, ::2, ::2, :] = ss
    assert torch.equal(z, ref)
    acc = torch.ones((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_scatter2_add(ss.data_ptr(), B, Hp, Wp, C, H, W, acc.data_ptr(), st()))
    close(acc, 1.0 + ref.float(), 1e-2, 1e-2)


def test_stem_im2col_and_pack():
    B, H, W = 2, 18, 22
    g = torch.Generator().manual_seed(13)
    img = torch.randn((B, 3, H, W), generator=g)
    w = torch.randn((64, 3, 7, 7), generator=g) * 0.1
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    col = torch.empty((B * Ho * Wo, 160), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_stem_im2col(img.to(DEV).data_ptr(), B, 3, H, W, Ho, Wo, 160, col.data_ptr(), st()))
    from iswm_b200 import ops
    wp = ops.pack_weight_fwd(w.to(DEV), stem=True).view(64, 192)
    got = (col.float() @ wp[:, :160].float().t()).view(B, Ho, Wo, 64)
    ref = F.conv2d(img.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), stride=2, padding=3)
    close(nchw(got), ref, 1e-3, 1e-3)
    assert torch.count_nonzero(col[:, 147:]).item() == 0


@pytest.mark.parametrize("B,H,W", [(1, 200, 200), (2, 65, 301)])
def test_stem_im2col_strips_and_edges(B, H, W):
    """several 64-pixel strips per row, ragged last strip, odd sizes: against unfold of the padded image."""
    g = torch.Generator().manual_seed(5)
    img = torch.randn((B, 3, H, W), generator=g)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    col = torch.full((B * Ho * Wo, 160), 7.0, dtype=torch.bfloat16, device=DEV)
    check(L().iswm_stem_im2col(img.to(DEV).data_ptr(), B, 3, H, W, Ho, Wo, 160, col.data_ptr(), st()))
    unf = F.unfold(img, kernel_size=7, padding=3, stride=2)            # [B, 3*49, Ho*Wo], row = c*49 + t
    ref = unf.view(B, 3, 49, Ho * Wo).permute(0, 3, 2, 1).reshape(B * Ho * Wo, 147)   # col = t*3 + c
    assert torch.equal(col[:, :147].cpu(), ref.to(torch.bfloat16))
    assert torch.count_nonzero(col[:, 147:]).item() == 0


def test_pack_weights_batched_matches_single_kernels():
    """the smem-tiled batched packer must reproduce the element-wise packers bit for bit."""
    import ctypes as C
    from iswm_b200 import ops, _lib
    g = torch.Generator().manual_seed(21)
    shapes = [(64, 3, 7, 7, True), (64, 64, 1, 1, False), (256, 304, 3, 3, False), (48, 256, 1, 1, False),
              (2, 256, 1, 1, False), (128, 128, 3, 3, False), (256, 1280, 1, 1, False), (72, 40, 3, 3, False)]
    jobs, expect = [], []
    keep = []
    for (Cout, Cin, R, S, stem) in shapes:
        w = (torch.randn((Cout, Cin, R, S), generator=g)).to(DEV)
        keep.append(w)
        RS = R * S
        if stem:
            cin_pad, row_ld = Cin, ((RS * Cin + 63) // 64) * 64
        else:
            cin_pad = ((Cin + 63) // 64) * 64
            row_ld = RS * cin_pad
        dst = torch.full((Cout * row_ld,), 3.0, dtype=torch.bfloat16, device=DEV)
        jobs.append((w.data_ptr(), dst.data_ptr(), Cout, Cin, RS, cin_pad, row_ld, 0))
        expect.append((dst, ops.pack_weight_fwd(w, stem=stem)))
        if not stem:
            cout_pad = ((Cout + 63) // 64) * 64
            dst2 = torch.full((Cin * RS * cout_pad,), 3.0, dtype=torch.bfloat16, device=DEV)
            jobs.append((w.data_ptr(), dst2.data_ptr(), Cout, Cin, RS, cout_pad, 0, 1))
            expect.append((dst2, ops.pack_weight_dgrad(w)))
    arr, nblk = _lib.fill_pack_jobs(jobs)
    dj = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone().to(DEV)
    check(L().iswm_pack_weights_batched(dj.data_ptr(), len(jobs), nblk, st()))
    torch.cuda.synchronize()
    for i, (got, ref) in enumerate(expect):
        assert torch.equal(got, ref), f"job {i} {jobs[i][2:]}"


def test_sgd_step_matches_torch():
    g = torch.Generator().manual_seed(14)
    p0 = torch.randn(10007, generator=g)
    p_ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.SGD([p_ref], lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    p = p0.clone().to(DEV)
    mom = torch.zeros_like(p)
    for step in range(3):
        grad = torch.randn(10007, generator=g)
        p_ref.grad = grad.clone()
        opt.step()
        check(L().iswm_sgd_step(p.data_ptr(), grad.to(DEV).data_ptr(), mom.data_ptr(), p.numel(), 1e-3, 0.9, 1e-4, 1, 1 if step == 0 else 0, None, st()))
    close(p, p_ref.detach(), 1e-6, 1e-7)


@pytest.mark.parametrize("B,C,H,W,p", [(4, 256, 16, 16, 0.1), (2, 64, 9, 7, 0.5), (3, 256, 32, 32, 0.25)])
def test_bn_backward_with_dropout_against_torch_with_the_kernels_own_mask(B, C, H, W, p):
    """ASPP projection unit (network/_deeplab.py:163-166: conv -> BN -> ReLU -> Dropout(0.1)): the forward kernel's keep
    mask is recovered from its output (kept elements are y / (1 - p), dropped ones 0 where relu(y) > 0) and INJECTED into a
    torch fp32 restatement y * mask / (1 - p); bn_bwd_reduce / bn_bwd_apply with drop_p > 0 (which regenerate the mask from
    the counter-based hash) must then produce torch's gradients. SURVEY 7 'hard parts': Dropout parity by mask injection."""
    x = rnd((B, C, H, W), 11, 2.0)
    g = torch.Generator().manual_seed(12)
    gamma = torch.rand(C, generator=g) + 0.5
    beta = torch.randn(C, generator=g) * 0.2
    dout = rnd((B, C, H, W), 13)
    M = B * H * W
    seed, step = 0x5EED + 41, torch.tensor([7], dtype=torch.int64, device=DEV)
    xd = nhwc(x).to(DEV)
    stats = torch.stack([x.double().sum((0, 2, 3)), (x.double() ** 2).sum((0, 2, 3))]).reshape(-1).to(DEV)
    out = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    save = torch.empty(2 * C, dtype=torch.float32, device=DEV)
    gd, bd = gamma.to(DEV), beta.to(DEV)
    check(L().iswm_bn_train_apply(xd.data_ptr(), C, stats.data_ptr(), 1, M, C, gd.data_ptr(), bd.data_ptr(), 1e-5, 0.1, None, None, None,
                                  save.data_ptr(), save[C:].data_ptr(), None, C, 1, p, seed, step.data_ptr(), out.data_ptr(), C, None, st()))
    # the keep mask depends on (seed, step, element index) only: the same launch WITHOUT the ReLU leaves bn(x) * keep / (1 - p),
    # which is zero exactly where the element was dropped (bn(x) == 0 itself has measure zero)
    probe = torch.empty_like(out)
    check(L().iswm_bn_train_apply(xd.data_ptr(), C, stats.data_ptr(), 1, M, C, gd.data_ptr(), bd.data_ptr(), 1e-5, 0.1, None, None, None,
                                  save.data_ptr(), save[C:].data_ptr(), None, C, 0, p, seed, step.data_ptr(), probe.data_ptr(), C, None, st()))
    mask = (nchw(probe).float().cpu() != 0).float()
    frac = float(mask.mean())
    assert abs(frac - (1 - p)) < 0.02, f"keep fraction {frac:.4f} vs 1-p = {1 - p}"
    # torch: the same unit with that mask injected
    xr = x.float().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    y = F.relu(F.batch_norm(xr, None, None, gr, br, True, 0.1, 1e-5))
    got = nchw(out).float().cpu()
    close(got, (y * mask / (1 - p)).detach(), 1e-2, 2e-2)
    (y * mask / (1 - p)).backward(dout.float())
    dd = nhwc(dout).to(DEV)
    sums = torch.zeros(2 * C, dtype=torch.float64, device=DEV)
    check(L().iswm_bn_bwd_reduce(dd.data_ptr(), C, xd.data_ptr(), C, None, C, M, C, save.data_ptr(), save[C:].data_ptr(),
                                 gd.data_ptr(), bd.data_ptr(), 1, p, seed, step.data_ptr(), sums.data_ptr(), st()))
    dx = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    dg = torch.zeros(C, dtype=torch.float32, device=DEV)
    db = torch.zeros(C, dtype=torch.float32, device=DEV)
    check(L().iswm_bn_bwd_apply(dd.data_ptr(), C, xd.data_ptr(), C, None, C, M, C, gd.data_ptr(), bd.data_ptr(), save.data_ptr(), save[C:].data_ptr(),
                                sums.data_ptr(), 1, p, seed, step.data_ptr(), dx.data_ptr(), C, None, 0, dg.data_ptr(), db.data_ptr(), st()))
    scale = float(xr.grad.abs().max())
    # an element whose bn(x) lies within bf16 rounding of the ReLU edge may carry a flipped ReLU mask: tolerated as a tiny population
    err = (nchw(dx).float().cpu() - xr.grad).abs()
    assert float((err > 2e-2 * scale + 2e-2 * xr.grad.abs()).float().mean()) < 2e-3
    close(dg, gr.grad, 3e-2, 2e-2 * float(gr.grad.abs().max()))
    close(db, br.grad, 3e-2, 2e-2 * float(br.grad.abs().max()))
    # a different step counter draws a different mask (the graph-replayed step advances it on the device)
    out2 = torch.empty_like(out)
    step2 = torch.tensor([8], dtype=torch.int64, device=DEV)
    check(L().iswm_bn_train_apply(xd.data_ptr(), C, stats.data_ptr(), 1, M, C, gd.data_ptr(), bd.data_ptr(), 1e-5, 0.1, None, None, None,
                                  save.data_ptr(), save[C:].data_ptr(), None, C, 1, p, seed, step2.data_ptr(), out2.data_ptr(), C, None, st()))
    assert not torch.equal(out2, out)


@pytest.mark.parametrize("B,C,H,W", [(2, 256, 9, 7), (3, 64, 8, 8), (2, 2048, 4, 4), (4, 512, 24, 24), (2, 1024, 9, 11)])
def test_dual_batchnorm_of_a_downsample_block_against_torch(B, C, H, W):
    """csrc/bn_dual.cu: out = relu(bn3(raw) + bn_ds(raw_ds)) and its backward, both BatchNorms per pass, against torch autograd
    (network/backbone/resnet.py:110-118 with a downsample branch) on the same bf16 inputs."""
    from iswm_b200 import _lib
    import ctypes as Ct
    xa, xb = rnd((B, C, H, W), 11, 2.0), rnd((B, C, H, W), 12, 1.5)
    g = torch.Generator().manual_seed(13)
    ga, ba = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.2
    gb, bb = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.2
    rma, rva = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    rmb, rvb = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    dout = rnd((B, C, H, W), 14)
    # torch
    xar, xbr = xa.float().requires_grad_(True), xb.float().requires_grad_(True)
    gar, bar_, gbr, bbr = (t.clone().requires_grad_(True) for t in (ga, ba, gb, bb))
    rma_r, rva_r, rmb_r, rvb_r = rma.clone(), rva.clone(), rmb.clone(), rvb.clone()
    y = F.relu(F.batch_norm(xar, rma_r, rva_r, gar, bar_, True, 0.1, 1e-5) + F.batch_norm(xbr, rmb_r, rvb_r, gbr, bbr, True, 0.1, 1e-5))
    y.backward(dout.float())
    # ours
    M = B * H * W
    xad, xbd = nhwc(xa).to(DEV), nhwc(xb).to(DEV)
    sta = torch.stack([xa.double().sum((0, 2, 3)), (xa.double() ** 2).sum((0, 2, 3))]).reshape(-1).to(DEV)
    stb = torch.stack([xb.double().sum((0, 2, 3)), (xb.double() ** 2).sum((0, 2, 3))]).reshape(-1).to(DEV)
    dev = lambda t: t.clone().to(DEV)
    gad, bad, gbd, bbd, rmad, rvad, rmbd, rvbd = (dev(t) for t in (ga, ba, gb, bb, rma, rva, rmb, rvb))
    nbta, nbtb = torch.zeros((), dtype=torch.long, device=DEV), torch.full((), 5, dtype=torch.long, device=DEV)
    sva, svb = torch.empty(2 * C, device=DEV), torch.empty(2 * C, device=DEV)
    out = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    bits = torch.zeros((M, C // 8), dtype=torch.uint8, device=DEV)
    sa = _lib.BnSide(sta.data_ptr(), gad.data_ptr(), bad.data_ptr(), rmad.data_ptr(), rvad.data_ptr(), nbta.data_ptr(), sva.data_ptr(), sva[C:].data_ptr())
    sb = _lib.BnSide(stb.data_ptr(), gbd.data_ptr(), bbd.data_ptr(), rmbd.data_ptr(), rvbd.data_ptr(), nbtb.data_ptr(), svb.data_ptr(), svb[C:].data_ptr())
    check(L().iswm_bn_dual_train_apply(xad.data_ptr(), C, Ct.byref(sa), xbd.data_ptr(), C, Ct.byref(sb), M, C, 1e-5, 0.1, out.data_ptr(), C, bits.data_ptr(), st()))
    close(nchw(out), y.detach(), 1e-2, 2e-2)
    close(rmad, rma_r, 1e-4, 1e-5); close(rvad, rva_r, 1e-3, 1e-4); close(rmbd, rmb_r, 1e-4, 1e-5); close(rvbd, rvb_r, 1e-3, 1e-4)
    assert nbta.item() == 1 and nbtb.item() == 6
    want = (out.float().reshape(M, C // 8, 8) > 0).to(torch.int32) * (2 ** torch.arange(8, device=DEV, dtype=torch.int32))
    assert torch.equal(bits.to(torch.int32), want.sum(-1))
    dd = nhwc(dout).to(DEV)
    s1, s2 = torch.zeros(2 * C, dtype=torch.float64, device=DEV), torch.zeros(2 * C, dtype=torch.float64, device=DEV)
    check(L().iswm_bn_dual_bwd_reduce(dd.data_ptr(), C, bits.data_ptr(), xad.data_ptr(), C, Ct.byref(sa), xbd.data_ptr(), C, Ct.byref(sb), M, C,
                                      s1.data_ptr(), s2.data_ptr(), st()))
    # each half against the single-branch reduction with the same sign bits
    for xd, sv, gd, bd, s in ((xad, sva, gad, bad, s1), (xbd, svb, gbd, bbd, s2)):
        ref = torch.zeros(2 * C, dtype=torch.float64, device=DEV)
        check(L().iswm_bn_bwd_reduce(dd.data_ptr(), C, xd.data_ptr(), C, bits.data_ptr(), 0, M, C, sv.data_ptr(), sv[C:].data_ptr(),
                                     gd.data_ptr(), bd.data_ptr(), 2, 0.0, 0, None, ref.data_ptr(), st()))
        mag = float(ref.abs().max()) + 1.0
        np.testing.assert_allclose(s.cpu().numpy(), ref.cpu().numpy(), rtol=1e-5, atol=1e-5 * mag)
    dxa, dxb = torch.empty_like(out), torch.empty_like(out)
    dga, dba, dgb, dbb = (torch.zeros(C, device=DEV) for _ in range(4))
    check(L().iswm_bn_dual_bwd_apply(dd.data_ptr(), C, bits.data_ptr(), xad.data_ptr(), C, Ct.byref(sa), s1.data_ptr(), xbd.data_ptr(), C, Ct.byref(sb),
                                     s2.data_ptr(), M, C, dxa.data_ptr(), C, dxb.data_ptr(), C, dga.data_ptr(), dba.data_ptr(), dgb.data_ptr(), dbb.data_ptr(), st()))
    torch.cuda.synchronize()
    for dx, xr_, dg, gr_, db, br_ in ((dxa, xar, dga, gar, dba, bar_), (dxb, xbr, dgb, gbr, dbb, bbr)):
        scale = float(xr_.grad.abs().max())
        close(nchw(dx), xr_.grad, 2e-2, 2e-2 * scale)
        close(dg, gr_.grad, 2e-2, 5e-2)
        close(db, br_.grad, 2e-2, 5e-2)


@pytest.mark.parametrize("kp", [32, 24])
@pytest.mark.parametrize("B,H,W", [(2, 18, 22), (1, 65, 49), (2, 200, 131), (1, 7, 9)])
def test_stem_row_taps_forward_and_weight_gradient(B, H, W, kp):
    """Stem 7x7 / stride 2 / pad 3 (network/backbone/resnet.py:144) in ROW-TAP form: iswm_stem_rows (image unrolled along x, two
    row-parity phases, bit-exact against the padded image), then the 7 kernel rows as taps of iswm_conv_igemm / iswm_conv_wgrad
    with the mode-2 packed weights and iswm_unpack_wgrad_stem, against F.conv2d and its autograd weight gradient. Odd sizes:
    the odd phase has one row less (zero row), ragged edges."""
    import ctypes as Ct
    from iswm_b200 import ops
    g = torch.Generator().manual_seed(17)
    img = torch.randn((B, 3, H, W), generator=g)
    w = torch.randn((64, 3, 7, 7), generator=g) * 0.1
    H1, W1 = (H + 1) // 2, (W + 1) // 2
    rows = torch.full((2 * B, H1, W1, kp), 7.0, dtype=torch.bfloat16, device=DEV)
    check(L().iswm_stem_rows(img.to(DEV).data_ptr(), B, 3, H, W, H1, W1, kp, rows.data_ptr(), st()))
    pad = F.pad(img, (3, 3 + 2, 0, 2))                                    # x: 3 left / right (+ slack for odd W), y: slack rows below
    ref = torch.zeros((2, B, H1, W1, 24))
    for p in range(2):
        for hh in range(H1):
            h = 2 * hh + p
            if h >= H:
                continue
            for s_ in range(7):
                # element [.., wo, s*3 + c] = img[b, c, h, 2*wo + s - 3]  (padded coordinates: 2*wo + s)
                ref[p, :, hh, :, 3 * s_:3 * s_ + 3] = pad[:, :, h, s_:s_ + 2 * W1:2][:, :, :W1].permute(0, 2, 1)
    assert torch.equal(rows.cpu().view(2, B, H1, W1, kp)[..., :24], ref.to(torch.bfloat16))
    assert torch.count_nonzero(rows[..., 21:]).item() == 0
    # forward: 7 row taps over the two phases
    arr, nblk = _lib.fill_pack_jobs([(w.to(DEV).data_ptr(), 0, 64, 3, 49, 64, 448, 2)])
    wd = w.to(DEV)
    wp = torch.empty(64 * 448, dtype=torch.bfloat16, device=DEV)
    arr, nblk = _lib.fill_pack_jobs([(wd.data_ptr(), wp.data_ptr(), 64, 3, 49, 64, 448, 2)])
    jobs = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone().to(DEV)
    check(L().iswm_pack_weights_batched(jobs.data_ptr(), 1, nblk, st()))
    taps = [((r - 3 - ((r + 1) & 1)) // 2, 0, (r + 1) & 1) for r in range(7)]
    out = torch.zeros((B, H1, W1, 64), dtype=torch.bfloat16, device=DEV)
    d = ops.make_conv_desc(B, H1, W1, kp, kp, 2 * B, H1, W1, 64, 64, taps)
    ops.conv_igemm(d, rows, wp, out)
    torch.cuda.synchronize()
    assert ops.abort_code() == 0
    wr = w.to(torch.bfloat16).float().requires_grad_(True)
    y = F.conv2d(img.to(torch.bfloat16).float(), wr, stride=2, padding=3)
    close(nchw(out), y.detach(), 1e-2, 1e-2)
    # weight gradient
    dy = rnd((B, 64, H1, W1), 18)
    y.backward(dy.float())
    acc = torch.zeros((64, 7, kp), dtype=torch.float32, device=DEV)
    ops.conv_wgrad(d, rows, nhwc(dy).to(DEV), acc)
    grad = torch.zeros((64, 3, 7, 7), dtype=torch.float32, device=DEV)
    check(L().iswm_unpack_wgrad_stem(acc.data_ptr(), 64, 3, 7, kp, 0.0, grad.data_ptr(), st()))
    torch.cuda.synchronize()
    assert ops.abort_code() == 0
    assert float((grad.cpu() - wr.grad).abs().max()) <= 5e-3 * float(wr.grad.abs().max())
    assert torch.count_nonzero(acc[:, :, 21:]).item() == 0


@pytest.mark.parametrize("B,H,W", [(2, 16, 16), (1, 33, 47), (3, 64, 40), (1, 9, 7)])
def test_stem_bn_relu_maxpool_forward_fused_against_the_separate_kernels(B, H, W):
    """csrc/stem_pool.cu (resnet.py:145-147): BatchNorm + ReLU + maxpool in one pass against bn_train_apply -> maxpool_fwd.
    Pooled values, argmax codes, saved statistics: bit-identical."""
    import ctypes as Ct
    C = 64
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    M = B * H * W
    raw = rnd((B, C, H, W), 41, 2.0)
    rawd = nhwc(raw).to(DEV)
    g = torch.Generator().manual_seed(42)
    gamma, beta = (torch.rand(C, generator=g) + 0.5).to(DEV), (torch.randn(C, generator=g) * 0.3).to(DEV)
    rep = 4
    st1 = torch.stack([raw.double().sum((0, 2, 3)), (raw.double() ** 2).sum((0, 2, 3))]).reshape(-1).to(DEV)
    stats = torch.zeros(rep * 2 * C, dtype=torch.float64, device=DEV)
    stats.view(rep, 2 * C)[0] = st1 * 0.25
    stats.view(rep, 2 * C)[1] = st1 * 0.5
    stats.view(rep, 2 * C)[3] = st1 * 0.25                       # copies that sum to the statistics (copy 2 stays empty)
    # separate kernels
    rm1, rv1 = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    nbt1 = torch.zeros((), dtype=torch.long, device=DEV)
    save1 = torch.empty(2 * C, device=DEV)
    act = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=DEV)
    check(L().iswm_bn_train_apply(rawd.data_ptr(), C, stats.data_ptr(), rep, M, C, gamma.data_ptr(), beta.data_ptr(), 1e-5, 0.1, rm1.data_ptr(), rv1.data_ptr(),
                                  nbt1.data_ptr(), save1.data_ptr(), save1[C:].data_ptr(), None, 0, 1, 0.0, 0, None, act.data_ptr(), C, None, st()))
    pooled1 = torch.empty((B, Ho, Wo, C), dtype=torch.bfloat16, device=DEV)
    idx1 = torch.empty((B, Ho, Wo, C), dtype=torch.uint8, device=DEV)
    check(L().iswm_maxpool_fwd(act.data_ptr(), B, H, W, C, Ho, Wo, pooled1.data_ptr(), idx1.data_ptr(), st()))
    # fused
    rm2, rv2 = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    nbt2 = torch.zeros((), dtype=torch.long, device=DEV)
    save2 = torch.empty(2 * C, device=DEV)
    side = _lib.BnSide(stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), rm2.data_ptr(), rv2.data_ptr(), nbt2.data_ptr(), save2.data_ptr(), save2[C:].data_ptr(), rep)
    pooled2 = torch.full((B, Ho, Wo, C), 7.0, dtype=torch.bfloat16, device=DEV)
    idx2 = torch.full((B, Ho, Wo, C), 77, dtype=torch.uint8, device=DEV)
    check(L().iswm_stem_pool_fwd(rawd.data_ptr(), Ct.byref(side), B, H, W, C, Ho, Wo, 1e-5, 0.1, pooled2.data_ptr(), idx2.data_ptr(), st()))
    assert torch.equal(pooled2, pooled1) and torch.equal(idx2, idx1)
    assert torch.equal(save2, save1) and torch.equal(rm2, rm1) and torch.equal(rv2, rv1) and nbt2.item() == 1


@pytest.mark.parametrize("B,C,Hi,Wi,ld", [(2, 256, 8, 8, 304), (1, 16, 5, 7, 24), (2, 64, 1, 3, 64), (1, 256, 32, 32, 256)])
def test_bilinear_up4_fast_path_is_bit_identical_to_the_generic_kernel(B, C, Hi, Wi, ld):
    """x4 upsampling (the decoder's interpolate, _deeplab.py:58): the 4x4-output-block kernel (9 loads per 16 stores) against the
    generic one-output-per-thread kernel - same weights, same expression: bit-equal, into a channel slice of a wider buffer."""
    import os
    x = rnd((B, C, Hi, Wi), 71)
    xd = nhwc(x).to(DEV)
    Ho, Wo = 4 * Hi, 4 * Wi
    outs = []
    for flag in ("1", "0"):
        os.environ["ISWM_BILINEAR_UP4"] = flag
        out = torch.full((B, Ho, Wo, ld), 3.0, dtype=torch.bfloat16, device=DEV)
        check(L().iswm_bilinear_fwd(xd.data_ptr(), C, B, Hi, Wi, C, Ho, Wo, out[..., ld - C:].data_ptr(), ld, st()))
        outs.append(out)
    os.environ.pop("ISWM_BILINEAR_UP4")
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    ref = F.interpolate(x.float(), size=(Ho, Wo), mode="bilinear", align_corners=False)
    close(nchw(outs[0][..., ld - C:]), ref, 1e-2, 1e-2)
    if ld > C:
        assert float(outs[0][..., :ld - C].float().min()) == 3.0
