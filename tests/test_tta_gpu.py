"""Test-time augmentation (multi-scale + flip) in the predict step: the input resize / mirror kernel against torch, the
multi-view predict epilogue against predict_epilogue (one view) and an fp64 evaluation of the view semantics (several
views), and predict_mask(scales=..., flip=True) against its torch composition on the bf16 and FP8 models."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from iswm_b200 import ops
from tests.test_model_gpu import build, report

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ----------------------------------------------------------------------------- resize + flip kernel
@pytest.mark.parametrize("shape,size", [((2, 3, 48, 64), (24, 32)), ((2, 3, 48, 64), (36, 48)), ((2, 3, 48, 64), (60, 80)),
                                        ((2, 3, 48, 64), (72, 96)), ((2, 3, 48, 64), (96, 128)), ((2, 3, 37, 53), (28, 40)),
                                        ((1, 3, 37, 53), (46, 66)), ((2, 3, 37, 53), (37, 53))])
@pytest.mark.parametrize("flip", [False, True])
def test_resize_flip_matches_torch(shape, size, flip):
    g = torch.Generator().manual_seed(shape[2] * 7 + size[1])
    x = (torch.randn(shape, generator=g) * 3).to(DEV)
    ref = F.interpolate(x, size=size, mode="bilinear", align_corners=False)
    ref = ref.flip(-1) if flip else ref
    got = ops.resize_flip_f32(x, size, flip)
    err = float((got - ref).abs().max())
    report("tta_resize_flip", shape=str(shape), size=str(size), flip=flip, max_abs_diff=err,
           share_bit_equal=float((got == ref).float().mean()))
    assert err <= 1e-6 * float(x.abs().max()), err
    if size == tuple(shape[2:]):
        assert torch.equal(got, x.flip(-1) if flip else x)          # scale 1: an exact copy
    # into a batch slice of a larger buffer, the rest untouched
    B = shape[0]
    buf = torch.full((B + 2, shape[1]) + tuple(size), float("nan"), device=DEV)
    ops.resize_flip_f32(x, size, flip, out=buf[1:B + 1])
    assert torch.equal(buf[1:B + 1], got) and bool(buf[0].isnan().all()) and bool(buf[B + 1].isnan().all())


# ----------------------------------------------------------------------------- multi-view epilogue
def _lowres(B, h, w, seed, scale=1.5):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((B, h, w, 2), generator=g) * scale).to(DEV)


def _labels(B, H, W, seed, dtype=torch.int64):
    g = torch.Generator().manual_seed(seed)
    y = (torch.rand((B, H, W), generator=g) < 0.3).long()
    y[torch.rand((B, H, W), generator=g) < 0.05] = 255
    return y.to(dtype).to(DEV)


def _counts(y, pred):
    t, p = y.long().cpu().numpy().ravel(), pred.long().cpu().numpy().ravel()
    ok = (t == 0) | (t == 1)
    return np.bincount(t[ok] * 2 + p[ok], minlength=4)


@pytest.mark.parametrize("B,h,w,up", [(2, 8, 12, 4), (1, 5, 7, 4), (3, 16, 33, 4), (1, 32, 32, 2)])
@pytest.mark.parametrize("mode,thr", [(1, 0.5), (1, 0.2), (0, 0.5)])
@pytest.mark.parametrize("ldt", [torch.int64, torch.uint8])
def test_single_view_equals_predict_epilogue(B, h, w, up, mode, thr, ldt):
    lo = _lowres(B, h, w, B * 100 + h)
    H, W = h * up, w * up
    y = _labels(B, H, W, 9, ldt)
    cm0, p0, c0 = ops.predict_epilogue(lo, H, W, y, mode=mode, threshold=thr)
    cm1, p1, c1 = ops.predict_tta_epilogue([(lo, (H, W), False)], H, W, y, mode=mode, threshold=thr)
    assert torch.equal(p0, p1) and torch.equal(c0, c1) and cm0.tolist() == cm1.tolist()
    _, p2, c2 = ops.predict_tta_epilogue([(lo, (H, W), False)], H, W, None, mode=mode, threshold=thr)
    assert torch.equal(p2, p0) and torch.equal(c2, c0)


def _p1_reference(views, Ho, Wo):
    """fp64 evaluation of the view semantics on the same low-resolution logits."""
    p = 0
    for lo, (Hv, Wv), f in views:
        v = F.interpolate(lo.double().cpu().permute(0, 3, 1, 2), size=(Hv, Wv), mode="bilinear", align_corners=False)
        if (Hv, Wv) != (Ho, Wo):
            v = F.interpolate(v, size=(Ho, Wo), mode="bilinear", align_corners=False)
        p = p + torch.softmax(v.flip(-1) if f else v, 1)
    return (p / len(views))[:, 1].numpy()


# (output size, [(low-res size, view size, flip)])
_MULTI = [
    ((40, 48), [((10, 12), (40, 48), False), ((10, 12), (40, 48), True)]),
    ((37, 50), [((7, 10), (28, 38), False), ((7, 10), (28, 38), True), ((10, 13), (37, 50), False), ((10, 13), (37, 50), True),
                ((12, 16), (46, 62), False), ((12, 16), (46, 62), True)]),
    ((64, 60), [((8, 8), (32, 30), True), ((16, 15), (64, 60), False), ((24, 23), (96, 90), True)]),
    ((33, 41), [((5, 6), (17, 21), False), ((7, 9), (25, 31), True), ((9, 11), (33, 41), True), ((11, 13), (41, 51), False),
                ((13, 16), (50, 62), True), ((15, 18), (58, 72), False), ((17, 21), (66, 82), True), ((9, 11), (33, 41), False)]),
]


@pytest.mark.parametrize("case", range(len(_MULTI)))
@pytest.mark.parametrize("ldt", [torch.int64, torch.uint8])
def test_multi_view_against_fp64_semantics(case, ldt):
    (Ho, Wo), spec = _MULTI[case]
    B = 2
    views = [(_lowres(B, hi, wi, 31 * i + case), hv, f) for i, ((hi, wi), hv, f) in enumerate(spec)]
    y = _labels(B, Ho, Wo, case, ldt)
    p1 = _p1_reference(views, Ho, Wo)
    worst = 0.0
    for thr in (0.2, 0.5, 0.7):
        cm, pred, conf = ops.predict_tta_epilogue(views, Ho, Wo, y, mode=1, threshold=thr)
        pn = pred.cpu().numpy()
        bad = (pn != (p1 > thr)) & (np.abs(p1 - thr) > 2e-6)
        assert not bad.any(), f"thr {thr}: {int(bad.sum())} decisions away from the threshold differ"
        d = np.abs(conf.cpu().numpy().astype(int) - (p1 * 255).astype(int))
        at_edge = np.abs(p1 * 255 - np.round(p1 * 255)) <= 255 * 2e-6
        assert d.max() <= 1 and not ((d == 1) & ~at_edge).any()
        assert cm[:4].cpu().tolist() == _counts(y, pred).tolist()
        worst = max(worst, float(np.abs(conf.cpu().numpy() / 255.0 - p1).max()))
    # mode 0: argmax of the averaged probabilities; conf is the mode-1 map only
    _, pred0, conf0 = ops.predict_tta_epilogue(views, Ho, Wo, None, mode=0)
    bad = (pred0.cpu().numpy() != (p1 > 0.5)) & (np.abs(p1 - 0.5) > 2e-6)
    assert not bad.any() and int(conf0.max()) == 0
    # the maps land in given batch slices
    pred_s = torch.full((B + 1, Ho, Wo), 7, dtype=torch.uint8, device=DEV)
    conf_s = torch.full((B + 1, Ho, Wo), 7, dtype=torch.uint8, device=DEV)
    ops.predict_tta_epilogue(views, Ho, Wo, None, mode=1, threshold=0.7, pred=pred_s[1:], conf=conf_s[1:])
    assert torch.equal(pred_s[1:], pred) and torch.equal(conf_s[1:], conf) and int(pred_s[0].min()) == int(conf_s[0].max()) == 7
    report("tta_epilogue_multi_view", case=case, views=len(views), conf_max_dev=worst)


def test_epilogue_limits():
    lo = _lowres(1, 4, 4, 0)
    with pytest.raises(RuntimeError):
        ops.predict_tta_epilogue([(torch.zeros((1, 4, 4, 3), device=DEV), (16, 16), False)], 16, 16)     # C != 2
    with pytest.raises(RuntimeError):
        ops.predict_tta_epilogue([(lo, (16, 16), i % 2 == 1) for i in range(9)], 16, 16)                # 9 views
    ops.predict_tta_epilogue([(lo, (16, 16), i % 2 == 1) for i in range(8)], 16, 16)                    # 8 is the cap


# ----------------------------------------------------------------------------- predict_mask end to end
SCALES = (0.75, 1.0, 1.25)


def _p1_composition(model, x, scales, flip):
    """The averaged foreground probability of the torch composition (what predict_mask(fused=False) thresholds)."""
    H, W = x.shape[-2:]
    p = 0
    for s in scales:
        Hs, Ws = (H, W) if s == 1.0 else (int(H * s + 0.5), int(W * s + 0.5))
        xs = x if s == 1.0 else F.interpolate(x, size=(Hs, Ws), mode="bilinear", align_corners=False)
        for f in ((False, True) if flip else (False,)):
            lv = model(xs.flip(-1) if f else xs)
            if (Hs, Ws) != (H, W):
                lv = F.interpolate(lv, size=(H, W), mode="bilinear", align_corners=False)
            p = p + torch.softmax(lv.flip(-1) if f else lv, 1)
    return (p[:, 1] / (len(scales) * (2 if flip else 1))).cpu().numpy()


def _check_against_composition(model, x, y, name):
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.predict import predict_mask
    m_f, m_r = StreamMetrics(2, device=DEV, shape_metrics=False), StreamMetrics(2, device=DEV, shape_metrics=False)
    pf, cf = predict_mask(model, x, 0.5, y, m_f, scales=SCALES, flip=True)
    pr, cr = predict_mask(model, x, 0.5, y, m_r, fused=False, scales=SCALES, flip=True)
    with torch.no_grad():
        p1 = _p1_composition(model, x, SCALES, True)
    assert np.array_equal(pr.cpu().numpy(), (p1 > 0.5).astype(np.uint8))       # the reference path is the composition
    dis = pf.cpu().numpy() != pr.cpu().numpy()
    agree = 1.0 - float(dis.mean())
    near = float(np.abs(p1[dis] - 0.5).max()) if dis.any() else 0.0
    conf_dev = int(np.abs(cf.cpu().numpy().astype(int) - cr.cpu().numpy().astype(int)).max())
    report(name, agreement=agree, disagree=int(dis.sum()), max_dist_to_threshold=near, conf_max_dev=conf_dev)
    assert agree >= 0.9999 and near <= 1e-3
    # the confusion matrices differ by exactly the disagreeing pixels
    t = y.long().cpu().numpy()
    ok = dis & ((t == 0) | (t == 1))
    moved = np.zeros(4, np.int64)
    np.add.at(moved, t[ok] * 2 + pf.cpu().numpy()[ok], 1)
    np.add.at(moved, t[ok] * 2 + pr.cpu().numpy()[ok], -1)
    assert (m_f._cm()[:4] - m_r._cm()[:4]).cpu().numpy().tolist() == moved.tolist()
    assert int(m_f._cm()[:4].sum()) == int(((t == 0) | (t == 1)).sum())
    return pf, cf


@pytest.mark.parametrize("backbone,os_", [("resnet50", 16), ("resnet101", 8)])
@pytest.mark.parametrize("shape", [(2, 160, 160), (1, 200, 232)])
def test_predict_mask_tta_against_torch_composition(backbone, os_, shape):
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.predict import predict_mask
    m, _ = build(backbone, os_)
    m.to(DEV).eval()
    B, H, W = shape
    g = torch.Generator(device=DEV).manual_seed(H + W)
    x = torch.randn((B, 3, H, W), device=DEV, generator=g)
    y = _labels(B, H, W, B, torch.uint8)
    _check_against_composition(m, x, y, f"tta_{backbone}_os{os_}_{B}x{H}x{W}")
    # the defaults are today's single-view path, bit for bit
    m0, m1 = StreamMetrics(2, device=DEV, shape_metrics=False), StreamMetrics(2, device=DEV, shape_metrics=False)
    p0, c0 = predict_mask(m, x, 0.5, y, m0)
    p1, c1 = predict_mask(m, x, 0.5, y, m1, scales=(1.0,), flip=False)
    assert torch.equal(p0, p1) and torch.equal(c0, c1) and torch.equal(m0._cm(), m1._cm())


def test_predict_mask_tta_fp8():
    from iswm_b200.quant import quantize_fp8
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn((2, 3, 160, 160), device=DEV, generator=g)
    qm = quantize_fp8(m, x)
    _check_against_composition(qm, x, _labels(2, 160, 160, 4, torch.int64), "tta_fp8_r50_os16_2x160x160")


def test_chunked_equals_unchunked(monkeypatch):
    """Batches whose views exceed the per-forward bound run in chunks (and a scale's two halves as separate forwards):
    the same maps and counts, bit for bit, as one forward per scale."""
    from iswm_b200 import predict
    from iswm_b200.metrics import StreamMetrics
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn((3, 3, 96, 96), device=DEV, generator=g)
    y = _labels(3, 96, 96, 6, torch.uint8)
    scales = (0.75, 1.0, 1.25)
    m0, m1 = StreamMetrics(2, device=DEV, shape_metrics=False), StreamMetrics(2, device=DEV, shape_metrics=False)
    p0, c0 = predict.predict_mask(m, x, 0.5, y, m0, scales=scales, flip=True)
    # 120^2 per image at s = 1.25: chunks of 2 + 1 images; in the first chunk the halves at s = 1.0 and 1.25 run as two
    # forwards, at s = 0.75 as one
    monkeypatch.setattr(predict, "MAX_FORWARD_PIXELS", 2 * 120 * 120)
    launches = []
    real = m.forward_lowres
    monkeypatch.setattr(m, "forward_lowres", lambda xv: (launches.append(tuple(xv.shape)), real(xv))[1])
    p1, c1 = predict.predict_mask(m, x, 0.5, y, m1, scales=scales, flip=True)
    assert launches == [(4, 3, 72, 72), (2, 3, 96, 96), (2, 3, 96, 96), (2, 3, 120, 120), (2, 3, 120, 120),
                        (2, 3, 72, 72), (2, 3, 96, 96), (2, 3, 120, 120)], launches
    assert torch.equal(p0, p1) and torch.equal(c0, c1) and torch.equal(m0._cm(), m1._cm())


def test_predict_mask_tta_rejects_bad_requests():
    from iswm_b200.network import modeling
    from iswm_b200.predict import predict_mask
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    x = torch.zeros((1, 3, 64, 64), device=DEV)
    for kw in (dict(scales=()), dict(scales=(0.0,)), dict(scales=(-1.0,)), dict(scales=(float("nan"),)),
               dict(scales=(float("inf"),)), dict(scales=(0.2,)), dict(scales=(0.5, 0.75, 1.0, 1.25, 1.5), flip=True)):
        with pytest.raises(ValueError):
            predict_mask(m, x, **kw)
    m3 = modeling.deeplabv3plus_resnet50(num_classes=3, output_stride=16, pretrained_backbone=False).to(DEV).eval()
    with pytest.raises(ValueError):
        predict_mask(m3, x, flip=True)


# ----------------------------------------------------------------------------- usefulness
def _band_tiles(n, size, seed):
    """Seeded synthetic tiles: thin bright oblique bands (foreground) on noise."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(size, dtype=torch.float32), torch.arange(size, dtype=torch.float32), indexing="ij")
    imgs, lbls = [], []
    for _ in range(n):
        lbl = torch.zeros(size, size, dtype=torch.bool)
        for _ in range(int(torch.randint(1, 4, (1,), generator=g))):
            ang = float(torch.rand(1, generator=g)) * 3.1416
            off = float(torch.rand(1, generator=g)) * size
            wid = 1.5 + 2.5 * float(torch.rand(1, generator=g))
            lbl |= ((xx - size / 2) * np.cos(ang) + (yy - size / 2) * np.sin(ang) + size / 2 - off).abs() < wid
        img = torch.randn(3, size, size, generator=g) * 0.6 + lbl.float() * 1.5
        imgs.append(img)
        lbls.append(lbl.long())
    return torch.stack(imgs), torch.stack(lbls)


def _flip_scale_jitter(x, y, g, lo=0.75, hi=1.25):
    """The training augmentation test-time augmentation presumes (the reference trains with random scale and horizontal
    flip): per tile a scale drawn from [lo, hi] (bilinear image, nearest labels), a 256^2 crop or a pad with ignored
    labels, and a flip with probability 1/2. Draws come from the CPU generator `g`."""
    xs, ys = [], []
    for i in range(x.shape[0]):
        S = int(256 * (lo + (hi - lo) * float(torch.rand(1, generator=g))) + 0.5)
        xi = F.interpolate(x[i:i + 1], size=(S, S), mode="bilinear", align_corners=False)
        yi = F.interpolate(y[i:i + 1, None].float(), size=(S, S), mode="nearest")[:, 0].long()
        if S >= 256:
            oy, ox = (int(torch.randint(0, S - 255, (1,), generator=g)) for _ in range(2))
            xi, yi = xi[..., oy:oy + 256, ox:ox + 256], yi[..., oy:oy + 256, ox:ox + 256]
        else:
            xi, yi = F.pad(xi, (0, 256 - S, 0, 256 - S)), F.pad(yi, (0, 256 - S, 0, 256 - S), value=255)
        if float(torch.rand(1, generator=g)) < 0.5:
            xi, yi = xi.flip(-1), yi.flip(-1)
        xs.append(xi)
        ys.append(yi)
    return torch.cat(xs).contiguous(), torch.cat(ys).contiguous()


def test_tta_is_useful_on_a_learnable_task():
    """Train briefly on synthetic band tiles with flip + scale jitter, then evaluate held-out tiles with one view and with
    (0.75, 1, 1.25) x flip. (Without scale jitter in training the 0.75 view is out of distribution for the thin bands and
    the three-scale set scores 0.004-0.017 foreground IoU below one view; DESIGN.md section 6.)"""
    from iswm_b200.graphs import GraphedTrainStep
    from iswm_b200.metrics.stream_metrics import StreamMetrics
    from iswm_b200.optim import FusedSGD
    from iswm_b200.predict import predict_mask
    from iswm_b200.utils.loss import CrossEntropyLoss
    torch.manual_seed(0)
    m, _ = build("resnet50", 16, seed=7)
    m.to(DEV).train()
    xs, ys = _band_tiles(64, 256, 1)
    xs, ys = xs.to(DEV), ys.to(DEV)
    crit = CrossEntropyLoss(weight=torch.tensor([1.0, 4.0])).to(DEV)
    opt = FusedSGD(m, lr=0.02, momentum=0.9, weight_decay=1e-4)
    step = GraphedTrainStep(m, crit, opt)
    g = torch.Generator().manual_seed(11)
    for i in range(150):
        j = (i * 8) % 64
        loss = step(*_flip_scale_jitter(xs[j:j + 8], ys[j:j + 8], g))
    m.eval()
    xt, yt = _band_tiles(16, 256, 2)
    xt, yt = xt.to(DEV), yt.to(DEV)
    res = {}
    for name, kw in (("single", {}), ("tta", dict(scales=SCALES, flip=True))):
        mt = StreamMetrics(2, device=DEV, shape_metrics=False)
        predict_mask(m, xt, 0.5, yt, mt, **kw)
        r = mt.get_results()
        res[name] = (r["Foreground IoU"], r["MIoU"])
    report("tta_usefulness", final_loss=float(loss), fg_iou_single=res["single"][0], fg_iou_tta=res["tta"][0],
           miou_single=res["single"][1], miou_tta=res["tta"][1])
    assert res["tta"][0] >= res["single"][0] - 0.01
