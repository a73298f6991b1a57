"""End-to-end parity of the CUDA DeepLabV3+ against (a) golden vectors produced by the REAL
reference code, (b) the fp32 torch oracle and (c) the precision-matched (bf16-storage) oracle, both
run on the host CPU with identical weights.

Stated tolerances (north_star asks for "a stated bf16 tolerance, e.g. <= 1e-2 on logits, <= 1e-3 on
the scalar loss vs the fp32 reference"):
  * eval mode (BatchNorm folded) against the REFERENCE's golden logits: relative L2 <= 1e-2 (north_star's figure) and
    worst logit within 2e-2 of the logit range for ResNet-50 at OS16 / OS8 (measured on B200, r2b: 7.5e-3 / 6.0e-3 /
    8.4e-3 at 320x320 with every ASPP tap in-image); ResNet-101 OS8 <= 1.5e-2 (measured 1.0e-2: 104 convolutions of bf16
    storage, 2^-9 per rounding, random walk). Odd-size cases on other weights: within 1.25x the precision-matched
    CPU oracle's own distance from fp32, never below the 1e-2 gate. Every test prints what it measured (PARITY lines).
  * train mode (batch statistics): bf16 rounding of the pre-BN conv outputs is amplified by every
    batch normalisation (noise relative to |x| becomes noise relative to |x - mean|), so ANY bf16
    implementation drifts several percent from fp32 on these random-weight nets — the
    precision-matched torch oracle itself is 6-10 % away. The engine must be no further from fp32
    than 1.5x that oracle (+0.5 %), i.e. at the bf16 noise floor; scalar loss <= 1e-2 relative.
    The loss KERNEL on identical logits is held to 1e-5 (tests/test_loss_metric_gpu.py), and every
    unit's forward and backward is checked to one bf16 rounding on the engine's own tensors in
    tests/test_unit_replay_gpu.py — that test, not this one, is the precise gradient gate.
  * gradients here (a wiring check; ReLU-mask flips turn a forward drift eps into a gradient drift
    ~sqrt(eps), so per-tensor agreement is loose by nature): whole-model gradient cosine >= 0.5 and
    every conv weight tensor's cosine >= 0.3 against the precision-matched oracle (a missing, doubled
    or sign-flipped gradient path gives ~0 or negative); train-mode scalar loss <= 1e-2 relative."""
import os

import numpy as np
import pytest
import torch

from iswm_b200 import _lib
from iswm_b200.network import modeling
from iswm_b200.utils.loss import CrossEntropyLoss
from oracle import torch_model as TM
from oracle.gen_golden import seeded_state_dict, synth_labels

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def rel_max(a, b):
    a, b = torch.as_tensor(a).float(), torch.as_tensor(b).float()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def rel_l2(a, b):
    a, b = torch.as_tensor(a).float().flatten(), torch.as_tensor(b).float().flatten()
    return float((a - b).norm() / (b.norm() + 1e-20))


def report(name, **vals):
    """Every parity test prints what it MEASURED (pytest -rP / -s shows it) and appends it to gpurun_out/parity_measured.txt
    when that directory exists (copied to profiles/ per round)."""
    line = "PARITY " + name + " " + " ".join(f"{k}={v:.4g}" if isinstance(v, float) else f"{k}={v}" for k, v in vals.items())
    print(line)
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(d):
        with open(os.path.join(d, "parity_measured.txt"), "a") as f:
            f.write(line + "\n")


def logits_close(got, ref, name="logits", l2_max=2e-2, mx_max=4e-2):
    l2, mx = rel_l2(got, ref), rel_max(got, ref)
    report(name, rel_l2=l2, max_over_range=mx, gate_l2=l2_max, gate_max=mx_max)
    assert l2 <= l2_max and mx <= mx_max, f"{name}: rel L2 {l2:.4g} (<={l2_max}), max/range {mx:.4g} (<={mx_max})"


def train_reference(backbone, os_, sd, x, y, w):
    """fp32 oracle and precision-matched oracle train steps on the host CPU."""
    from oracle import torch_model_q as TQ
    res = {}
    for kind in ("fp32", "matched"):
        o = TM.oracle_model(backbone, 2, os_)
        o.load_state_dict(sd)
        o.train()
        for mod in o.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
        logits, loss = (TM.train_step if kind == "fp32" else TQ.train_step_q)(o, x, y, w)
        res[kind] = (logits, loss, {n: p.grad.clone() for n, p in o.named_parameters()}, dict(o.named_buffers()))
    return res


def check_train_against_noise_floor(logits, loss, ref):
    f32_logits, f32_loss = ref["fp32"][0], ref["fp32"][1]
    floor = rel_l2(ref["matched"][0], f32_logits)
    mine = rel_l2(logits, f32_logits)
    report("train_vs_fp32", logits_rel_l2=mine, matched_oracle_floor=floor, loss=float(loss), loss_fp32=f32_loss.item(),
           loss_rel=abs(loss - f32_loss.item()) / abs(f32_loss.item()), loss_floor_rel=abs(ref["matched"][1].item() - f32_loss.item()) / abs(f32_loss.item()))
    assert mine <= 1.5 * floor + 5e-3, f"train logits {mine:.4g} from fp32; bf16 noise floor (matched oracle) {floor:.4g}"
    # scalar loss: the batch-2 golden case normalises the ASPP pooling branch over TWO samples, so bf16
    # rounding is amplified by 1/sqrt(eps); the precision-matched oracle's own distance from fp32 is the floor
    lfloor = abs(ref["matched"][1].item() - f32_loss.item())
    assert abs(loss - f32_loss.item()) <= 1.5 * lfloor + 5e-3 * abs(f32_loss.item()), (loss, f32_loss.item(), lfloor)


def cosine(a, b):
    a, b = torch.as_tensor(a).float().flatten(), torch.as_tensor(b).float().flatten()
    return float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-30))


def build(backbone, os_, seed=1234):
    ctor = modeling.deeplabv3plus_resnet50 if backbone == "resnet50" else modeling.deeplabv3plus_resnet101
    m = ctor(num_classes=2, output_stride=os_, pretrained_backbone=False)
    sd = seeded_state_dict(m.state_dict(), seed)
    m.load_state_dict(sd)
    return m, sd


def test_r50_os16_eval_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "model_r50_os16.npz"))
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    out = m(torch.tensor(g["x"]).to(DEV))
    assert out.dtype == torch.float32 and tuple(out.shape) == g["eval_logits"].shape
    logits_close(out.cpu(), g["eval_logits"], "r50_os16_eval_vs_reference_golden", 1e-2, 2e-2)


def test_r50_os16_eval_loss_vs_reference(golden_dir):
    """Scalar loss of the whole bf16 network vs the fp32 reference on the reference's own eval logits.
    north_star asks <= 1e-3 relative; the criterion kernel meets that on identical logits (test_wce_* in
    test_loss_metric_gpu.py, <= 1e-5), but 63 layers of bf16 activations move the logits of a RANDOM-weight
    network by ~1e-2, which moves this loss by ~4e-3 even for the CPU precision-matched oracle. The gate is
    therefore: within 1.5x the matched oracle's own distance from fp32 (+2e-3), and never above 1e-2."""
    from oracle import oracle_np as O
    from oracle import torch_model_q as TQ
    g = np.load(os.path.join(golden_dir, "model_r50_os16.npz"))
    m, sd = build("resnet50", 16)
    m.to(DEV).eval()
    y, w = torch.tensor(g["y"]), torch.tensor(g["w"])
    out = m(torch.tensor(g["x"]).to(DEV))
    loss = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)(out, y.to(DEV)).item()
    ref_loss, _ = O.weighted_ce(g["eval_logits"], g["y"], g["w"])
    o = TM.oracle_model("resnet50", 2, 16)
    o.load_state_dict(sd)
    o.eval()
    with torch.no_grad():
        floor_loss, _ = O.weighted_ce(TQ.forward_q(o, torch.tensor(g["x"]), False).numpy(), g["y"], g["w"])
    floor = abs(floor_loss - ref_loss)
    assert abs(loss - ref_loss) <= 1.5 * floor + 2e-3 * abs(ref_loss), (loss, ref_loss, floor_loss)
    assert abs(loss - ref_loss) <= 1e-2 * abs(ref_loss), (loss, ref_loss)
    # the criterion itself, on the reference's logits: <= 1e-5
    ref_t = torch.tensor(g["eval_logits"]).to(DEV)
    l2 = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)(ref_t, y.to(DEV)).item()
    assert abs(l2 - ref_loss) <= 1e-5 * abs(ref_loss), (l2, ref_loss)


def test_r101_os8_eval_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "model_r101_os8.npz"))
    m, _ = build("resnet101", 8)
    m.to(DEV).eval()
    out = m(torch.tensor(g["x"]).to(DEV))
    logits_close(out.cpu(), g["eval_logits"], "r101_os8_eval_vs_reference_golden", 1.5e-2, 3e-2)   # 104 convolutions deep: measured 1.0e-2


def test_r50_os8_eval_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "model_r50_os8.npz"))
    m, _ = build("resnet50", 8)
    m.to(DEV).eval()
    out = m(torch.tensor(g["x"]).to(DEV))
    logits_close(out.cpu(), g["eval_logits"], "r50_os8_eval_vs_reference_golden", 1e-2, 2e-2)


def test_r50_os8_320_eval_matches_reference_golden(golden_dir):
    """ResNet-50 at output stride 8 on a 320 x 320 tile: the 40 x 40 feature map is larger than every ASPP rate
    (12 / 24 / 36, network/modeling.py:27-33; layer3 d=2, layer4 d=4), so EVERY tap of the dilated branches reads pixels inside
    the image - a wrong tap offset at d=24 / d=36 cannot hide behind the zero padding as it can in the small fixtures.
    Golden: oracle/gen_golden_r2.py (the real reference); full-resolution map additionally vs the fp32 oracle."""
    from oracle.gen_golden_r2 import golden_input
    g = np.load(os.path.join(golden_dir, "model_r50_os8_320.npz"))
    x = golden_input()
    assert abs(float(x.double().sum()) - float(g["x_sum"])) < 1e-6 and np.array_equal(x.flatten()[:16].numpy(), g["x_head"])
    m, sd = build("resnet50", 8)
    m.to(DEV).eval()
    out = m(x.to(DEV)).cpu()
    logits_close(out[:, :, ::4, ::4], g["logits_s4"], "r50_os8_320_eval_vs_reference_golden(stride-4 lattice)", 1e-2, 2e-2)
    got = out.flatten(2)[0][:, torch.tensor(g["pos"])]
    logits_close(got, g["logits_at_pos"], "r50_os8_320_eval_vs_reference_golden(4096 samples)", 1e-2, 2e-2)
    o = TM.oracle_model("resnet50", 2, 8)
    o.load_state_dict(sd)
    o.eval()
    with torch.no_grad():
        ref = o(x)
    assert rel_l2(ref[:, :, ::4, ::4], g["logits_s4"]) <= 1e-4          # the oracle is pinned to the reference here too
    logits_close(out, ref, "r50_os8_320_eval_vs_fp32_oracle(full map)", 1e-2, 2e-2)


def test_r50_os16_train_step_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "model_r50_os16.npz"))
    m, sd = build("resnet50", 16)
    x, y, w = torch.tensor(g["x"]), torch.tensor(g["y"]), torch.tensor(g["w"])
    ref = train_reference("resnet50", 16, sd, x, y, w)
    # the fp32 oracle is itself pinned to the reference's own output
    assert rel_l2(ref["fp32"][0], g["train_logits"]) <= 1e-3
    m.to(DEV).train()
    m.engine().dropout_p = 0.0                      # the golden run disables Dropout (gen_golden.py)
    crit = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)
    logits = m(x.to(DEV))
    loss = crit(logits, y.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    check_train_against_noise_floor(logits.detach().cpu(), loss.item(), ref)
    assert abs(loss.item() - float(g["train_loss"])) <= 2.5e-2 * float(g["train_loss"])
    sdm = m.state_dict()
    np.testing.assert_allclose(sdm["backbone.bn1.running_mean"].cpu().numpy(), g["bn1_running_mean_after"], rtol=2e-2, atol=2e-3)
    np.testing.assert_allclose(sdm["backbone.bn1.running_var"].cpu().numpy(), g["bn1_running_var_after"], rtol=2e-2, atol=2e-3)
    assert int(sdm["backbone.bn1.num_batches_tracked"]) == 1


@pytest.mark.parametrize("backbone,os_,B,H,W", [("resnet50", 16, 4, 96, 96), ("resnet50", 16, 3, 72, 104), ("resnet50", 8, 4, 64, 64),
                                                 ("resnet50", 16, 4, 97, 65), ("resnet101", 8, 4, 64, 64)])   # odd sizes; R101-OS8 (cfg3). Batch >= 3: the pooled ASPP
# branch normalises over B samples, and with B = 2 its BatchNorm output is sign(a - b) per channel - any rounding flips it
def test_train_step_full_gradients_vs_oracle(backbone, os_, B, H, W):
    m, sd = build(backbone, os_, seed=77)
    g = torch.Generator().manual_seed(5)
    x = torch.randn((B, 3, H, W), generator=g)
    y = synth_labels((B, H, W), seed=6, fg=0.2, ign=0.05)
    w = torch.tensor([1.0, 3.0])
    ref = train_reference(backbone, os_, sd, x, y, w)
    m.to(DEV).train()
    m.engine().dropout_p = 0.0
    crit = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)
    logits = m(x.to(DEV))
    loss = crit(logits, y.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    check_train_against_noise_floor(logits.detach().cpu(), loss.item(), ref)
    ref_grads = ref["matched"][2]
    worst = []
    mine_all, ref_all = [], []
    for name, p in m.named_parameters():
        rg = ref_grads[name]
        c = cosine(p.grad.cpu(), rg)
        mine_all.append(p.grad.cpu().flatten())
        ref_all.append(rg.flatten())
        if rg.dim() == 4 and rg.norm() > 1e-6 and c < 0.3:      # conv weights: large tensors, stable cosine
            worst.append((name, round(c, 4)))
    assert not worst, f"{len(worst)} gradient tensors with cosine < 0.3 vs the matched oracle, first: {worst[:12]}"
    whole = cosine(torch.cat(mine_all), torch.cat(ref_all))
    assert whole >= 0.5, f"whole-model gradient cosine {whole:.4f} < 0.5"
    ob = ref["fp32"][3]
    for name, b in m.named_buffers():
        if name.endswith("running_var") or name.endswith("running_mean"):
            a, r = b.cpu(), ob[name]
            assert rel_l2(a, r) <= 5e-2, (name, rel_l2(a, r))


@pytest.mark.parametrize("H,W", [(200, 200), (65, 49), (513, 513)])
def test_eval_odd_sizes_vs_oracle(H, W):
    m, sd = build("resnet50", 16, seed=3)
    oracle = TM.oracle_model("resnet50", 2, 16)
    oracle.load_state_dict(sd)
    oracle.eval()
    g = torch.Generator().manual_seed(9)
    x = torch.randn((1, 3, H, W), generator=g)
    with torch.no_grad():
        ref = oracle(x)
    m.to(DEV).eval()
    out = m(x.to(DEV))
    # seed-3 weights, unlike the golden seed, leave these logits with a small range: the precision-matched CPU oracle (bf16
    # storage at the engine's rounding points) is itself ~1.3e-2 from fp32 here, reported next to the measurement
    from oracle import torch_model_q as TQ
    with torch.no_grad():
        floor = rel_l2(TQ.forward_q(oracle, x, False), ref)
    report(f"eval_odd_{H}x{W}_matched_oracle_floor", rel_l2=floor)
    logits_close(out.cpu(), ref, f"eval_odd_{H}x{W}_vs_fp32_oracle", max(1e-2, 1.25 * floor), 4e-2)


def test_state_dict_roundtrip_and_dataparallel_prefix():
    m, sd = build("resnet50", 16, seed=4)
    m2 = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False)
    m2.load_state_dict({k: v.clone() for k, v in m.state_dict().items()})
    wrapped = {("module." + k): v for k, v in m.state_dict().items()}            # predict.py:83-85 strips this
    m2.load_state_dict({k.replace("module.", ""): v for k, v in wrapped.items()})
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)


def test_train_two_steps_with_torch_optimizer_changes_output():
    m, _ = build("resnet50", 16, seed=8)
    m.to(DEV).train()
    opt = torch.optim.SGD(m.parameters(), lr=1e-2, momentum=0.9, nesterov=True)   # train.py:424-431
    crit = CrossEntropyLoss(weight=torch.tensor([1.0, 7.0])).to(DEV)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((2, 3, 64, 64), generator=g).to(DEV)
    y = synth_labels((2, 64, 64), seed=2, fg=0.3).to(DEV)
    losses = []
    for _ in range(4):
        logits = m(x)
        loss = crit(logits, y)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses


def test_predict_mask_matches_reference_semantics(golden_dir):
    """predict.py:262-278 on our logits: class map and uint8 confidence bit-exact vs the numpy oracle applied to the SAME
    logits, confusion counts equal to StreamMetrics._fast_hist of that class map."""
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.predict import predict_mask
    from oracle import oracle_np as O
    g = np.load(os.path.join(golden_dir, "model_r50_os16.npz"))
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    x, y = torch.tensor(g["x"]).to(DEV), torch.tensor(g["y"]).to(DEV)
    sm = StreamMetrics(2, device=DEV)
    pred, conf = predict_mask(m, x, threshold=0.5, labels=y, metrics=sm)
    logits = m(x).cpu().numpy()
    ref_pred, ref_conf = O.threshold_pred(logits, 0.5)
    assert pred.dtype == torch.uint8 and conf.dtype == torch.uint8
    assert np.array_equal(pred.cpu().numpy(), ref_pred.astype(np.uint8))
    assert np.abs(conf.cpu().numpy().astype(np.int32) - ref_conf.astype(np.int32)).max() <= 1     # uint8(p*255) at a rounding edge
    ref_cm = O.fast_hist(g["y"].reshape(-1), ref_pred.reshape(-1), 2)
    assert sm.confusion_matrix.astype(np.int64).tolist() == ref_cm.tolist()


def test_forward_branch_overlap_changes_nothing():
    """The low-level projection and the pooled ASPP branch run on the side stream under the main chain
    (Engine._fwd_fork): the forward must stay BIT-identical to the in-line order (train and eval), the gradients equal
    up to the weight-gradient atomics noise."""
    m, sd = build("resnet50", 16, seed=21)
    m.to(DEV)
    g = torch.Generator().manual_seed(8)
    x = torch.randn((4, 3, 96, 80), generator=g).to(DEV)
    y = synth_labels((4, 96, 80), seed=9, fg=0.2, ign=0.05).to(DEV)
    crit = CrossEntropyLoss(weight=torch.tensor([1.0, 3.0])).to(DEV)
    eng = m.engine()
    eng.dropout_p = 0.1
    outs = {}
    for overlap in (False, True, True):
        eng.fwd_overlap = overlap
        eng.step = 0
        eng._step_dev = None                       # same Dropout mask in every run
        for p in m.parameters():
            p.grad = None
        bufs = [b.detach().clone() for b in m.buffers()]
        m.train()
        logits = m(x)
        loss = crit(logits, y)
        loss.backward()
        m.eval()
        with torch.no_grad():
            ev = m(x).clone()
        torch.cuda.synchronize()
        outs.setdefault(overlap, []).append((logits.detach().clone(), eng.flat_g.clone(), ev))
        with torch.no_grad():
            for b, v in zip(m.buffers(), bufs):    # BatchNorm running statistics back to the start
                b.copy_(v)
    (l0, g0, e0), = outs[False]
    for l1, g1, e1 in outs[True]:
        assert torch.equal(l0, l1) and torch.equal(e0, e1)
        assert rel_l2(g1, g0) <= 1e-5


def test_batched_unpack_equals_per_layer_and_accumulates():
    """k x k weight gradients unpacked in one launch at the end of the sweep == the per-layer unpack (to the atomics
    noise of wgrad), and a second backward without zeroing accumulates (.grad semantics of train.py:1047-1048)."""
    m, sd = build("resnet50", 16, seed=31)
    m.to(DEV).train()
    g = torch.Generator().manual_seed(4)
    x = torch.randn((3, 3, 64, 80), generator=g).to(DEV)
    y = synth_labels((3, 64, 80), seed=5, fg=0.2, ign=0.05).to(DEV)
    crit = CrossEntropyLoss(weight=torch.tensor([1.0, 3.0])).to(DEV)
    eng = m.engine()
    eng.dropout_p = 0.0
    grads = {}
    for mode in (False, True):
        eng.batch_unpack = mode
        bufs = [b.detach().clone() for b in m.buffers()]
        for p in m.parameters():
            p.grad = None
        crit(m(x), y).backward()
        g1 = eng.flat_g.clone()
        crit(m(x), y).backward()                      # no zero_grad in between: accumulates
        grads[mode] = (g1, eng.flat_g.clone())
        with torch.no_grad():
            for b, v in zip(m.buffers(), bufs):
                b.copy_(v)
    assert rel_l2(grads[True][0], grads[False][0]) <= 1e-5
    assert rel_l2(grads[True][1], 2 * grads[True][0]) <= 1e-3     # second pass: running statistics moved nothing in train mode
    assert rel_l2(grads[True][1], grads[False][1]) <= 1e-5


def test_fused_aspp_backward_matches_the_four_launch_form():
    """ASPP backward as one K-concatenated data-gradient GEMM (iswm_aspp_bwd, the default) against the four separate
    launches (engine.aspp_fused_bwd = False): same loss bit for bit (the forward is
    untouched); the fused form accumulates the four branches in fp32 where the unfused one rounds to bf16 three times, so the
    parameter gradients agree to bf16 noise."""
    x = torch.randn((4, 3, 96, 96), generator=torch.Generator().manual_seed(5))
    y = synth_labels((4, 96, 96), seed=6, fg=0.2, ign=0.05)
    w = torch.tensor([1.0, 3.0])
    res = []
    for fused in (True, False):
        m, _ = build("resnet50", 16, seed=77)
        m.to(DEV).train()
        eng = m.engine()
        eng.dropout_p = 0.0
        eng.aspp_fused_bwd = fused
        crit = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)
        loss = crit(m(x.to(DEV)), y.to(DEV))
        loss.backward()
        torch.cuda.synchronize()
        assert bool(eng._aspp_cat_slot()) == fused
        res.append((float(loss.detach()), eng.flat_g.clone(), {n: p.grad.clone() for n, p in m.named_parameters()}))
    assert res[0][0] == res[1][0]
    rel = rel_l2(res[0][1], res[1][1])
    cos = cosine(res[0][1], res[1][1])
    report("fused_aspp_bwd_vs_unfused", flat_grad_rel_l2=rel, cosine=cos)
    assert rel <= 3e-2 and cos >= 0.999
    # the ASPP branches' own weight gradients do not depend on the data-gradient path at all
    for n in ("classifier.aspp.convs.0.0.weight", "classifier.aspp.convs.2.0.weight"):
        assert rel_l2(res[0][2][n], res[1][2][n]) <= 1e-5


def test_masked_identity_gradient_equals_the_materialised_form():
    """Backward of non-first bottleneck blocks (resnet.py:99-120): the identity path's gradient dz = dout . relu_mask folded
    into conv1's data-gradient epilogue (ISWM_EPI_RES_MASK, the default) against bn_bwd_apply writing dz as a tensor that the
    epilogue reads back. Same arithmetic (the mask is 0/1, dz is dout's own bf16 value), so every activation gradient is
    bit-identical; parameter gradients differ only by the weight-gradient kernels' fp32 atomics order."""
    x = torch.randn((4, 3, 96, 96), generator=torch.Generator().manual_seed(15))
    y = synth_labels((4, 96, 96), seed=16, fg=0.2, ign=0.05)
    w = torch.tensor([1.0, 3.0])
    res = []
    for masked in (True, False):
        m, _ = build("resnet50", 16, seed=78)
        m.to(DEV).train()
        eng = m.engine()
        eng.dropout_p = 0.0
        eng.masked_identity = masked
        crit = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)
        loss = crit(m(x.to(DEV)), y.to(DEV))
        loss.backward()
        torch.cuda.synchronize()
        res.append((float(loss.detach()), eng.flat_g.clone(), m.backbone.bn1.weight.grad.clone()))
    assert res[0][0] == res[1][0]
    rel = rel_l2(res[0][1], res[1][1])
    report("masked_identity_vs_materialised", flat_grad_rel_l2=rel)
    assert rel <= 1e-5
    assert rel_l2(res[0][2], res[1][2]) <= 1e-5          # the very last gradient of the sweep (stem BatchNorm weight)


def test_dual_batchnorm_blocks_match_the_two_kernel_form():
    """First block of every ResNet layer (resnet.py:176-186): closing BatchNorm + downsample BatchNorm as one kernel per pass
    (csrc/bn_dual.cu, the default) against the separate kernels. The fused forward adds the shortcut in fp32 instead of
    rounding it to bf16 first; at this size a train-mode forward amplifies ANY bf16-level change to ~8 % of the logits (the
    pooled ASPP branch normalises over 4 samples: see train_vs_fp32 / matched_oracle_floor), so the two forms are compared
    through their distance to the fp32 oracle, which must not grow. The kernels themselves are checked against torch
    autograd in tests/test_glue_gpu.py::test_dual_batchnorm_of_a_downsample_block_against_torch."""
    x = torch.randn((4, 3, 96, 96), generator=torch.Generator().manual_seed(35))
    y = synth_labels((4, 96, 96), seed=36, fg=0.2, ign=0.05)
    w = torch.tensor([1.0, 3.0])
    _, sd = build("resnet50", 16, seed=80)
    ref = train_reference("resnet50", 16, sd, x, y, w)["fp32"]
    ref_flat = torch.cat([ref[2][n].flatten() for n, _ in build("resnet50", 16, seed=80)[0].named_parameters()])
    res = []
    for dual in (True, False):
        m, _ = build("resnet50", 16, seed=80)
        m.to(DEV).train()
        eng = m.engine()
        eng.dropout_p = 0.0
        eng.dual_bn = dual
        crit = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)
        n0 = _lib.launch_count()
        logits = m(x.to(DEV))
        loss = crit(logits, y.to(DEV))
        loss.backward()
        torch.cuda.synchronize()
        flat = torch.cat([p.grad.flatten() for _, p in m.named_parameters()]).cpu()
        res.append(dict(loss=float(loss.detach()), launches=_lib.launch_count() - n0, d_logits=rel_l2(logits.detach().cpu(), ref[0]),
                        cos=cosine(flat, ref_flat), d_loss=abs(float(loss.detach()) - ref[1].item()) / abs(ref[1].item()),
                        bufs={k: v.clone() for k, v in m.state_dict().items() if "downsample.1.running" in k or "num_batches" in k}))
    d, s_ = res
    report("dual_bn_vs_two_kernels", logits_to_fp32_dual=d["d_logits"], logits_to_fp32_separate=s_["d_logits"], loss_rel_dual=d["d_loss"],
           loss_rel_separate=s_["d_loss"], grad_cos_to_fp32_dual=d["cos"], grad_cos_to_fp32_separate=s_["cos"],
           launches_dual=d["launches"], launches_separate=s_["launches"])
    assert s_["launches"] - d["launches"] == 12           # 4 blocks x (apply + reduce + bwd apply) fewer launches
    assert d["d_logits"] <= 1.25 * s_["d_logits"] + 5e-3
    assert d["d_loss"] <= 1.5 * s_["d_loss"] + 5e-3
    assert d["cos"] >= s_["cos"] - 0.05
    for k in d["bufs"]:                                   # running statistics / step counters of the downsample BatchNorms keep moving
        a, b = d["bufs"][k].float(), s_["bufs"][k].float()
        assert rel_l2(a, b) <= 2e-2, (k, rel_l2(a, b))


def test_fused_stem_tail_forward_matches_the_separate_kernels():
    """Stem BatchNorm + ReLU + maxpool as one forward pass (csrc/stem_pool.cu, the default) against bn_train_apply + maxpool_fwd:
    the forward is bit-identical (same logits, same loss); both forms run the same three backward kernels."""
    x = torch.randn((4, 3, 96, 96), generator=torch.Generator().manual_seed(45))
    y = synth_labels((4, 96, 96), seed=46, fg=0.2, ign=0.05)
    w = torch.tensor([1.0, 3.0])
    res = []
    for fused in (True, False):
        m, _ = build("resnet50", 16, seed=81)
        m.to(DEV).train()
        eng = m.engine()
        eng.dropout_p = 0.0
        eng.stem_pool = fused
        crit = CrossEntropyLoss(weight=w, ignore_index=255).to(DEV)
        n0 = _lib.launch_count()
        logits = m(x.to(DEV))
        loss = crit(logits, y.to(DEV))
        loss.backward()
        torch.cuda.synchronize()
        res.append((float(loss.detach()), eng.flat_g.clone(), _lib.launch_count() - n0, logits.detach().clone(),
                    m.backbone.bn1.running_var.clone(), m.backbone.conv1.weight.grad.clone(), m.backbone.bn1.weight.grad.clone()))
    assert torch.equal(res[0][3], res[1][3]) and res[0][0] == res[1][0]
    assert torch.equal(res[0][4], res[1][4])
    assert res[1][2] - res[0][2] == 1                    # (apply + maxpool) -> 1
    rel = rel_l2(res[0][1], res[1][1])
    report("fused_stem_tail_vs_separate", flat_grad_rel_l2=rel, stem_weight_grad_rel_l2=rel_l2(res[0][5], res[1][5]),
           bn1_weight_grad_rel_l2=rel_l2(res[0][6], res[1][6]))
    assert rel <= 1e-4 and rel_l2(res[0][5], res[1][5]) <= 2e-3 and rel_l2(res[0][6], res[1][6]) <= 1e-4
