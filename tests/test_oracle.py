"""CPU suite (no GPU): pins the oracle (oracle/) against golden vectors produced by the real reference
(tests/golden/make_golden.py)."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import decode_oracle as D
from oracle import hourglass_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    z = np.load(os.path.join(GOLD, name), allow_pickle=False)
    return {k: z[k] for k in z.files}


def _sd(gold, prefix="sd/"):
    return {k[len(prefix):]: torch.from_numpy(v.copy()) for k, v in gold.items() if k.startswith(prefix)}


def _rel(a, b):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def train_gold():
    return _load("hg_s2f64_train.npz")


def test_oracle_forward_loss_grads_match_reference_golden(train_gold):
    torch.set_num_threads(4)
    g = train_gold
    sd = _sd(g)
    params = {k: v.requires_grad_(True) for k, v in sd.items() if v.dtype == torch.float32 and "running" not in k}
    sd.update(params)
    x = torch.from_numpy(g["x"])
    outs = O.hourglass_net(sd, x, num_stacks=2, num_blocks=1, training=True)
    for i, o in enumerate(outs):
        assert _rel(o.detach(), g["out%d" % i]) < 2e-5
    loss, pose, _ = O.fpd_loss(outs, torch.from_numpy(g["target"]), torch.from_numpy(g["target_weight"]))
    assert abs(loss.item() - float(g["loss"])) < 1e-6 * abs(float(g["loss"]))
    loss.backward()
    worst = 0.0
    for k, p in params.items():
        worst = max(worst, _rel(p.grad, g["grad/" + k]))
    assert worst < 2e-3, worst   # fp32 round-off through ~60 train-mode BN layers (see DESIGN.md on conditioning)
    # running statistics are updated like nn.BatchNorm2d does
    assert _rel(sd["bn1.running_mean"], g["after/bn1.running_mean"]) < 1e-6
    assert _rel(sd["fc.1.1.running_var"], g["after/fc.1.1.running_var"]) < 1e-6


def test_oracle_fpd_loss_matches_reference_golden(train_gold):
    torch.set_num_threads(4)
    g, f = train_gold, _load("hg_fpd.npz")
    sd = _sd(g)
    params = {k: v.requires_grad_(True) for k, v in sd.items() if v.dtype == torch.float32 and "running" not in k}
    sd.update(params)
    tsd = _sd(f, "tsd/")
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        tout = O.hourglass_net(tsd, x, num_stacks=1, training=False)[-1]
    assert _rel(tout, f["teacher_out"]) < 1e-5
    outs = O.hourglass_net(sd, x, num_stacks=2, training=True)
    loss, pose, kd = O.fpd_loss(outs, torch.from_numpy(g["target"]), torch.from_numpy(g["target_weight"]), tout,
                                float(f["alpha"]))
    for got, key in ((pose, "pose"), (kd, "kd"), (loss, "loss")):
        assert abs(got.item() - float(f[key])) < 2e-5 * abs(float(f[key])), key
    loss.backward()
    for k in [k[5:] for k in f if k.startswith("grad/")]:
        assert _rel(params[k].grad, f["grad/" + k]) < 2e-3, k
    norms = dict(zip(f["grad_names"].tolist(), f["grad_norms"].tolist()))
    for k, p in params.items():
        assert abs(p.grad.double().norm().item() - norms[k]) < 2e-3 * norms[k] + 1e-12, k


def test_joints_mse_closed_form_matches_reference_golden():
    g = _load("loss.npz")
    o, t, w = (torch.from_numpy(g[k]) for k in ("out", "target", "tw"))
    assert abs(O.joints_mse(o, t, w, True).item() - float(g["with_w"])) < 1e-6 * float(g["with_w"])
    assert abs(O.joints_mse(o, t, w, False).item() - float(g["without_w"])) < 1e-6 * float(g["without_w"])


def test_decode_and_nms_match_reference_golden():
    g = _load("decode.npz")
    preds, maxvals = D.get_max_preds(g["hm"])
    assert np.array_equal(preds, g["preds"]) and np.array_equal(maxvals, g["maxvals"])
    assert np.array_equal(D.flip_back(g["hm_flipped_raw"], D.MPII_FLIP_PAIRS), g["flip_back"])
    merged = D.flip_test_merge(g["hm"], g["hm_flipped_raw"], D.MPII_FLIP_PAIRS, True)
    assert np.array_equal(merged, g["merged"])
    mp, mv = D.get_max_preds(merged)
    assert np.array_equal(mp, g["merged_preds"]) and np.array_equal(mv, g["merged_maxvals"])
    assert D.nms(g["dets"], float(g["nms_thresh"])) == g["nms_keep"].tolist()
    assert D.nms(np.zeros((0, 5), np.float32), 0.5) == []


def test_oracle_matches_reference_module_golden():
    """The reference's hourglass module at its default initialisation (tests/golden/hg_s1f64_modes.npz), train and eval
    mode. The drop-in module draws the same weights from the same seed; their sums pin that."""
    import fpd_b200  # noqa: F401
    from fpd_b200.lib.models import hourglass as H
    torch.set_num_threads(4)
    g = _load("hg_s1f64_modes.npz")
    NS = types.SimpleNamespace
    cfg = NS(MODEL=NS(EXTRA=NS(NUM_FEATURES=64, NUM_STACKS=1, NUM_BLOCKS=1), NUM_JOINTS=16))
    torch.manual_seed(3)
    sd = H.get_pose_net(cfg, True).state_dict()
    x = torch.randn(2, 3, 64, 64)
    assert list(sd.keys()) == [str(k) for k in g["keys"]]
    sums = np.array([v.double().sum().item() for v in sd.values()])
    np.testing.assert_allclose(sums, g["sums"], rtol=1e-9, atol=1e-9)
    assert abs(x.double().sum().item() - float(g["x_sum"])) < 1e-9 * x.numel()
    with torch.no_grad():
        got = O.hourglass_net({k: v.clone() for k, v in sd.items()}, x, num_stacks=1, training=True)
        assert _rel(got[0], g["out_train"]) < 1e-5
        # eval mode with the running statistics the reference's train-mode pass left
        after = torch.from_numpy(g["running_after_train"])
        sd_eval, off = {}, 0
        for k, v in sd.items():
            if "running" in k:
                v = after[off:off + v.numel()].reshape(v.shape)
                off += v.numel()
            sd_eval[k] = v
        assert off == after.numel()
        got = O.hourglass_net(sd_eval, x, num_stacks=1, training=False)
        assert _rel(got[0], g["out_eval"]) < 1e-5


def test_dropin_module_state_dict_matches_reference_keys(train_gold):
    """Boundary (SURVEY 8b): same state_dict keys/shapes as the reference => strict=True checkpoint loading."""
    import fpd_b200  # noqa: F401
    from fpd_b200.lib.models import hourglass as H
    NS = types.SimpleNamespace
    cfg = NS(MODEL=NS(EXTRA=NS(NUM_FEATURES=64, NUM_STACKS=2, NUM_BLOCKS=1), NUM_JOINTS=16))
    net = H.get_pose_net(cfg, is_train=True)
    gold_sd = _sd(train_gold)
    own = net.state_dict()
    assert list(own.keys()) == list(gold_sd.keys())
    assert all(own[k].shape == gold_sd[k].shape for k in own)
    net.load_state_dict(gold_sd, strict=True)
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        net(torch.zeros(1, 3, 64, 64))


# ---------------------------------------------------------------------------------------------- HRNet
def _hr_cfg():
    class Cfg(dict):
        def __getattr__(self, k):
            try:
                return self[k]
            except KeyError:
                raise AttributeError(k)

    def wrap(d):
        return Cfg({k: wrap(v) for k, v in d.items()}) if isinstance(d, dict) else d

    def stage(nmod, chans):
        return dict(NUM_MODULES=nmod, NUM_BRANCHES=len(chans), BLOCK='BASIC', NUM_BLOCKS=[1] * len(chans),
                    NUM_CHANNELS=chans, FUSE_METHOD='SUM')
    return wrap(dict(MODEL=dict(NUM_JOINTS=17, INIT_WEIGHTS=False, PRETRAINED='', EXTRA=dict(
        PRETRAINED_LAYERS=['*'], FINAL_CONV_KERNEL=1, STAGE2=stage(1, [8, 16]), STAGE3=stage(2, [8, 16, 32]),
        STAGE4=stage(1, [8, 16, 32, 64])))))


def test_hrnet_oracle_matches_reference_golden():
    from oracle import hrnet_oracle as HO
    torch.set_num_threads(4)
    g = _load("hrnet_small.npz")
    sd = _sd(g)
    params = {k: v.requires_grad_(True) for k, v in sd.items() if v.dtype == torch.float32 and "running" not in k}
    sd.update(params)
    sda = HO.annotate_strides(sd)
    x = torch.from_numpy(g["x"])
    out = HO.hrnet(sda, x, training=True)
    assert _rel(out.detach(), g["out_train"]) < 2e-5
    loss = O.joints_mse(out, torch.from_numpy(g["target"]), torch.from_numpy(g["target_weight"]))
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * abs(float(g["loss"]))
    loss.backward()
    for k in [k[5:] for k in g if k.startswith("grad/")]:
        assert _rel(params[k].grad, g["grad/" + k]) < 2e-3, k
    sd_eval = HO.annotate_strides(_sd(g))
    with torch.no_grad():
        assert _rel(HO.hrnet(sd_eval, x, training=False), g["out_eval"]) < 2e-5


def test_hrnet_dropin_state_dict_matches_reference_keys():
    import fpd_b200  # noqa: F401
    from fpd_b200.lib.models import pose_hrnet as H
    g = _load("hrnet_small.npz")
    net = H.get_pose_net(_hr_cfg(), is_train=False)
    gold_sd = _sd(g)
    own = net.state_dict()
    assert list(own.keys()) == list(gold_sd.keys())
    assert all(own[k].shape == gold_sd[k].shape for k in own)
    net.load_state_dict(gold_sd, strict=True)
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        net(torch.zeros(1, 3, 64, 64))


# ---------------------------------------------------------------------------------------------- pose_resnet
RESNET_CASES = {"r18": (18, 17, (64, 32, 32), (4, 3, 2), 3, True), "r50": (50, 16, (128, 64, 64), (4, 4, 4), 1, False)}


def _resnet_cfg(tag):
    layers, J, filters, kernels, fk, bias = RESNET_CASES[tag]
    NS = types.SimpleNamespace
    return NS(MODEL=NS(NUM_JOINTS=J, INIT_WEIGHTS=False, PRETRAINED='', EXTRA=NS(
        NUM_LAYERS=layers, DECONV_WITH_BIAS=bias, NUM_DECONV_LAYERS=len(filters), NUM_DECONV_FILTERS=list(filters),
        NUM_DECONV_KERNELS=list(kernels), FINAL_CONV_KERNEL=fk)))


def _resnet_state(tag):
    """The golden run's weights, regenerated from the seed over the drop-in's own state_dict layout."""
    import fpd_b200  # noqa: F401
    from fpd_b200.lib.models import pose_resnet as R
    from oracle.resnet_oracle import synthetic_state
    net = R.get_pose_net(_resnet_cfg(tag), is_train=False)
    return net, synthetic_state({k: v.shape for k, v in net.state_dict().items()}, seed=7)


@pytest.mark.parametrize("tag", ["r18", "r50"])
def test_resnet_oracle_matches_reference_golden(tag):
    from oracle import resnet_oracle as RO
    torch.set_num_threads(4)
    g = {k[len(tag) + 1:]: v for k, v in _load("resnet_small.npz").items() if k.startswith(tag + "/")}
    net, sd = _resnet_state(tag)
    assert list(net.state_dict().keys()) == [str(k) for k in g["keys"]]       # the reference's keys, in its order
    params = {k: v.requires_grad_(True) for k, v in sd.items() if v.dtype == torch.float32 and "running" not in k}
    sd = dict(sd)
    sd.update(params)
    x = torch.from_numpy(g["x"])
    out = RO.resnet(sd, x, training=True)
    assert _rel(out.detach(), g["out_train"]) < 2e-5
    loss = O.joints_mse(out, torch.from_numpy(g["target"]), torch.from_numpy(g["target_weight"]))
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * abs(float(g["loss"]))
    loss.backward()
    assert _rel(sd["bn1.running_mean"], g["bn1.running_mean"]) < 1e-5       # train-mode side effect, momentum 0.1
    assert _rel(sd["bn1.running_var"], g["bn1.running_var"]) < 1e-5
    worst = 0.0
    for k, p in params.items():
        gd = p.grad.reshape(-1)
        ref = torch.from_numpy(g["grad/" + k])
        n = float(g["gnorm/" + k])
        # digest: leading entries (whole tensor when small) relative to the tensor's RMS, plus the L2 norm
        rms = max(n / gd.numel() ** 0.5, 1e-30)
        worst = max(worst, ((gd[:ref.numel()] - ref).abs().max() / rms).item())
        assert abs(gd.double().norm().item() - n) <= 2e-3 * n + 1e-12, k
    assert worst < 5e-3, worst
    _, sd_eval = _resnet_state(tag)
    with torch.no_grad():
        assert _rel(RO.resnet(sd_eval, x, training=False), g["out_eval"]) < 2e-5


def test_resnet_dropin_matches_reference_layout_and_refuses_cpu():
    net, sd = _resnet_state("r50")
    net.load_state_dict(sd, strict=True)
    assert type(net.deconv_layers[0]).__name__ == "ConvTranspose2d" and net.deconv_layers[0].bias is None
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        net(torch.zeros(1, 3, 64, 64))
    # every depth of the reference's resnet_spec has the same keys / shapes (tests/golden/resnet_layout.npz)
    g = _load("resnet_layout.npz")
    from fpd_b200.lib.models import pose_resnet as M
    assert {k: list(v[1]) for k, v in M.resnet_spec.items()} == {
        int(k.split("/")[1]): g[k].tolist() for k in g if k.startswith("resnet_spec/")}

    def layout(tag, cfg):
        sd = M.get_pose_net(cfg, is_train=False).state_dict()
        assert list(sd.keys()) == [str(k) for k in g[tag + "/keys"]], tag
        assert [",".join(str(n) for n in v.shape) for v in sd.values()] == [str(s) for s in g[tag + "/shapes"]], tag
    for tag in ("r18", "r50"):
        layout(tag, _resnet_cfg(tag))
    for depth in (34, 101, 152):          # the shipped d256x3 head on the remaining depths of resnet_spec
        cfg = _resnet_cfg("r50")
        cfg.MODEL.EXTRA.NUM_LAYERS = depth
        cfg.MODEL.EXTRA.NUM_DECONV_FILTERS = [256, 256, 256]
        layout("d%d" % depth, cfg)
    # init_weights without a checkpoint (pose_resnet.py:229-247): N(0, 0.001) convs / deconvs, unit BatchNorm
    cfg = _resnet_cfg("r18")
    cfg.MODEL.INIT_WEIGHTS = True
    net = M.get_pose_net(cfg, is_train=True)
    assert 5e-4 < net.layer2[0].conv1.weight.std().item() < 2e-3
    assert 5e-4 < net.deconv_layers[0].weight.std().item() < 2e-3 and float(net.deconv_layers[0].bias.detach().abs().max()) == 0.0
    assert torch.equal(net.deconv_layers[1].weight, torch.ones_like(net.deconv_layers[1].weight))


@pytest.mark.parametrize("k,pad,outpad", [(4, 1, 0), (3, 1, 1), (2, 0, 0)])
def test_transposed_conv_as_3x3_conv_plus_depth_to_space(k, pad, outpad):
    """The identity Engine.deconv / csrc/elementwise.cu deconv_weight_map_kernel rest on, in plain torch:
    ConvTranspose2d(k, stride 2, pad) == depth_to_space(conv3x3(x, W3)), W3[(rh,rw,co), ci, th, tw] =
    Wd[ci, co, rh + pad - 2 (th - 1), rw + pad - 2 (tw - 1)] (zero outside the kernel); and the gradient map back."""
    g = torch.Generator().manual_seed(k)
    Cin, Cout, H, W = 5, 3, 6, 4
    x = torch.randn(2, Cin, H, W, generator=g, dtype=torch.float64)
    wd = torch.randn(Cin, Cout, k, k, generator=g, dtype=torch.float64)
    ref = torch.nn.functional.conv_transpose2d(x, wd, stride=2, padding=pad, output_padding=outpad)
    w3 = torch.zeros(2, 2, Cout, Cin, 3, 3, dtype=torch.float64)
    where = {}
    for rh in range(2):
        for rw in range(2):
            for th in range(3):
                for tw in range(3):
                    kh, kw = rh + pad - 2 * (th - 1), rw + pad - 2 * (tw - 1)
                    if 0 <= kh < k and 0 <= kw < k:
                        w3[rh, rw, :, :, th, tw] = wd[:, :, kh, kw].t()
                        assert (kh, kw) not in where          # every deconv tap lands in exactly one place
                        where[(kh, kw)] = (rh, rw, th, tw)
    assert len(where) == k * k
    y = torch.nn.functional.conv2d(x, w3.reshape(4 * Cout, Cin, 3, 3), padding=1)          # [B, (rh,rw,co), H, W]
    out = y.reshape(2, 2, 2, Cout, H, W).permute(0, 3, 4, 1, 5, 2).reshape(2, Cout, 2 * H, 2 * W)
    assert ref.shape == out.shape and (ref - out).abs().max() < 1e-12
    # the kernel's closed form for the way back: rh = (kh - pad) & 1, th = (rh + pad - kh) / 2 + 1
    for (kh, kw), (rh, rw, th, tw) in where.items():
        assert rh == (kh - pad) & 1 and rw == (kw - pad) & 1
        assert th == (rh + pad - kh) // 2 + 1 and tw == (rw + pad - kw) // 2 + 1
        assert (rh + pad - kh) % 2 == 0 and (rw + pad - kw) % 2 == 0


# --------------------------------------------------------------------------------------------------------------------
# decode tail (tests/golden/decode2.npz: the reference's get_final_preds / accuracy / oks_nms / generate_target)
# --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def decode2():
    return _load("decode2.npz")


@pytest.mark.parametrize("tag", ["sq", "rect"])
def test_oracle_final_preds_and_accuracy_match_reference_golden(decode2, tag):
    z = decode2
    for pp in (1, 0):
        preds, maxvals = D.get_final_preds(bool(pp), z[tag + "/hm"].copy(), z[tag + "/center"], z[tag + "/scale"])
        assert np.abs(preds - z["%s/preds_pp%d" % (tag, pp)]).max() < 1e-9
        assert np.array_equal(maxvals, z["%s/maxvals_pp%d" % (tag, pp)])
    acc, avg, cnt, pred = D.accuracy(z[tag + "/acc_out"], z[tag + "/acc_target"])
    assert np.array_equal(acc, z[tag + "/acc"]) and avg == float(z[tag + "/avg_acc"]) and cnt == int(z[tag + "/cnt"])
    assert np.array_equal(pred, z[tag + "/acc_pred"])


def test_closed_form_transform_preds_matches_reference_golden(decode2):
    """lib.core.inference.transform_preds restates the reference's float32 corner points + cv2's 3-point solve."""
    import fpd_b200  # noqa: F401
    from fpd_b200.lib.core.inference import transform_preds
    z = decode2
    for tag in ("sq", "rect"):
        hm = z[tag + "/hm"]
        coords, _ = D.get_max_preds(hm)
        W, H = hm.shape[3], hm.shape[2]
        for i in range(hm.shape[0]):
            got = transform_preds(coords[i], z[tag + "/center"][i], z[tag + "/scale"][i], [W, H])
            ref = z[tag + "/preds_pp0"][i]
            # get_final_preds stores the result into the float32 `preds` array (inference.py:71-77): bit-exact after the cast
            assert np.array_equal(got.astype(np.float32), ref), (tag, i, np.abs(got - ref).max())


def test_oracle_oks_nms_and_rescore_match_reference_golden(decode2):
    z = decode2
    for tag in ("oks_a", "oks_b", "oks_c"):
        r = D.rescore(z[tag + "/kpts"], z[tag + "/box_score"], float(z["oks/in_vis_thre"]))
        assert np.array_equal(r, z[tag + "/rescored"])
        assert D.oks_nms(z[tag + "/kpts"], z[tag + "/area"], r, float(z["oks/oks_thre"])) == list(z[tag + "/keep"])
        assert D.oks_nms(z[tag + "/kpts"], z[tag + "/area"], r, 0.5, None, 0.3) == list(z[tag + "/keep_vis"])


def test_oracle_generate_target_matches_reference_golden(decode2):
    z = decode2
    jw = np.array([1., 1., 1., 1., 1., 1., 1., 1.2, 1.2, 1.5, 1.5, 1., 1., 1.2, 1.2, 1.5, 1.5], np.float32).reshape(17, 1)
    for tag, img, hm, w in (("tgt_sq", (256, 256), (64, 64), None), ("tgt_rect", (192, 256), (48, 64), jw)):
        for i in range(z[tag + "/joints"].shape[0]):
            t, tw = D.generate_target(z[tag + "/joints"][i], z[tag + "/joints_vis"][i], img, hm, 2, w)
            assert np.array_equal(t, z[tag + "/target"][i]) and np.array_equal(tw, z[tag + "/target_weight"][i])


def test_host_oks_helpers_match_reference_golden(decode2):
    """lib.nms.nms.oks_iou / soft_oks_nms are host numpy in the drop-in too: same numbers as the oracle's oks_iou."""
    import fpd_b200  # noqa: F401
    from fpd_b200.lib.nms import nms as M
    z = decode2
    k = z["oks_a/kpts"].reshape(40, -1)
    a = z["oks_a/area"]
    got = M.oks_iou(k[3], k[4:], a[3], a[4:], None, 0.3)
    ref = D.oks_iou(k[3], k[4:], a[3], a[4:], None, 0.3)
    assert np.array_equal(got, ref)
    db = [{"keypoints": z["oks_a/kpts"][i], "area": a[i], "score": z["oks_a/rescored"][i]} for i in range(40)]
    keep = M.soft_oks_nms(db, 0.9)
    assert len(keep) == 20 and keep[0] == int(np.argmax(z["oks_a/rescored"]))
