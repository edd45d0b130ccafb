"""Generate the golden vectors under tests/golden/ by running the REAL reference
(/root/reference, read-only) on seeded synthetic inputs. Run in the build container only:

    python tests/golden/make_golden.py [decode2 | resnet | hg_modes | resnet_layout]

The reference has no tests / fixtures of its own (SURVEY.md section 4), so these vectors -- outputs of its
own lib/models/hourglass.py, lib/core/loss.py, lib/core/inference.py, lib/utils/transforms.py and
lib/nms/nms.py -- are what pins the oracle (tests/test_oracle.py) and, through it, the CUDA path.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))
NS = types.SimpleNamespace


def load(name, rel):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def cfg(f, s, j=16):
    return NS(MODEL=NS(EXTRA=NS(NUM_FEATURES=f, NUM_STACKS=s, NUM_BLOCKS=1), NUM_JOINTS=j))


def gaussian_targets(rng, B, J, h, w):
    """Reference-style targets (lib/dataset/JointsDataset.py:251-284): sigma=2, 13x13 patch, peak 1."""
    t = np.zeros((B, J, h, w), np.float32)
    size = 13
    xs = np.arange(size, dtype=np.float32)
    g = np.exp(-((xs[None] - 6) ** 2 + (xs[:, None] - 6) ** 2) / (2 * 2.0 ** 2))
    for b in range(B):
        for j in range(J):
            mx, my = rng.randint(0, w), rng.randint(0, h)
            ul = (mx - 6, my - 6)
            gx = (max(0, -ul[0]), min(ul[0] + size, w) - ul[0])
            gy = (max(0, -ul[1]), min(ul[1] + size, h) - ul[1])
            ix = (max(0, ul[0]), min(ul[0] + size, w))
            iy = (max(0, ul[1]), min(ul[1] + size, h))
            t[b, j, iy[0]:iy[1], ix[0]:ix[1]] = g[gy[0]:gy[1], gx[0]:gx[1]]
    return t


def main_decode2():
    """Section 6: the host-side decode tail the drop-in replaces -- get_final_preds (inference.py:49-79, POST_PROCESS on
    and off, non-trivial centre / scale, via the reference's cv2 affine), accuracy (evaluate.py:41-71), and OKS-NMS with
    the rescoring loop of lib/dataset/coco.py:334-369 (nms.py:75-124). Own RNG: does not disturb the other vectors."""
    sys.path.insert(0, os.path.join(REF, "lib"))
    from core.inference import get_final_preds, get_max_preds   # noqa: E402
    from core.evaluate import accuracy                           # noqa: E402
    src = open(os.path.join(REF, "lib/nms/nms.py")).read().replace("from .cpu_nms import cpu_nms", "").replace(
        "from .gpu_nms import gpu_nms", "")
    nms_ns = {}
    exec(compile(src, "ref_nms.py", "exec"), nms_ns)
    rng = np.random.RandomState(7)
    save = {}
    for tag, (B, J, h, w) in (("sq", (3, 16, 64, 64)), ("rect", (3, 17, 64, 48))):
        # peaky maps: low noise + a Gaussian bump per joint (some at the border, one all-negative, one flat)
        hm = (rng.randn(B, J, h, w) * 0.05).astype(np.float32)
        hm += gaussian_targets(rng, B, J, h, w) * rng.uniform(0.3, 1.0, (B, J, 1, 1)).astype(np.float32)
        hm[0, 0] = -0.5
        hm[0, 1] = 0.25
        hm[1, 2, 0, 0] = 3.0          # arg-max in the corner: no quarter-pixel nudge
        hm[1, 3, h - 1, w - 1] = 3.0
        hm[2, 4, 1, 1] = 3.0          # px == 1: excluded by the strict 1 < px test
        hm[2, 5, 2, 2] = 3.0          # first position that is nudged
        center = np.stack([rng.uniform(100, 900, B), rng.uniform(100, 700, B)], 1).astype(np.float32)
        sc = rng.uniform(0.6, 3.2, B).astype(np.float32)
        scale = np.stack([sc, sc * (1.0 if tag == "sq" else 1.25)], 1).astype(np.float32)
        save[tag + "/hm"] = hm
        save[tag + "/center"] = center
        save[tag + "/scale"] = scale
        for pp in (True, False):
            cfgt = NS(TEST=NS(POST_PROCESS=pp))
            preds, maxvals = get_final_preds(cfgt, hm.copy(), center, scale)
            save["%s/preds_pp%d" % (tag, int(pp))] = preds
            save["%s/maxvals_pp%d" % (tag, int(pp))] = maxvals
        # accuracy(): output = hm, target = clean Gaussians (some joints with target arg-max <= 1 -> ignored)
        tgt = gaussian_targets(rng, B, J, h, w)
        tgt[0, 2] = 0.0
        tgt[1, 3] = 0.0
        tgt[1, 3, 0, 5] = 1.0
        tgt[:, 6] = 0.0               # a joint ignored in every sample: acc = -1, not counted
        sig = rng.choice([0.1, 0.3, 0.45], size=(B, J, 1, 1)).astype(np.float32)
        out = tgt + (rng.randn(B, J, h, w).astype(np.float32) * sig)
        acc, avg, cnt, pred = accuracy(out, tgt)
        save[tag + "/acc_out"] = out
        save[tag + "/acc_target"] = tgt
        save[tag + "/acc"] = acc
        save[tag + "/avg_acc"] = np.float64(avg)
        save[tag + "/cnt"] = np.int64(cnt)
        save[tag + "/acc_pred"] = pred
    # OKS-NMS + rescoring (coco.py:343-369): persons of one image
    for tag, n in (("oks_a", 40), ("oks_b", 7), ("oks_c", 1)):
        base = rng.uniform(50, 400, (max(n // 4, 1), 17, 2))
        kp = np.zeros((n, 17, 3), np.float64)
        for i in range(n):
            kp[i, :, :2] = base[i % base.shape[0]] + rng.randn(17, 2) * rng.choice([1.0, 6.0, 40.0])
            kp[i, :, 2] = rng.uniform(0.0, 1.0, 17)
        area = rng.uniform(2000, 40000, n)
        box_score = rng.uniform(0.1, 1.0, n)
        in_vis_thre, oks_thre = 0.2, 0.9
        db = []
        for i in range(n):
            ks, vn = 0.0, 0
            for j in range(17):
                if kp[i, j, 2] > in_vis_thre:
                    ks += kp[i, j, 2]
                    vn += 1
            if vn:
                ks /= vn
            db.append({"keypoints": kp[i], "area": area[i], "score": ks * box_score[i]})
        keep = nms_ns["oks_nms"](db, oks_thre)
        save[tag + "/kpts"] = kp
        save[tag + "/area"] = area
        save[tag + "/box_score"] = box_score
        save[tag + "/rescored"] = np.array([d["score"] for d in db])
        save[tag + "/keep"] = np.array(keep, np.int64)
        save[tag + "/keep_vis"] = np.array(nms_ns["oks_nms"](db, 0.5, None, 0.3), np.int64)
    # Gaussian target generation (lib/dataset/JointsDataset.py:233-289), called unbound on a stub `self`
    JointsDataset = load("ref_joints_dataset", "lib/dataset/JointsDataset.py").JointsDataset   # dataset/__init__ needs json_tricks
    for tag, (J, img, hms, diffw) in (("tgt_sq", (16, (256, 256), (64, 64), False)),
                                      ("tgt_rect", (17, (192, 256), (48, 64), True))):
        stub = NS(num_joints=J, target_type="gaussian", heatmap_size=np.array(hms), image_size=np.array(img), sigma=2,
                  use_different_joints_weight=diffw,
                  joints_weight=np.array([1., 1., 1., 1., 1., 1., 1., 1.2, 1.2, 1.5, 1.5, 1., 1., 1.2, 1.2, 1.5, 1.5],
                                         np.float32).reshape(17, 1)[:J])
        n = 12
        joints = np.zeros((n, J, 3), np.float32)
        joints[:, :, 0] = rng.uniform(-20, img[0] + 20, (n, J))     # some centres off the image
        joints[:, :, 1] = rng.uniform(-20, img[1] + 20, (n, J))
        joints[0, 0, :2] = (-40.0, 10.0)                            # Gaussian entirely out of bounds -> weight 0
        joints[0, 1, :2] = (img[0] + 39.9, 30.0)
        joints[0, 2, :2] = (1.9, 2.1)                               # rounding of mu = int(x / stride + 0.5)
        joints[0, 3, :2] = (img[0] - 0.1, img[1] - 0.1)
        vis = np.zeros((n, J, 3), np.float32)
        vis[:, :, 0] = vis[:, :, 1] = (rng.rand(n, J) > 0.25).astype(np.float32)
        tg, tw = [], []
        for i in range(n):
            t_, w_ = JointsDataset.generate_target(stub, joints[i], vis[i])
            tg.append(t_)
            tw.append(w_)
        save[tag + "/joints"] = joints
        save[tag + "/joints_vis"] = vis
        save[tag + "/target"] = np.stack(tg)
        save[tag + "/target_weight"] = np.stack(tw)
    save["oks/in_vis_thre"] = np.float64(0.2)
    save["oks/oks_thre"] = np.float64(0.9)
    np.savez_compressed(os.path.join(OUT, "decode2.npz"), **save)
    print("decode2.npz", os.path.getsize(os.path.join(OUT, "decode2.npz")))


RESNET_CASES = {   # tag: (NUM_LAYERS, joints, deconv filters, deconv kernels, FINAL_CONV_KERNEL, DECONV_WITH_BIAS)
    "r18": (18, 17, (64, 32, 32), (4, 3, 2), 3, True),       # BasicBlock; every head geometry of pose_resnet.py:159-174
    "r50": (50, 16, (128, 64, 64), (4, 4, 4), 1, False),     # Bottleneck; the shipped configs' geometry
}


def resnet_cfg(layers, j, filters, kernels, fk, bias):
    return NS(MODEL=NS(NUM_JOINTS=j, INIT_WEIGHTS=False, PRETRAINED='', EXTRA=NS(
        NUM_LAYERS=layers, DECONV_WITH_BIAS=bias, NUM_DECONV_LAYERS=len(filters), NUM_DECONV_FILTERS=list(filters),
        NUM_DECONV_KERNELS=list(kernels), FINAL_CONV_KERNEL=fk)))


def grad_digest(g):
    """Whole tensor when small, else its first 512 entries + L2 norm (ResNet gradients are too large to commit)."""
    g = g.detach().reshape(-1)
    return (g.numpy() if g.numel() <= 2048 else g[:512].numpy()), np.float64(g.double().norm().item())


def main_resnet():
    """Section 7: the reference's lib/models/pose_resnet.py (ResNet-18 and -50 bodies, all three deconv geometries) on
    oracle.resnet_oracle.synthetic_state() weights -- regenerated from the seed by the tests, the networks are too large to
    commit -- 64x64 inputs, train-mode forward + JointsMSELoss + backward, and the eval-mode forward."""
    sys.path.insert(0, os.path.join(OUT, "..", ".."))
    from oracle.resnet_oracle import synthetic_state
    torch.set_num_threads(4)
    R = load("ref_pose_resnet", "lib/models/pose_resnet.py")
    L = load("ref_loss", "lib/core/loss.py")
    crit = L.JointsMSELoss(use_target_weight=True)
    save = {}
    for tag, (layers, J, filters, kernels, fk, bias) in RESNET_CASES.items():
        net = R.get_pose_net(resnet_cfg(layers, J, filters, kernels, fk, bias), is_train=False)
        sd0 = synthetic_state({k: v.shape for k, v in net.state_dict().items()}, seed=7)
        net.load_state_dict(sd0, strict=True)
        rng = np.random.RandomState(11)
        g = torch.Generator().manual_seed(5)
        x = torch.randn(2, 3, 64, 64, generator=g)
        target = torch.from_numpy(gaussian_targets(rng, 2, J, 16, 16))
        tw = torch.from_numpy((rng.rand(2, J, 1) > 0.2).astype(np.float32))
        net.train()
        out = net(x)
        loss = crit(out, target, tw)
        loss.backward()
        save[tag + "/x"], save[tag + "/target"], save[tag + "/target_weight"] = x.numpy(), target.numpy(), tw.numpy()
        save[tag + "/out_train"] = out.detach().numpy()
        save[tag + "/loss"] = np.float64(loss.item())
        for k, p_ in net.named_parameters():
            d, n = grad_digest(p_.grad)
            save["%s/grad/%s" % (tag, k)] = d
            save["%s/gnorm/%s" % (tag, k)] = n
        save[tag + "/bn1.running_mean"] = net.bn1.running_mean.numpy().copy()
        save[tag + "/bn1.running_var"] = net.bn1.running_var.numpy().copy()
        net.load_state_dict(sd0)
        net.eval()
        with torch.no_grad():
            save[tag + "/out_eval"] = net(x).numpy()
        save[tag + "/keys"] = np.array(list(net.state_dict().keys()))
    np.savez_compressed(os.path.join(OUT, "resnet_small.npz"), **save)
    print("resnet_small.npz", os.path.getsize(os.path.join(OUT, "resnet_small.npz")))


def main_hg_modes():
    """Section 8: the reference's lib/models/hourglass.py, s=1 f=64 with its default initialisation under
    torch.manual_seed(3), then x = torch.randn(2, 3, 64, 64): the first output in train mode, and in eval mode with the
    running statistics that train-mode pass left (stored too, concatenated in state_dict order). The weights and x are
    regenerated from the seed by the test -- the network is too large to commit -- and pinned by their float64 sums."""
    torch.set_num_threads(4)
    hg = load("ref_hourglass", "lib/models/hourglass.py")
    torch.manual_seed(3)
    net = hg.get_pose_net(cfg(64, 1), True)
    x = torch.randn(2, 3, 64, 64)
    sd = net.state_dict()
    save = {"x_sum": np.float64(x.double().sum().item()), "keys": np.array(list(sd.keys())),
            "sums": np.array([v.double().sum().item() for v in sd.values()], np.float64)}
    with torch.no_grad():
        net.train()
        save["out_train"] = net(x)[0].numpy()
        save["running_after_train"] = torch.cat([v.reshape(-1) for k, v in net.state_dict().items()
                                                 if "running" in k]).numpy()
        net.eval()
        save["out_eval"] = net(x)[0].numpy()
    np.savez_compressed(os.path.join(OUT, "hg_s1f64_modes.npz"), **save)
    print("hg_s1f64_modes.npz", os.path.getsize(os.path.join(OUT, "hg_s1f64_modes.npz")))


def main_resnet_layout():
    """Section 9: the state_dict layout (keys in order, shapes) of the reference's pose_resnet for both RESNET_CASES and,
    with the shipped 3 x 256-filter 4x4 deconv head, for the remaining depths of its resnet_spec; and the block counts of
    resnet_spec itself."""
    R = load("ref_pose_resnet", "lib/models/pose_resnet.py")
    save = {}
    for depth, (_, blocks) in R.resnet_spec.items():
        save["resnet_spec/%d" % depth] = np.array(blocks, np.int64)
    cases = dict(RESNET_CASES)
    for depth in (34, 101, 152):
        cases["d%d" % depth] = (depth, 16, (256, 256, 256), (4, 4, 4), 1, False)
    for tag, case in cases.items():
        sd = R.get_pose_net(resnet_cfg(*case), is_train=False).state_dict()
        save[tag + "/keys"] = np.array(list(sd.keys()))
        save[tag + "/shapes"] = np.array([",".join(str(n) for n in v.shape) for v in sd.values()])
    np.savez_compressed(os.path.join(OUT, "resnet_layout.npz"), **save)
    print("resnet_layout.npz", os.path.getsize(os.path.join(OUT, "resnet_layout.npz")))


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "decode2":
        return main_decode2()
    if len(sys.argv) > 1 and sys.argv[1] == "resnet":
        return main_resnet()
    if len(sys.argv) > 1 and sys.argv[1] == "hg_modes":
        return main_hg_modes()
    if len(sys.argv) > 1 and sys.argv[1] == "resnet_layout":
        return main_resnet_layout()
    torch.set_num_threads(4)
    hg = load("ref_hourglass", "lib/models/hourglass.py")
    loss_mod = load("ref_loss", "lib/core/loss.py")
    sys.path.insert(0, os.path.join(REF, "lib"))
    from core.inference import get_max_preds           # noqa: E402
    from utils.transforms import flip_back             # noqa: E402
    # nms.py imports two Cython extensions that are not built here; stub them (pure-numpy `nms` is what we use)
    sys.modules.setdefault("cpu_nms", types.SimpleNamespace(cpu_nms=None))
    sys.modules.setdefault("gpu_nms", types.SimpleNamespace(gpu_nms=None))
    src = open(os.path.join(REF, "lib/nms/nms.py")).read().replace("from .cpu_nms import cpu_nms", "").replace(
        "from .gpu_nms import gpu_nms", "")
    nms_ns = {}
    exec(compile(src, "ref_nms.py", "exec"), nms_ns)

    rng = np.random.RandomState(0)
    B, H, W, J = 2, 128, 128, 16  # 32x32 heat-maps: deepest hourglass level is 2x2 (well-conditioned BN)
    h, w = H // 4, W // 4

    # ---- 1. hourglass s=2 f=64, train mode, plain MSE (function.train semantics, function.py:44-63) ----
    torch.manual_seed(0)
    net = hg.get_pose_net(cfg(64, 2), True)
    net.train()
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    x = torch.randn(B, 3, H, W)
    target = torch.from_numpy(gaussian_targets(rng, B, J, h, w))
    tw = torch.from_numpy((rng.rand(B, J, 1) > 0.2).astype(np.float32))
    crit = loss_mod.JointsMSELoss(use_target_weight=True)
    outs = net(x)
    loss = crit(outs[0], target, tw)
    for o in outs[1:]:
        loss = loss + crit(o, target, tw)
    net.zero_grad()
    loss.backward()
    sd1 = net.state_dict()
    save = {"x": x.numpy(), "target": target.numpy(), "target_weight": tw.numpy(), "loss": np.float32(loss.item())}
    for i, o in enumerate(outs):
        save["out%d" % i] = o.detach().numpy()
    for k, v in sd0.items():
        save["sd/" + k] = v.numpy()
    for k, p in net.named_parameters():
        save["grad/" + k] = p.grad.numpy()
    for k in ("bn1.running_mean", "bn1.running_var", "hg.1.hg.0.3.0.bn2.running_mean", "fc.1.1.running_var",
              "bn1.num_batches_tracked"):
        save["after/" + k] = sd1[k].numpy()
    np.savez_compressed(os.path.join(OUT, "hg_s2f64_train.npz"), **save)

    # ---- 2. FPD: same student, frozen teacher s=1 f=64 in eval mode (function.py:119-134), alpha=0.5 ----
    torch.manual_seed(1)
    tnet = hg.get_pose_net(cfg(64, 1), False)
    # give the teacher non-trivial running statistics
    for m in tnet.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0, 0.1)
            m.running_var.uniform_(0.5, 1.5)
    tnet.eval()
    net.load_state_dict(sd0)
    net.train()
    net.zero_grad()
    outs = net(x)
    with torch.no_grad():
        tout = tnet(x)[-1]
    pose = crit(outs[0], target, tw)
    kd = crit(outs[0], tout, tw)
    for o in outs[1:]:
        pose = pose + crit(o, target, tw)
        kd = kd + crit(o, tout, tw)
    alpha = 0.5
    total = (1 - alpha) * pose + alpha * kd
    total.backward()
    save = {"alpha": np.float32(alpha), "pose": np.float32(pose.item()), "kd": np.float32(kd.item()),
            "loss": np.float32(total.item()), "teacher_out": tout.numpy()}
    for k, v in tnet.state_dict().items():
        save["tsd/" + k] = v.numpy()
    names, norms = [], []
    for k, p in net.named_parameters():
        names.append(k)
        norms.append(float(p.grad.double().norm()))
    save["grad_names"] = np.array(names)
    save["grad_norms"] = np.array(norms, np.float64)
    for k in ("conv1.weight", "layer2.0.conv2.weight", "hg.0.hg.0.3.0.conv2.weight", "hg.1.hg.3.0.0.bn1.weight",
              "fc.0.0.weight", "score.1.bias", "score_.0.weight", "fc_.0.bias"):
        save["grad/" + k] = dict(net.named_parameters())[k].grad.numpy()
    np.savez_compressed(os.path.join(OUT, "hg_fpd.npz"), **save)

    # ---- 3. JointsMSELoss module on its own (loss.py:21-39) ----
    o = torch.randn(3, J, 8, 8)
    t = torch.rand(3, J, 8, 8)
    w3 = torch.rand(3, J, 1)
    np.savez_compressed(os.path.join(OUT, "loss.npz"), out=o.numpy(), target=t.numpy(), tw=w3.numpy(),
                        with_w=np.float32(loss_mod.JointsMSELoss(True)(o, t, w3).item()),
                        without_w=np.float32(loss_mod.JointsMSELoss(False)(o, t, w3).item()))

    # ---- 4. decode: get_max_preds / flip_back (+shift, average as in function.py:224-240) / nms ----
    hm = rng.randn(3, J, 16, 12).astype(np.float32)
    hm[0, 0] = 0.5           # ties: first index wins
    hm[0, 1] = -1.0          # max <= 0 -> preds zeroed
    hf = rng.randn(3, J, 16, 12).astype(np.float32)
    pairs = [[0, 5], [1, 4], [2, 3], [10, 15], [11, 14], [12, 13]]  # lib/dataset/mpii.py:32
    preds, maxvals = get_max_preds(hm)
    fb = flip_back(hf.copy(), pairs)
    shifted = fb.copy()
    shifted[:, :, :, 1:] = shifted.copy()[:, :, :, 0:-1]
    merged = (hm + shifted) * np.float32(0.5)
    mp, mv = get_max_preds(merged)
    n = 300
    x1 = rng.uniform(0, 200, n); y1 = rng.uniform(0, 200, n)
    dets = np.stack([x1, y1, x1 + rng.uniform(8, 128, n), y1 + rng.uniform(8, 128, n), rng.uniform(0, 1, n)],
                    1).astype(np.float32)
    keep = np.array(nms_ns["nms"](dets, 0.6), np.int64)
    np.savez_compressed(os.path.join(OUT, "decode.npz"), hm=hm, hm_flipped_raw=hf, flip_back=fb, merged=merged,
                        preds=preds, maxvals=maxvals, merged_preds=mp, merged_maxvals=mv, dets=dets, nms_keep=keep,
                        nms_thresh=np.float32(0.6))
    # ---- 5. HRNet (lib/models/pose_hrnet.py) small config: all structural cases (bottleneck layer1, transitions,
    #         2/3/4-branch modules, up/down fuse chains, single-output last module), J=17, 128x96 input ----
    import warnings
    warnings.simplefilter("ignore")
    hr = load("ref_pose_hrnet", "lib/models/pose_hrnet.py")

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
    hcfg = wrap(dict(MODEL=dict(NUM_JOINTS=17, INIT_WEIGHTS=False, PRETRAINED='', EXTRA=dict(
        PRETRAINED_LAYERS=['*'], FINAL_CONV_KERNEL=1, STAGE2=stage(1, [8, 16]), STAGE3=stage(2, [8, 16, 32]),
        STAGE4=stage(1, [8, 16, 32, 64])))))
    torch.manual_seed(5)
    hnet = hr.get_pose_net(hcfg, False)
    hnet.train()
    hsd0 = {k: v.clone() for k, v in hnet.state_dict().items()}
    hx = torch.randn(2, 3, 128, 96)
    htarget = torch.from_numpy(gaussian_targets(rng, 2, 17, 32, 24))
    htw = torch.from_numpy((rng.rand(2, 17, 1) > 0.2).astype(np.float32))
    hout = hnet(hx)
    hloss = crit(hout, htarget, htw)
    hnet.zero_grad()
    hloss.backward()
    save = {"x": hx.numpy(), "target": htarget.numpy(), "target_weight": htw.numpy(), "out_train": hout.detach().numpy(),
            "loss": np.float32(hloss.item())}
    for k, v in hsd0.items():
        save["sd/" + k] = v.numpy()
    names, norms = [], []
    for k, p in hnet.named_parameters():
        names.append(k)
        norms.append(float(p.grad.double().norm()))
    save["grad_names"] = np.array(names)
    save["grad_norms"] = np.array(norms, np.float64)
    for k in ("conv1.weight", "layer1.0.downsample.0.weight", "transition1.1.0.0.weight",
              "stage3.1.fuse_layers.2.0.1.0.weight", "stage3.0.fuse_layers.0.2.1.weight",
              "stage4.0.branches.3.0.bn2.bias", "final_layer.bias"):
        save["grad/" + k] = dict(hnet.named_parameters())[k].grad.numpy()
    hnet.load_state_dict(hsd0)
    hnet.eval()
    with torch.no_grad():
        save["out_eval"] = hnet(hx).numpy()
    np.savez_compressed(os.path.join(OUT, "hrnet_small.npz"), **save)

    main_decode2()
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
