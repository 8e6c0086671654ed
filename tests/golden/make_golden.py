"""Generates the golden fixtures under tests/golden/ by running the UNMODIFIED reference (frgfm/Holocron,
mounted read-only at /root/reference) on seeded CPU inputs.  Run in the build container only:

    python tests/golden/make_golden.py

Every fixture is a dict of small tensors (inputs + the reference's outputs / gradients / updated state); the
tests compare the oracle (CPU) and the CUDA path (GPU) against them.
"""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle import reference_loader  # noqa: E402

OUT = Path(__file__).resolve().parent
holocron = reference_loader.load()
F = holocron.nn.functional
ops = holocron.ops.boxes


def grad_of(fn, *inputs, skip=()):
    """Runs fn on clones and returns (output, grads of output.sum()); inputs listed in `skip` get no grad
    (the reference's in-place patch normalisation makes its own backward fail when x requires grad)."""
    ins = [t.clone().requires_grad_(i not in skip) for i, t in enumerate(inputs)]
    out = fn(*ins)
    wrt = [t for t in ins if t.requires_grad]
    gs = list(torch.autograd.grad(out.sum() if out.ndim else out, wrt, allow_unused=True))
    full = [gs.pop(0) if t.requires_grad else None for t in ins]
    return out.detach(), full


def gen_activations():
    torch.manual_seed(11)
    x = torch.randn(4, 6, 9, 7) * 2.5
    x.view(-1)[:8] = torch.tensor([-3.0, -2.0, -1.0, 0.0, 1.0, 2.0, -2.5, 0.5])
    d = {"x": x}
    y, (g,) = grad_of(lambda t: F.hard_mish(t), x)
    d["hard_mish"], d["hard_mish_grad"] = y, g
    for beta in (1.0, 0.5):
        y, (g,) = grad_of(lambda t: F.nl_relu(t, beta=beta), x)
        d[f"nl_relu_b{beta}"], d[f"nl_relu_b{beta}_grad"] = y, g
    torch.save(d, OUT / "activations.pt")


def gen_losses():
    torch.manual_seed(12)
    d = {}
    # classification-shaped (N, K) and segmentation-shaped (N, K, H, W)
    for tag, shape in (("cls", (16, 10)), ("seg", (2, 5, 6, 7))):
        x = torch.randn(*shape) * 2
        k = shape[1]
        tshape = (shape[0],) + tuple(shape[2:])
        t = torch.randint(0, k, tshape)
        w = torch.rand(k) + 0.5
        d[f"{tag}_x"], d[f"{tag}_t"], d[f"{tag}_w"] = x, t, w
        for red in ("mean", "sum", "none"):
            for ii in (-100, 1):
                for use_w in (False, True):
                    key = f"{tag}_{red}_ii{ii}_w{int(use_w)}"
                    wt = w if use_w else None
                    y, (g,) = grad_of(lambda a: F.focal_loss(a, t, wt, ii, red, 2.0), x)
                    d["focal_" + key], d["focal_grad_" + key] = y, g
                    y, (g,) = grad_of(lambda a: F.poly_loss(a, t, 2.0, wt, ii, red), x)
                    d["poly_" + key], d["poly_grad_" + key] = y, g
        y, (g,) = grad_of(lambda a: F.focal_loss(a, t, None, -100, "mean", 0.5), x)
        d[f"focal_{tag}_gamma0.5"], d[f"focal_grad_{tag}_gamma0.5"] = y, g
        # soft targets for poly
        soft = torch.softmax(torch.randn(*shape), dim=1)
        d[f"{tag}_soft"] = soft
        for red in ("mean", "sum", "none"):
            for ii in (-100, 1):
                y, (g,) = grad_of(lambda a: F.poly_loss(a, soft, 2.0, None, ii, red), x)
                d[f"polysoft_{tag}_{red}_ii{ii}"], d[f"polysoft_grad_{tag}_{red}_ii{ii}"] = y, g
        if tag == "cls":
            y, (g,) = grad_of(lambda a: F.poly_loss(a, soft, 1.5, w, -100, "mean"), x)
            d["polysoft_cls_w"], d["polysoft_grad_cls_w"] = y, g
        # dice on probabilities
        prob = torch.softmax(x, dim=1)
        onehot = torch.nn.functional.one_hot(t, k).movedim(-1, 1).float()
        d[f"{tag}_prob"], d[f"{tag}_onehot"] = prob, onehot
        for gamma in ((1.0, 2.0) if tag == "seg" else ()):  # dice needs >= 3 dims (flatten(2) in the reference)
            for use_w in (False, True):
                wt = w if use_w else None
                y, (g,) = grad_of(lambda a: F.dice_loss(a, onehot, wt, gamma), prob)
                d[f"dice_{tag}_g{gamma}_w{int(use_w)}"], d[f"dice_grad_{tag}_g{gamma}_w{int(use_w)}"] = y, g
    torch.save(d, OUT / "losses.pt")


def gen_boxes():
    torch.manual_seed(13)
    kat = torch.tensor([[0, 0, 100, 100], [50, 50, 100, 100], [50, 50, 150, 150], [100, 100, 200, 200]],
                       dtype=torch.float32)  # reference tests/test_ops.py:9-13
    xy = torch.rand(37, 2) * 80
    wh = torch.rand(37, 2) * 40 + 1
    b1 = torch.cat([xy, xy + wh], 1)
    xy = torch.rand(23, 2) * 80
    wh = torch.rand(23, 2) * 40 + 1
    b2 = torch.cat([xy, xy + wh], 1)
    d = {"kat": kat, "b1": b1, "b2": b2}
    for name, (a, b) in (("kat", (kat, kat)), ("rnd", (b1, b2))):
        d[f"{name}_giou"] = ops.box_giou(a, b)
        d[f"{name}_penalty"] = ops.iou_penalty(a, b)
        d[f"{name}_diou"] = ops.diou_loss(a, b)
        d[f"{name}_ciou"] = ops.ciou_loss(a, b)
        d[f"{name}_arc"] = ops.aspect_ratio_consistency(a, b)
    d["kat_aspect"] = ops.aspect_ratio(kat)
    for fn in ("box_giou", "diou_loss", "ciou_loss"):
        _, gs = grad_of(lambda a, b: getattr(ops, fn)(a, b), b1, b2)
        d[f"rnd_{fn}_grad1"], d[f"rnd_{fn}_grad2"] = gs
    # weighted upstream gradient (not all-ones) for the loss used by YOLOv4
    up = torch.rand(37, 23)
    a = b1.clone().requires_grad_(True)
    b = b2.clone().requires_grad_(True)
    (ops.ciou_loss(a, b) * up).sum().backward()
    d["up"], d["rnd_ciou_wgrad1"], d["rnd_ciou_wgrad2"] = up, a.grad, b.grad
    torch.save(d, OUT / "boxes.pt")


def gen_convs():
    torch.manual_seed(14)
    d = {}
    x = torch.randn(2, 8, 9, 10)
    w = torch.randn(16, 8, 3, 3) * 0.2
    b = torch.randn(16) * 0.1
    d.update(x=x, w=w, b=b)
    for tag, kw in (("p1", dict(padding=1)), ("s2p1", dict(stride=2, padding=1)), ("d2p2", dict(dilation=2, padding=2)),
                    ("p0", dict())):
        y, gs = grad_of(lambda a, ww, bb: F.norm_conv2d(a, ww, bb, **kw), x, w, b, skip=(0,))
        d[f"normconv_{tag}"] = y
        d[f"normconv_{tag}_gw"], d[f"normconv_{tag}_gb"] = gs[1:]
        for ns in (False, True):
            y, gs = grad_of(lambda a, ww, bb: F.add2d(a, ww, bb, normalize_slices=ns, **kw), x, w, b,
                            skip=(0,) if ns else ())
            d[f"add2d_{tag}_n{int(ns)}"] = y
            if not ns:
                d[f"add2d_{tag}_n{int(ns)}_gx"] = gs[0]
            d[f"add2d_{tag}_n{int(ns)}_gw"], d[f"add2d_{tag}_n{int(ns)}_gb"] = gs[1:]
    # modules with seeded init: state_dict + output (+ input grad)
    nn = holocron.nn
    torch.manual_seed(15)
    fr = nn.FReLU(8)
    fr.bn.running_mean.normal_()
    fr.bn.running_var.uniform_(0.5, 1.5)
    fr.bn.weight.data.uniform_(0.5, 1.5)
    fr.bn.bias.data.normal_()
    d["frelu_state"] = {k: v.clone() for k, v in fr.state_dict().items()}
    fr.eval()
    y, (g,) = grad_of(lambda a: fr(a), x)
    d["frelu_eval"], d["frelu_eval_gx"] = y, g
    fr.train()
    y, (g,) = grad_of(lambda a: fr(a), x)
    d["frelu_train"], d["frelu_train_gx"] = y, g
    d["frelu_train_running_mean"], d["frelu_train_running_var"] = fr.bn.running_mean.clone(), fr.bn.running_var.clone()
    torch.manual_seed(16)
    sl = nn.SlimConv2d(8, 3, padding=1, r=4, L=2)
    d["slim_state"] = {k: v.clone() for k, v in sl.state_dict().items()}
    sl.eval()
    y, (g,) = grad_of(lambda a: sl(a), x)
    d["slim_eval"], d["slim_eval_gx"] = y, g
    # dropblock: noise drawn exactly like the reference (torch.rand((N, H, W)) on CPU under the seed)
    xd = torch.randn(2, 3, 12, 12)
    torch.manual_seed(17)
    d["dropblock_x"] = xd
    d["dropblock_out"] = F.dropblock2d(xd, 0.3, 3)
    torch.manual_seed(17)
    d["dropblock_noise"] = torch.rand((2, 12, 12))
    torch.save(d, OUT / "convs.pt")


def gen_optim():
    optim = holocron.optim
    d = {}
    shapes = [(7, 5), (33,), (4, 3, 3, 3), (1,)]
    torch.manual_seed(18)
    p0 = [torch.randn(*s) for s in shapes]
    grads = [[torch.randn(*s) * 0.3 for s in shapes] for _ in range(3)]
    d["p0"], d["grads"] = p0, grads
    cfgs = {
        "adabelief": (optim.AdaBelief, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-8)),
        "adabelief_wd_ams": (optim.AdaBelief, dict(lr=1e-2, betas=(0.95, 0.99), eps=1e-6, weight_decay=1e-2, amsgrad=True)),
        "lamb": (optim.LAMB, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-8)),
        "lamb_wd": (optim.LAMB, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-6, weight_decay=1e-2, scale_clip=(0.1, 2.0))),
        "tadam": (optim.TAdam, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-8)),
        "tadam_wd_ams_dof": (optim.TAdam, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-6, weight_decay=1e-2, amsgrad=True, dof=5.0)),
    }
    for name, (cls, kw) in cfgs.items():
        params = [torch.nn.Parameter(p.clone()) for p in p0]
        opt = cls(params, **kw)
        traj = []
        for step in range(3):
            for p, g in zip(params, grads[step]):
                p.grad = g.clone()
            opt.step()
            traj.append([p.detach().clone() for p in params])
        d[name] = traj
        d[name + "_kw"] = kw
    # AdamP (reference optim/adamp.py): tensors of several sizes, one of them with a gradient orthogonal to the weights so
    # that the projection branch fires; gradient of step k = k * g
    torch.manual_seed(1)
    shapes = [(64, 32, 3, 3), (64,), (10, 64), (1,), (4099,)]
    ps = [torch.randn(s) * 0.1 for s in shapes]
    gs = [torch.randn(s) * 1e-2 for s in shapes]
    gs[0] = gs[0] - (gs[0] * ps[0]).sum() / (ps[0] * ps[0]).sum() * ps[0]
    after = {}
    for amsgrad, wd in ((False, 0.0), (True, 1e-2)):
        params = [torch.nn.Parameter(p.clone()) for p in ps]
        opt = optim.AdamP(params, lr=1e-2, betas=(0.9, 0.99), eps=1e-8, weight_decay=wd, amsgrad=amsgrad, delta=0.1)
        for it in range(1, 4):
            for p, g in zip(params, gs):
                p.grad = g * it
            opt.step()
        after[f"adamp_{int(amsgrad)}"] = [p.detach().clone() for p in params]
    d["adamp"] = dict(params=ps, grads=gs, after=after)
    torch.save(d, OUT / "optim.pt")


def gen_models():
    models = holocron.models
    d = {}
    # fuse_conv_bn identity (reference tests/test_models.py:55-83)
    torch.manual_seed(19)
    conv = torch.nn.Conv2d(6, 8, 3, padding=1, bias=False)
    bn = torch.nn.BatchNorm2d(8).eval()
    bn.weight.data.uniform_(0.5, 1.5)
    bn.bias.data.normal_()
    bn.running_mean.normal_()
    bn.running_var.uniform_(0.5, 1.5)
    k, b = models.utils.fuse_conv_bn(conv, bn)
    d["fuse"] = dict(conv_w=conv.weight.detach().clone(), gamma=bn.weight.detach().clone(), beta=bn.bias.detach().clone(),
                     mean=bn.running_mean.clone(), var=bn.running_var.clone(), eps=bn.eps, k=k.clone(), b=b.clone())
    # RepBlock train-mode forward/backward on a small shape (stride 1 with identity, stride 2 without)
    from holocron.models.classification.repvgg import RepBlock
    for tag, (cin, cout, stride, ident) in (("s1", (16, 16, 1, True)), ("s2", (16, 32, 2, False))):
        torch.manual_seed(20)
        blk = RepBlock(cin, cout, stride, ident)
        for m in blk.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.data.uniform_(0.5, 1.5)
                m.bias.data.normal_(0, 0.2)
        state = {k_: v.clone() for k_, v in blk.state_dict().items()}
        x = torch.randn(4, cin, 10, 10)
        blk.train()
        xin = x.clone().requires_grad_(True)
        y = blk(xin)
        up = torch.randn_like(y)
        (y * up).sum().backward()
        grads = {n: p.grad.clone() for n, p in blk.named_parameters()}
        d[f"repblock_{tag}"] = dict(state=state, x=x, up=up, y=y.detach(), gx=xin.grad.clone(), grads=grads,
                                     state_after={k_: v.clone() for k_, v in blk.state_dict().items()})
        blk.eval()
        y_eval = blk(x).detach()
        blk.reparametrize()
        d[f"repblock_{tag}"]["y_eval"] = y_eval
        d[f"repblock_{tag}"]["y_reparam"] = blk(x).detach()
        d[f"repblock_{tag}"]["rep_w"] = blk.branches.weight.detach().clone()
        d[f"repblock_{tag}"]["rep_b"] = blk.branches.bias.detach().clone()
    # config 1: repvgg_a0, seed 0, 1x3x224x224 CPU input (BASELINE.json configs[0])
    torch.manual_seed(0)
    m = models.repvgg_a0(num_classes=1000).eval()
    x = torch.rand(1, 3, 224, 224)
    with torch.no_grad():
        logits = m(x)
        m.reparametrize()
        logits_rep = m(x)
    d["cfg1"] = dict(logits=logits, logits_rep=logits_rep, argmax=int(logits.argmax()), argmax_rep=int(logits_rep.argmax()),
                     x_sum=float(x.double().sum()), n_params=sum(p.numel() for p in m.parameters()))
    torch.manual_seed(0)
    m = models.repvgg_a0(num_classes=1000)
    d["cfg1"]["param_sum"] = float(sum(p.double().sum() for p in m.parameters()))
    d["cfg1"]["param_abs_sum"] = float(sum(p.double().abs().sum() for p in m.parameters()))
    d["cfg1"]["n_params_train"] = sum(p.numel() for p in m.parameters())
    torch.save(d, OUT / "models.pt")


def gen_optim2():
    """The remaining optimizers of the reference (SURVEY §8 f2): Adan, AdEMAMix, LARS, RaLars and the Lookahead wrapper, four
    steps each on tensors of several sizes (gradient of step k = k * g + 0.01 * p0) -> tests/golden/optim2.pt."""
    optim = holocron.optim
    torch.manual_seed(7)
    shapes = [(16, 8, 3, 3), (33,), (10, 16), (1,), (4099,)]
    ps = [torch.randn(s) * 0.2 for s in shapes]
    gs = [torch.randn(s) * 5e-2 for s in shapes]
    cfgs = {
        "adan": (optim.Adan, dict(lr=1e-2, betas=(0.98, 0.92, 0.99), eps=1e-8)),
        "adan_wd_ams": (optim.Adan, dict(lr=1e-2, betas=(0.9, 0.8, 0.95), eps=1e-6, weight_decay=2e-2, amsgrad=True)),
        "ademamix": (optim.AdEMAMix, dict(lr=1e-2, betas=(0.9, 0.99, 0.999), alpha=5.0, eps=1e-8)),
        "ademamix_wd": (optim.AdEMAMix, dict(lr=1e-2, betas=(0.8, 0.95, 0.99), alpha=2.0, eps=1e-6, weight_decay=1e-2)),
        "lars": (optim.LARS, dict(lr=1e-1)),
        "lars_mom_wd": (optim.LARS, dict(lr=1e-1, momentum=0.9, dampening=0.1, weight_decay=1e-2)),
        "lars_nesterov": (optim.LARS, dict(lr=1e-1, momentum=0.8, nesterov=True, weight_decay=1e-3)),
        "ralars": (optim.RaLars, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-8)),               # sma_t <= 4 during the first steps
        "ralars_rect_wd": (optim.RaLars, dict(lr=1e-2, betas=(0.5, 0.6), eps=1e-6, weight_decay=1e-2, scale_clip=(0.1, 1.0))),
        "ralars_force": (optim.RaLars, dict(lr=1e-2, betas=(0.9, 0.99), eps=1e-8, force_adaptive_momentum=True)),
    }
    d = dict(params=ps, grads=gs, steps=6)
    for name, (cls, kw) in cfgs.items():
        params = [torch.nn.Parameter(p.clone()) for p in ps]
        opt = cls(params, **kw)
        traj = []
        for it in range(1, 7):
            for p, p0, g in zip(params, ps, gs):
                p.grad = g * it + 0.01 * p0
            opt.step()
            if it in (1, 3, 6):
                traj.append([p.detach().clone() for p in params])
        d[name] = dict(kw=kw, traj=traj)      # parameters after steps 1, 3 and 6
        if "lars_mom" in name:
            d[name]["grad_after"] = [p.grad.clone() for p in params]     # the reference decays the gradient IN PLACE
        if name.startswith("ralars"):
            d[name]["local_lr"] = [float(opt.state[p]["local_lr"]) for p in params]
    # Lookahead over SGD with momentum: sync every 3 steps
    params = [torch.nn.Parameter(p.clone()) for p in ps]
    base = torch.optim.SGD(params, lr=0.1, momentum=0.9)
    la = optim.wrapper.Lookahead(base, sync_rate=0.5, sync_period=3)
    traj = []
    for it in range(1, 8):
        for p, p0, g in zip(params, ps, gs):
            p.grad = g * it + 0.01 * p0
        la.step()
        if it in (2, 3, 7):
            traj.append([p.detach().clone() for p in params])
    d["lookahead"] = dict(traj=traj, slow=[p.clone() for p in la.param_groups[0]["params"]], repr=repr(la))
    torch.save(d, OUT / "optim2.pt")


if __name__ == "__main__" and "--optim2" in sys.argv:
    gen_optim2()
    print("optim2.pt", (OUT / "optim2.pt").stat().st_size)


if __name__ == "__main__" and not any(f in sys.argv for f in ("--zoo", "--zoo-resnet", "--zoo-f3", "--zoo-f3b", "--yolo", "--trainers", "--seg", "--api", "--trainer", "--optim2", "--cross")):
    gen_activations()
    gen_losses()
    gen_boxes()
    gen_convs()
    gen_optim()
    gen_models()
    for f in sorted(OUT.glob("*.pt")):
        print(f.name, f.stat().st_size)


def gen_zoo():
    """Model-zoo fixtures (rows a10-a14, a21 of SURVEY §8) from the UNMODIFIED reference: seeded init (identical in both
    implementations, checked by the state_dict tests) + the shared conditioning of tests/_conditioning.py, then for every
    model two fp32 runs on seeded inputs:
      "eval"  - training-mode model with frozen (running-statistics) BatchNorm: outputs, loss, first / last / one BatchNorm
                gradient. Well conditioned -> the GPU test holds the bf16 CUDA path to <= 2e-2 against these directly.
      "train" - batch-statistics BatchNorm: outputs, loss, last-layer gradient (see oracle/eager.py for how the chaotic
                amplification of bf16 rounding in this mode is handled)."""
    sys.path.insert(0, str(ROOT / "tests"))
    import _conditioning as C
    models = holocron.models
    from holocron.nn import DropBlock2d
    d = {}

    def grads_of(model, names):
        ps = dict(model.named_parameters())
        return {n: ps[n].grad.clone() for n in names}

    def build(factory, **kw):
        torch.manual_seed(0)
        m = factory(**kw)
        for mod in m.modules():          # device-specific RNG streams off
            if isinstance(mod, DropBlock2d):
                mod.p = 0.0
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
        return C.condition(m)

    def pick_names(m, last):
        names = [n for n, _ in m.named_parameters()]
        bn_w = [n for n, mod in m.named_modules() if isinstance(mod, torch.nn.BatchNorm2d)]
        mid = bn_w[len(bn_w) // 2] + ".weight" if bn_w else names[len(names) // 2]
        return names[0], mid, last

    for name in C.CLS:
        out = {}
        for mode in ("eval", "train"):
            m = build(getattr(models, name), num_classes=10)
            m = C.freeze_bn(m) if mode == "eval" else m.train()
            x, t = C.cls_inputs(name, mode)
            store = {}
            C.capture(m, C.PROBE[name], store)
            logits = m(x)
            loss = torch.nn.functional.cross_entropy(logits, t)
            loss.backward()
            last = [n for n, _ in m.named_parameters()][-2]
            first, mid, last = pick_names(m, last)
            out[mode] = dict(logits=logits.detach(), loss=loss.detach(), first=first, mid=mid, last=last,
                             grads=grads_of(m, [first, mid, last]), probe=store["probe"][:2].half() if mode == "train" else None)
        d[name] = out
    # UNet3+ with DiceLoss (BASELINE config 5, at 64x64)
    out = {}
    for mode in ("eval", "train"):
        m = build(models.segmentation.unet3p, num_classes=21)
        m = C.freeze_bn(m) if mode == "eval" else m.train()
        x, mask = C.unet_inputs()
        onehot = torch.nn.functional.one_hot(mask, 21).movedim(-1, 1).float()
        store = {}
        C.capture(m, C.PROBE["unet3p"], store)
        o = m(x)
        loss = F.dice_loss(torch.softmax(o, 1), onehot)
        loss.backward()
        first, mid, last = pick_names(m, "classifier.weight")
        out[mode] = dict(out=o.detach(), loss=loss.detach(), first=first, mid=mid, last=last, grads=grads_of(m, [first, mid, last]),
                         probe=store["probe"][:2].half() if mode == "train" else None)
    d["unet3p"] = out
    # YOLOv4 (BASELINE config 4, at 128x128): the four losses, gradients of an output convolution, a neck and a backbone filter
    out = {}
    for mode in ("eval", "train"):
        m = build(models.detection.yolov4, pretrained_backbone=False, num_classes=80)
        m = C.freeze_bn(m) if mode == "eval" else m.train()
        x, target = C.yolo_inputs()
        store = {}
        C.capture(m, C.PROBE["yolov4"], store)
        losses = m(x, target)
        sum(losses.values()).backward()
        names = ["head.head1.3.weight", "head.head3.24.weight", "neck.pan2.convs.0.weight", "backbone.stem.0.weight"]
        ps = dict(m.named_parameters())
        names = [n for n in names if n in ps]
        out[mode] = dict(losses={k: v.detach() for k, v in losses.items()}, grads=grads_of(m, names), probe=store["probe"][:1].half() if mode == "train" else None)
    d["yolov4"] = out
    # shared (cell, anchor) slot: two boxes of one image collapse into one assigned prediction in the reference's masks
    m = C.freeze_bn(build(models.detection.yolov4, pretrained_backbone=False, num_classes=80))
    x, target = C.yolo_dup_inputs()
    losses = m(x, target)
    sum(losses.values()).backward()
    ps = dict(m.named_parameters())
    d["yolov4_dup"] = dict(losses={k: v.detach() for k, v in losses.items()},
                           grads={"head.head1.3.weight": ps["head.head1.3.weight"].grad.clone()})
    torch.save(d, OUT / "zoo.pt")


def gen_zoo_resnet(which="CLS_RESNET", outfile="zoo_resnet.pt"):
    """ResNet-family fixtures (SURVEY §8 f3), same recipe as gen_zoo's classification part -> tests/golden/zoo_resnet.pt;
    ``--zoo-f3``: Res2Net / SKNet / ConvNeXt (tests/_conditioning.py CLS_F3) -> tests/golden/zoo_f3.pt."""
    sys.path.insert(0, str(ROOT / "tests"))
    import _conditioning as C
    d = {}
    for name in getattr(C, which):
        out = {}
        for mode in ("eval", "train"):
            torch.manual_seed(0)
            m = C.condition(getattr(holocron.models, name)(num_classes=10))
            m = C.freeze_bn(m) if mode == "eval" else m.train()
            x, t = C.cls_inputs(name, mode)
            store = {}
            C.capture(m, C.PROBE[name], store)
            logits = m(x)
            loss = torch.nn.functional.cross_entropy(logits, t)
            loss.backward()
            names = [n for n, _ in m.named_parameters()]
            bns = [n for n, mod in m.named_modules() if isinstance(mod, (torch.nn.BatchNorm2d, torch.nn.LayerNorm))]
            ps = dict(m.named_parameters())
            # first filter with more than one tap per output channel: a depth-wise 1x1 filter in front of a batch-statistics
            # BatchNorm (MobileOne's scale branch) has a structurally ZERO gradient - nothing to compare but round-off
            first = next(n for n in names if ps[n].ndim == 4 and ps[n][0].numel() > 1)
            mid, last = bns[len(bns) // 2] + ".weight", names[-2]
            out[mode] = dict(logits=logits.detach(), loss=loss.detach(), first=first, mid=mid, last=last,
                             grads={n: ps[n].grad.clone() for n in (first, mid, last)},
                             probe=store["probe"][:2].half() if mode == "train" else None)
            # conditioning of the fixture itself: the SAME reference model on inputs scaled by (1 + 1e-7). With batch-statistics
            # BatchNorm the early-layer gradients of MobileOne-S0 move by 3-4 % (fp32!), those of the ResNets by < 1e-4; the
            # tests bound their comparison by max(tolerance, 2 x this).
            torch.manual_seed(0)
            m2 = C.condition(getattr(holocron.models, name)(num_classes=10))
            m2 = C.freeze_bn(m2) if mode == "eval" else m2.train()
            torch.nn.functional.cross_entropy(m2(x * (1 + 1e-7)), t).backward()
            ps2 = dict(m2.named_parameters())
            out[mode]["sensitivity"] = {n: float((ps2[n].grad - ps[n].grad).norm() / ps[n].grad.norm()) for n in (first, mid, last)}
        if hasattr(getattr(holocron.models, name)(num_classes=10), "reparametrize"):
            # inference form (reference mobileone.py:222-230): eval-mode logits before / after folding the branches
            torch.manual_seed(0)
            m = C.condition(getattr(holocron.models, name)(num_classes=10)).eval()
            x, _ = C.cls_inputs(name, "eval")
            with torch.no_grad():
                before = m(x)
                m.reparametrize()
                out["reparam"] = dict(before=before, after=m(x), keys=list(m.state_dict().keys())[:6])
        d[name] = out
    torch.save(d, OUT / outfile)


if __name__ == "__main__" and "--zoo-f3b" in sys.argv:
    gen_zoo_resnet("CLS_F3B", "zoo_f3b.pt")
    print("zoo_f3b.pt", (OUT / "zoo_f3b.pt").stat().st_size)


if __name__ == "__main__" and "--zoo-f3" in sys.argv:
    gen_zoo_resnet("CLS_F3", "zoo_f3.pt")
    print("zoo_f3.pt", (OUT / "zoo_f3.pt").stat().st_size)


def gen_yolo():
    """YOLOv1 / YOLOv2 fixtures (SURVEY §8 f3: reference models/detection/yolo.py, yolov2.py) -> tests/golden/zoo_yolo.pt:
    the four losses in frozen-BatchNorm and batch-statistics mode, gradients of the first / a middle / the last parameter,
    an early probe activation, and eval-mode detections of a model whose objectness bias is raised so that boxes survive."""
    sys.path.insert(0, str(ROOT / "tests"))
    import _conditioning as C
    d = {}
    for name in ("yolov1", "yolov2"):
        out = {}
        for mode in ("eval", "train"):
            torch.manual_seed(0)
            m = getattr(holocron.models.detection, name)(pretrained_backbone=False, num_classes=20)
            for mod in m.modules():
                if isinstance(mod, torch.nn.Dropout):
                    mod.p = 0.0
            m = C.condition(m)
            m = C.freeze_bn(m) if mode == "eval" else m.train()
            x, target = C.yolo12_inputs(name)
            store = {}
            C.capture(m, C.PROBE[name], store)
            losses = m(x, target)
            sum(losses.values()).backward()
            ps = dict(m.named_parameters())
            names = [n for n, _ in m.named_parameters()]
            bns = [n for n, mod in m.named_modules() if isinstance(mod, torch.nn.BatchNorm2d)]
            # YOLOv1 has no normalisation layers by default (convolution bias + LeakyReLU): a middle filter instead
            keys = [names[0], bns[len(bns) // 2] + ".weight" if bns else names[len(names) // 2 // 2 * 2], names[-2]]
            out[mode] = dict(losses={k: v.detach() for k, v in losses.items()}, grads={k: C.head_rows(ps[k].grad).clone() for k in keys},
                             probe=store["probe"][:1, :32].half() if mode == "train" else None)
        d[name] = out
    torch.save(d, OUT / "zoo_yolo.pt")


if __name__ == "__main__" and "--yolo" in sys.argv:
    gen_yolo()
    print("zoo_yolo.pt", (OUT / "zoo_yolo.pt").stat().st_size)


if __name__ == "__main__" and "--zoo-resnet" in sys.argv:
    gen_zoo_resnet()
    print("zoo_resnet.pt", (OUT / "zoo_resnet.pt").stat().st_size)


if __name__ == "__main__" and "--zoo" in sys.argv:
    gen_zoo()
    print("zoo.pt", (OUT / "zoo.pt").stat().st_size)


# ------------------------------------------------------------------------------------------------ public API surface
API_SURFACE = {
    "nn.functional": ["hard_mish", "nl_relu", "focal_loss", "poly_loss", "dice_loss", "norm_conv2d", "add2d", "dropblock2d",
                      "concat_downsample2d"],
    "nn": ["HardMish", "NLReLU", "FReLU", "NormConv2d", "Add2d", "SlimConv2d", "FocalLoss", "PolyLoss", "DiceLoss", "DropBlock2d",
           "GlobalAvgPool2d", "SPP", "ConcatDownsample2d", "PyConv2d"],
    "ops.boxes": ["box_giou", "diou_loss", "ciou_loss", "iou_penalty", "aspect_ratio", "aspect_ratio_consistency"],
    "optim": ["AdaBelief", "LAMB", "TAdam", "AdamP", "Adan", "AdEMAMix", "LARS", "RaLars"],
    "optim.wrapper": ["Lookahead"],
    "models": ["repvgg_a0", "repvgg_a1", "repvgg_a2", "repvgg_b0", "repvgg_b1", "repvgg_b2", "repvgg_b3", "rexnet1_0x", "rexnet1_3x",
               "rexnet1_5x", "rexnet2_0x", "rexnet2_2x", "darknet24", "darknet19", "darknet53", "cspdarknet53", "cspdarknet53_mish",
               "resnet18", "resnet34", "resnet50", "resnet50d", "resnet101", "resnet152", "resnext50_32x4d", "resnext101_32x8d",
               "mobileone_s0", "mobileone_s1", "mobileone_s2", "mobileone_s3", "res2net50_26w_4s", "sknet50", "sknet101", "sknet152",
               "convnext_atto", "convnext_femto", "convnext_pico", "convnext_nano", "convnext_tiny", "convnext_small",
               "convnext_base", "convnext_large", "convnext_xl", "tridentnet50", "pyconv_resnet50", "pyconvhg_resnet50"],
    "models.detection": ["yolov4", "yolov1", "yolov2", "YOLOv1", "YOLOv2"],
    "models.segmentation": ["unet3p", "unet", "unet2", "unetp", "unetpp", "unet_rexnet13", "unet_tvvgg11", "unet_tvresnet34", "UNet",
                            "DynamicUNet", "UNetp", "UNetpp"],
}


def describe_signature(obj):
    """[(name, kind, repr(default))] of a callable / of a class' constructor - annotations left out on purpose."""
    import inspect
    target = obj.__init__ if inspect.isclass(obj) else obj
    out = []
    for name, p in inspect.signature(target).parameters.items():
        if name == "self":
            continue
        default = None if p.default is inspect.Parameter.empty else repr(p.default)
        out.append([name, p.kind.name, default])
    return out


def gen_api():
    """Signatures of the reference's public hot-path surface (SURVEY §8b) -> tests/golden/api_signatures.json."""
    import functools
    import json
    d = {}
    for mod_path, names in API_SURFACE.items():
        mod = functools.reduce(getattr, mod_path.split("."), holocron)
        for name in names:
            d[f"{mod_path}.{name}"] = describe_signature(getattr(mod, name))
    (OUT / "api_signatures.json").write_text(json.dumps(d, indent=1, sort_keys=True))
    # classes: public base classes (isinstance contract, e.g. AdaBelief is a torch.optim.Adam) and public properties
    # (e.g. DropBlock2d.drop_prob) of the reference's classes -> tests/golden/api_classes.json
    import inspect
    c = {}
    for mod_path, names in API_SURFACE.items():
        mod = functools.reduce(getattr, mod_path.split("."), holocron)
        for name in names:
            obj = getattr(mod, name)
            if not inspect.isclass(obj):
                continue
            bases = [f"{b.__module__}.{b.__qualname__}" for b in obj.__mro__[1:] if b.__module__.startswith("torch")]
            props = sorted(k for k, v in vars(obj).items() if isinstance(v, property) and not k.startswith("_"))
            c[f"{mod_path}.{name}"] = {"torch_bases": bases, "properties": props}
    (OUT / "api_classes.json").write_text(json.dumps(c, indent=1, sort_keys=True))


if __name__ == "__main__" and "--api" in sys.argv:
    gen_api()
    print("api_signatures.json", (OUT / "api_signatures.json").stat().st_size)


def describe_state_dict(model):
    """(number of entries, total elements, sha1 over 'key:shape:dtype' lines, sha1 over the seeded VALUES)."""
    import hashlib
    sd = model.state_dict()
    lines = [f"{k}:{tuple(v.shape)}:{str(v.dtype).replace('torch.', '')}" for k, v in sd.items()]
    h_vals = hashlib.sha1()
    for v in sd.values():
        h_vals.update(v.detach().contiguous().cpu().numpy().tobytes())
    return {"entries": len(lines), "numel": int(sum(v.numel() for v in sd.values())),
            "layout_sha1": hashlib.sha1("\n".join(lines).encode()).hexdigest(), "values_sha1": h_vals.hexdigest(),
            "first": lines[:3], "last": lines[-3:]}


def gen_state_dicts():
    """state_dict layout and seeded initial values of every factory -> tests/golden/state_dicts.json (checkpoint
    compatibility + init RNG order: torch.manual_seed(0) before each constructor)."""
    import json
    d = {}
    for name in API_SURFACE["models"]:
        torch.manual_seed(0)
        d[name] = describe_state_dict(getattr(holocron.models, name)(num_classes=10))
    torch.manual_seed(0)
    d["yolov4"] = describe_state_dict(holocron.models.detection.yolov4(pretrained_backbone=False, num_classes=80))
    torch.manual_seed(0)
    d["unet3p"] = describe_state_dict(holocron.models.segmentation.unet3p(num_classes=21))
    for name in ("yolov1", "yolov2"):
        torch.manual_seed(0)
        d[name] = describe_state_dict(getattr(holocron.models.detection, name)(pretrained_backbone=False, num_classes=20))
    for name in ("unet", "unetp", "unetpp", "unet2", "unet_rexnet13", "unet_tvvgg11", "unet_tvresnet34"):
        torch.manual_seed(0)
        kw = {} if name in ("unet", "unetp", "unetpp", "unet2") else {"pretrained_backbone": False}
        d[name] = describe_state_dict(getattr(holocron.models.segmentation, name)(num_classes=5, **kw))
    (OUT / "state_dicts.json").write_text(json.dumps(d, indent=1, sort_keys=True))


if __name__ == "__main__" and "--api" in sys.argv:
    gen_state_dicts()
    print("state_dicts.json", (OUT / "state_dicts.json").stat().st_size)


# ------------------------------------------------------------------------------------------------ trainer semantics
def gen_trainer():
    """Golden runs of the UNMODIFIED reference Trainer (holocron/trainer/core.py: _fit_epoch, _backprop_step, _reset_opt,
    _reset_scheduler) on a tiny RepVGG, CPU fp32 -> tests/golden/trainer.pt. matplotlib / fastprogress (absent here, only used
    for plots and progress bars) are stubbed before the import; nothing of the training logic is touched."""
    import types
    for name in ("matplotlib", "matplotlib.pyplot", "fastprogress", "fastprogress.fastprogress"):
        sys.modules.setdefault(name, types.ModuleType(name))

    class _Bar(list):
        def __init__(self, it, parent=None):
            super().__init__(it)
            self.comment = ""
            self.main_bar = types.SimpleNamespace(comment="")

        def write(self, *a, **k):
            pass
    sys.modules["fastprogress"].master_bar = _Bar
    sys.modules["fastprogress"].progress_bar = _Bar
    sys.modules["fastprogress.fastprogress"].ConsoleMasterBar = _Bar
    import importlib
    core = importlib.import_module("holocron.trainer.core")
    tutils = importlib.import_module("holocron.trainer.utils")
    from holocron.models.classification.repvgg import RepVGG
    from holocron.optim import AdaBelief

    def tiny():
        torch.manual_seed(0)
        return RepVGG([1, 1, 1], [16, 32, 64], 1, 1, num_classes=10)

    def batches(n, nan_at=None):
        g = torch.Generator().manual_seed(31)
        out = []
        for i in range(n):
            x = (torch.rand(8, 3, 32, 32, generator=g) - 0.45) / 0.225
            if nan_at is not None and i == nan_at:
                x = x.clone()
                x[0, 0, 0, 0] = float("nan")
            out.append((x, torch.randint(0, 10, (8,), generator=g)))
        return out

    class T(core.Trainer):
        def evaluate(self):
            return {"val_loss": 0.0}

        @staticmethod
        def _eval_metrics_str(m):
            return ""

    d = {}
    scenarios = {
        "acc2_clip_onecycle": dict(gradient_acc=2, gradient_clip=0.5, skip_nan_loss=False, sched="onecycle", lr=2e-3, nan_at=None),
        "nan_skip_cosine": dict(gradient_acc=1, gradient_clip=None, skip_nan_loss=True, sched="cosine", lr=1e-3, nan_at=3),
    }
    for tag, cfg in scenarios.items():
        model = tiny()
        data = batches(8, cfg["nan_at"])
        opt = AdaBelief(model.parameters(), lr=1e-3, betas=(0.95, 0.99), eps=1e-6)
        tr = T(model, data, data, torch.nn.CrossEntropyLoss(), opt, gpu=None, output_file="/tmp/_hb_golden_ckpt.pth", amp=False,
               skip_nan_loss=cfg["skip_nan_loss"], nan_tolerance=5, gradient_acc=cfg["gradient_acc"], gradient_clip=cfg["gradient_clip"])
        losses, lrs, beta1s = [], [], []
        orig = tr._get_loss

        def rec(x, t, return_logits=False, orig=orig, tr=tr):
            lrs.append(tr.optimizer.param_groups[0]["lr"])
            beta1s.append(tr.optimizer.param_groups[0]["betas"][0])
            loss = orig(x, t, return_logits)
            losses.append(float(loss.detach()))
            return loss
        tr._get_loss = rec
        tutils.freeze_model(tr.model.train(), None)
        tr._reset_opt(cfg["lr"], None)
        tr._reset_scheduler(cfg["lr"], 1, cfg["sched"])
        tr._fit_epoch(_Bar(range(1)))
        d[tag] = dict(cfg=cfg, losses=torch.tensor(losses), lrs=torch.tensor(lrs, dtype=torch.float64),
                      beta1s=torch.tensor(beta1s, dtype=torch.float64),
                      state={k: v.clone() for k, v in model.state_dict().items()},
                      opt_steps=int(next(iter(opt.state.values()))["step"]))
    # freezing helpers on the reference's tiny model: names of frozen parameters / eval-mode BatchNorms, normalisation split
    model = tiny()
    tutils.freeze_model(model.train(), "features.1")
    d["freeze"] = dict(frozen=[n for n, p in model.named_parameters() if not p.requires_grad],
                       bn_eval=[n for n, m in model.named_modules() if isinstance(m, torch.nn.BatchNorm2d) and not m.training])
    norm, other = tutils.split_normalization_params(tiny())
    d["split"] = dict(norm=len(norm), other=len(other), norm_numel=sum(p.numel() for p in norm), other_numel=sum(p.numel() for p in other))
    torch.save(d, OUT / "trainer.pt")


if __name__ == "__main__" and "--trainer" in sys.argv:
    gen_trainer()
    print("trainer.pt", (OUT / "trainer.pt").stat().st_size)


# ------------------------------------------------------------------------------------------------ trainer classes
def gen_trainers():
    """The UNMODIFIED reference trainer classes (ClassificationTrainer, BinaryClassificationTrainer, SegmentationTrainer,
    DetectionTrainer, assign_iou, fit_n_epochs / find_lr / check_setup) on the scenarios of tests/_trainer_cases.py ->
    tests/golden/trainers.pt. fastprogress / matplotlib / tqdm are stubbed (progress bars and plots only)."""
    import types
    for name in ("matplotlib", "matplotlib.pyplot", "fastprogress", "fastprogress.fastprogress", "tqdm", "tqdm.auto"):
        sys.modules.setdefault(name, types.ModuleType(name))

    class _Bar(list):
        def __init__(self, it, parent=None):
            super().__init__(it)
            self.comment = ""
            self.main_bar = types.SimpleNamespace(comment="")

        def write(self, *a, **k):
            pass
    sys.modules["fastprogress"].master_bar = _Bar
    sys.modules["fastprogress"].progress_bar = _Bar
    sys.modules["fastprogress.fastprogress"].ConsoleMasterBar = _Bar
    for fn in ("plot", "xlabel", "ylabel", "grid", "show", "xscale", "ylim", "subplots"):
        setattr(sys.modules["matplotlib.pyplot"], fn, lambda *a, **k: None)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    for m in ("tqdm", "tqdm.auto"):
        sys.modules[m].tqdm = lambda it, *a, **k: it
    import importlib
    T = importlib.import_module("holocron.trainer")
    sys.path.insert(0, str(ROOT / "tests"))
    import _trainer_cases as cases
    import tempfile
    d = {}
    with tempfile.TemporaryDirectory() as tmp:
        cases.run_scenarios(T, lambda tag, rec: d.__setitem__(tag, rec), str(Path(tmp) / "ckpt.pth"))
    torch.save(d, OUT / "trainers.pt")


if __name__ == "__main__" and "--trainers" in sys.argv:
    gen_trainers()
    print("trainers.pt", (OUT / "trainers.pt").stat().st_size)


def gen_seg():
    """U-Net family fixtures (reference models/segmentation/unet.py, unetpp.py) -> tests/golden/zoo_seg.pt: logits, cross-entropy
    loss, first / middle / last parameter gradients (large ones cut to their first rows), an encoder probe."""
    sys.path.insert(0, str(ROOT / "tests"))
    import _conditioning as C
    d = {}
    for name in C.SEG:
        out = {}
        for mode in ("eval", "train"):
            torch.manual_seed(0)
            m = C.condition(getattr(holocron.models.segmentation, name)(**C.seg_kwargs(name)))
            m = C.freeze_bn(m) if mode == "eval" else m.train()
            x, mask = C.seg_inputs()
            store = {}
            C.capture(m, C.PROBE[name], store)
            o = m(x)
            loss = torch.nn.functional.cross_entropy(o, mask)
            loss.backward()
            names = [n for n, p in m.named_parameters() if p.grad is not None]
            ps = dict(m.named_parameters())
            keys = [names[0], names[len(names) // 2 // 2 * 2], names[-2]]
            out[mode] = dict(out=o.detach(), loss=loss.detach(), grads={k: C.head_rows(ps[k].grad).clone() for k in keys},
                             probe=store["probe"][:1, :32].half() if mode == "train" else None)
        d[name] = out
    torch.save(d, OUT / "zoo_seg.pt")


if __name__ == "__main__" and "--seg" in sys.argv:
    gen_seg()
    print("zoo_seg.pt", (OUT / "zoo_seg.pt").stat().st_size)


# ------------------------------------------------------------------------------------------------ module / format cross-checks
def gen_cross():
    """What the reference's own PyConv2d / TridentConv2d / ConcatDownsample2d modules, its Mixup collate and its hub loader
    produce on seeded inputs -> tests/golden/cross_checks.pt (tests/test_zoo_wiring_cpu.py, tests/test_host_logic.py,
    tests/test_formats_cpu.py compare against it)."""
    import importlib.util
    import types
    for name in ("matplotlib", "matplotlib.pyplot", "tqdm", "tqdm.auto"):     # plots / progress bars of holocron.utils only
        try:
            missing = name not in sys.modules and importlib.util.find_spec(name) is None
        except (ImportError, ValueError):
            missing = True
        if missing:
            stub = types.ModuleType(name)
            stub.tqdm = lambda it, *a, **k: it
            sys.modules[name] = stub
    d = {}
    g = torch.Generator().manual_seed(20)
    x = torch.rand(2, 8, 8, 8, generator=g)
    pyconv = []
    for kwargs in (dict(num_levels=1), dict(num_levels=2), dict(num_levels=3, groups=[1, 2, 4]), dict(num_levels=4, stride=2)):
        torch.manual_seed(0)
        ref = holocron.nn.PyConv2d(8, 16, 3, padding=1, **kwargs)
        pyconv.append(dict(kwargs=kwargs, params=[p.detach().clone() for p in ref.parameters()], num_levels=ref.num_levels,
                           out=ref(x).detach()))
    d["pyconv"] = dict(x=x, cases=pyconv)
    from holocron.models.classification.tridentnet import TridentConv2d as RefTrident
    x3 = torch.rand(1, 24, 8, 8, generator=g)
    trident = []
    for k, dil in ((1, 1), (3, 3)):
        torch.manual_seed(1)
        ref = RefTrident(8, 8, k, padding=k // 2, dilation=dil, bias=False)
        trident.append(dict(k=k, dil=dil, state={n: v.clone() for n, v in ref.state_dict().items()}, out=ref(x3).detach()))
    d["trident"] = dict(x=x3, cases=trident)
    xc = torch.rand(2, 6, 8, 12, generator=g)
    d["concat_downsample"] = dict(x=xc, out=holocron.nn.ConcatDownsample2d(2)(xc))
    from holocron.utils.data import Mixup as RefMixup
    mixup = []
    for num_classes, alpha, seed in ((7, 0.2, 0), (7, 1.0, 1), (1, 0.4, 2)):
        gm = torch.Generator().manual_seed(seed)
        xm = torch.rand(6, 3, 5, 5, generator=gm)
        tm = torch.randint(0, max(num_classes, 2), (6,), generator=gm)
        torch.manual_seed(100 + seed)
        xr, tr = RefMixup(num_classes, alpha)(xm.clone(), tm.clone())
        mixup.append(dict(num_classes=num_classes, alpha=alpha, seed=seed, x=xm, t=tm, x_out=xr, t_out=tr))
    d["mixup"] = mixup
    # hub format: the architecture keys the reference's model_from_hf_hub resolves (holocron.models.__dict__[cfg["arch"]]) and
    # the state_dict layout its strict load_state_dict accepts for a 10-class rexnet1_0x, read back through that loader
    import json
    import tempfile
    ref_utils = holocron.models.utils
    torch.manual_seed(4)
    src = holocron.models.rexnet1_0x(num_classes=10)
    with tempfile.TemporaryDirectory() as tmp:
        folder = Path(tmp)
        (folder / "config.json").write_text(json.dumps({"arch": "rexnet1_0x", "classes": [str(i) for i in range(10)]}))
        torch.save(src.state_dict(), folder / "pytorch_model.bin")
        orig = ref_utils.hf_hub_download
        ref_utils.hf_hub_download = lambda repo_id, filename, **kw: str(folder / filename)
        try:
            loaded = ref_utils.model_from_hf_hub("frgfm/rexnet1_0x")
        finally:
            ref_utils.hf_hub_download = orig
    d["hub"] = dict(arch="rexnet1_0x", num_classes=10,
                    registry=sorted(k for k, v in vars(holocron.models).items() if callable(v) and not k.startswith("_")),
                    layout=[(k, tuple(v.shape), v.dtype) for k, v in loaded.state_dict().items()])
    torch.save(d, OUT / "cross_checks.pt")


if __name__ == "__main__" and "--cross" in sys.argv:
    gen_cross()
    print("cross_checks.pt", (OUT / "cross_checks.pt").stat().st_size)
