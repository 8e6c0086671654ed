"""Shared scenarios for the trainer-class parity tests: tiny stock-torch models and seeded batches, used by
tests/golden/make_golden.py --trainers (driving the UNMODIFIED reference trainers) and by tests/test_trainers_cpu.py (driving
holocron_b200.trainer's classes through the same calls). CPU, fp32, generic (host-driven) optimizer path."""
import torch
from torch import nn


def cls_model(num_out: int = 7):
    torch.manual_seed(0)
    return nn.Sequential(nn.Conv2d(3, 8, 3, padding=1, bias=False), nn.BatchNorm2d(8), nn.ReLU(), nn.AdaptiveAvgPool2d(1),
                         nn.Flatten(), nn.Linear(8, num_out))


def seg_model(num_classes: int = 5):
    torch.manual_seed(0)
    return nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, num_classes, 1))


def cls_batches(n: int, seed: int, num_out: int = 7, binary: bool = False):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        x = torch.randn(8, 3, 12, 12, generator=g)
        t = torch.randint(0, 2, (8,), generator=g) if binary else torch.randint(0, num_out, (8,), generator=g)
        out.append((x, t))
    return out


def seg_batches(n: int, seed: int, num_classes: int = 5):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        x = torch.randn(4, 3, 12, 12, generator=g)
        t = torch.randint(0, num_classes, (4, 12, 12), generator=g)
        t[:, :2, :3] = 255                       # ignored region
        out.append((x, t))
    return out


class FixedDetector(nn.Module):
    """Detector stand-in: a loss dict in training mode, canned detections in eval mode (one entry per image)."""

    def __init__(self, detections):
        super().__init__()
        self.w = nn.Parameter(torch.tensor(0.5))
        self.detections = detections
        self._i = 0

    def forward(self, x, target=None):
        if self.training:
            s = sum(img.mean() for img in x)
            return {"obj_loss": (self.w * s - 1.0) ** 2, "clf_loss": self.w ** 2 * 0.1}
        out = self.detections[self._i: self._i + len(x)]
        self._i = (self._i + len(x)) % len(self.detections)
        return out


def det_data():
    """Two batches of two images: exact hits, a wrong label, a missed box, a spurious detection, two ground-truth boxes
    claiming the same prediction (assign_iou's de-duplication loop), an empty image."""
    b = lambda *rows: torch.tensor(rows, dtype=torch.float32)   # noqa: E731
    targets = [
        {"boxes": b([0.1, 0.1, 0.4, 0.4], [0.5, 0.5, 0.9, 0.9]), "labels": torch.tensor([1, 2])},
        {"boxes": b([0.2, 0.2, 0.6, 0.6], [0.22, 0.2, 0.62, 0.6]), "labels": torch.tensor([3, 3])},
        {"boxes": torch.zeros((0, 4)), "labels": torch.zeros(0, dtype=torch.long)},
        {"boxes": b([0.0, 0.0, 0.3, 0.3]), "labels": torch.tensor([4])},
    ]
    detections = [
        {"boxes": b([0.1, 0.1, 0.4, 0.42], [0.5, 0.5, 0.9, 0.88], [0.0, 0.6, 0.2, 0.9]), "scores": torch.tensor([0.9, 0.8, 0.7]),
         "labels": torch.tensor([1, 5, 2])},
        {"boxes": b([0.2, 0.2, 0.6, 0.6]), "scores": torch.tensor([0.9]), "labels": torch.tensor([3])},
        {"boxes": b([0.3, 0.3, 0.5, 0.5]), "scores": torch.tensor([0.6]), "labels": torch.tensor([1])},
        {"boxes": torch.zeros((0, 4)), "scores": torch.zeros(0), "labels": torch.zeros(0, dtype=torch.long)},
    ]
    g = torch.Generator().manual_seed(5)
    images = [torch.rand(3, 8, 8, generator=g) for _ in range(4)]
    loader = [(images[:2], targets[:2]), (images[2:], targets[2:])]
    return loader, detections


class FlakyCrossEntropy(nn.CrossEntropyLoss):
    """Cross-entropy whose ``bad``-th call returns NaN (a NaN input would poison the BatchNorm running statistics and with
    them every later evaluation; this keeps the model healthy and exercises the skip logic alone)."""

    def __init__(self, bad: int):
        super().__init__()
        self.bad, self.calls = bad, 0

    def forward(self, out, target):
        self.calls += 1
        loss = super().forward(out, target)
        return loss * float("nan") if self.calls == self.bad else loss


def run_scenarios(T, record, output_file):
    """Drives the trainer classes of namespace ``T`` (reference or this package) through every scenario; ``record(tag, dict)``
    stores the observable results. The trainers write their checkpoints to ``output_file``."""
    sd = lambda m: {k: v.detach().clone() for k, v in m.state_dict().items()}   # noqa: E731
    # 1. classification: two epochs, one-cycle schedule, gradient accumulation + clipping
    model = cls_model()
    seen = []
    tr = T.ClassificationTrainer(model, cls_batches(6, 1), cls_batches(3, 2), nn.CrossEntropyLoss(),
                                 torch.optim.Adam(model.parameters(), lr=1e-3), gpu=None, output_file=output_file,
                                 gradient_acc=2, gradient_clip=0.5, on_epoch_end=lambda m: seen.append(dict(m)))
    tr.fit_n_epochs(2, 3e-3, sched_type="onecycle")
    ckpt = torch.load(output_file, map_location="cpu")
    record("cls_fit", dict(metrics=seen, state=sd(model), step=tr.step, epoch=tr.epoch, min_loss=tr.min_loss,
                           ckpt_keys=sorted(ckpt), ckpt_epoch=ckpt["epoch"], ckpt_step=ckpt["step"],
                           msg=tr._eval_metrics_str(seen[-1])))
    # 2. frozen first layer, cosine schedule, separate weight decay for the normalisation parameters, NaN skipping
    model = cls_model()
    data = cls_batches(5, 3)
    tr = T.ClassificationTrainer(model, data, cls_batches(2, 4), FlakyCrossEntropy(bad=3),
                                 torch.optim.SGD(model.parameters(), lr=1e-2, momentum=0.9, weight_decay=1e-2), gpu=None,
                                 output_file=output_file, skip_nan_loss=True)
    tr.fit_n_epochs(1, 5e-2, freeze_until="0", sched_type="cosine", norm_weight_decay=0.0)
    record("cls_frozen_cosine", dict(state=sd(model), groups=[(len(g["params"]), g["weight_decay"]) for g in tr.optimizer.param_groups],
                                     frozen=[n for n, p in model.named_parameters() if not p.requires_grad], step=tr.step,
                                     metrics=tr.evaluate()))
    # 3. binary classification
    model = cls_model(1)
    tr = T.BinaryClassificationTrainer(model, cls_batches(4, 5, binary=True), cls_batches(2, 6, binary=True), nn.BCEWithLogitsLoss(),
                                       torch.optim.Adam(model.parameters(), lr=1e-3), gpu=None, output_file=output_file)
    tr.fit_n_epochs(1, 1e-2)
    m = tr.evaluate()
    record("binary", dict(state=sd(model), metrics=m, msg=tr._eval_metrics_str(m)))
    # 4. segmentation
    model = seg_model()
    tr = T.SegmentationTrainer(model, seg_batches(3, 7), seg_batches(2, 8), nn.CrossEntropyLoss(ignore_index=255),
                               torch.optim.Adam(model.parameters(), lr=1e-3), gpu=None, output_file=output_file,
                               num_classes=5)
    tr.fit_n_epochs(1, 1e-2)
    m = tr.evaluate()
    record("segmentation", dict(state=sd(model), metrics=m, msg=tr._eval_metrics_str(m)))
    # 5. detection: training on the model's own loss dict, evaluation metrics on canned detections, assign_iou on its own
    loader, detections = det_data()
    model = FixedDetector(detections)
    tr = T.DetectionTrainer(model, loader, loader, None, torch.optim.SGD(model.parameters(), lr=1e-2), gpu=None,
                            output_file=output_file)
    tr.fit_n_epochs(1, 1e-2)
    m = tr.evaluate()
    assign_iou = getattr(T, "assign_iou", None) or __import__(T.__name__ + ".detection", fromlist=["assign_iou"]).assign_iou
    gi, pi = assign_iou(loader[0][1][1]["boxes"], torch.tensor([[0.2, 0.2, 0.6, 0.6], [0.9, 0.9, 1.0, 1.0]]))
    record("detection", dict(w=float(model.w), metrics=m, msg=tr._eval_metrics_str(m), assign=([int(i) for i in gi], [int(i) for i in pi]),
                             msg_none=tr._eval_metrics_str({"loc_err": None, "clf_err": None, "det_err": None})))
    # 6. learning-rate finder and set-up check
    model = cls_model()
    tr = T.ClassificationTrainer(model, cls_batches(8, 9), cls_batches(2, 10), nn.CrossEntropyLoss(),
                                 torch.optim.Adam(model.parameters(), lr=1e-3), gpu=None, output_file=output_file)
    tr.find_lr(start_lr=1e-5, end_lr=1e-1, num_it=6)
    rec = dict(lrs=list(tr.lr_recorder), losses=list(tr.loss_recorder))
    tr.check_setup(lr=1e-3, num_it=4)
    rec["state_after_check"] = sd(model)
    try:
        tr.find_lr(num_it=100)
        rec["too_many"] = None
    except ValueError as e:
        rec["too_many"] = str(e)
    record("find_lr", rec)
