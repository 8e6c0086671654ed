"""The trainer CLASSES of SURVEY §8 f1 (reference holocron/trainer: Trainer.fit_n_epochs / find_lr / check_setup / save / load,
ClassificationTrainer, BinaryClassificationTrainer, SegmentationTrainer, DetectionTrainer, assign_iou) against golden runs of
the UNMODIFIED reference classes on the same scenarios (tests/_trainer_cases.py, tests/golden/make_golden.py --trainers):
stock-torch models and optimizers on the CPU, i.e. the host-driven path of holocron_b200.trainer.Trainer - every epoch's
evaluation metrics, the final parameters, the step / epoch counters, the checkpoint layout, the printed summaries, parameter
groups, frozen layers, the learning-rate finder's recordings. The device-driven path (TrainStep) is covered on the GPU by
tests/test_gpu_trainer.py."""
import math

import pytest
import torch

import holocron_b200 as hb

import _trainer_cases as cases
from conftest import load_golden


def _close(a, b, tol=1e-5):
    if a is None or b is None:
        assert a is b
        return
    assert math.isclose(a, b, rel_tol=tol, abs_tol=tol), (a, b)


def _same_state(got, want, tol=1e-5):
    assert list(got) == list(want)
    for k in want:
        g, w = got[k].double(), want[k].double()
        assert g.shape == w.shape and float((g - w).norm()) <= tol * (1.0 + float(w.norm())), k


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    ours = {}
    cases.run_scenarios(hb.trainer, lambda tag, rec: ours.__setitem__(tag, rec), str(tmp_path_factory.mktemp("trainers") / "ckpt.pth"))
    return ours, load_golden("trainers")


def test_classification_fit_n_epochs_matches_reference(runs):
    ours, ref = runs
    a, b = ours["cls_fit"], ref["cls_fit"]
    assert len(a["metrics"]) == len(b["metrics"]) == 2
    for ma, mb in zip(a["metrics"], b["metrics"]):
        assert set(ma) == set(mb) == {"val_loss", "acc1", "acc5"}
        for k in mb:
            _close(ma[k], mb[k])
    _same_state(a["state"], b["state"])
    assert (a["step"], a["epoch"]) == (b["step"], b["epoch"]) == (12, 2)
    _close(a["min_loss"], b["min_loss"])
    assert a["ckpt_keys"] == b["ckpt_keys"] == ["epoch", "min_loss", "model", "step"]
    assert (a["ckpt_epoch"], a["ckpt_step"]) == (b["ckpt_epoch"], b["ckpt_step"])
    assert a["msg"] == b["msg"]


def test_frozen_layers_param_groups_cosine_and_nan_skip_match_reference(runs):
    ours, ref = runs
    a, b = ours["cls_frozen_cosine"], ref["cls_frozen_cosine"]
    assert a["groups"] == b["groups"] and a["frozen"] == b["frozen"] == ["0.weight"] and a["step"] == b["step"] == 5
    _same_state(a["state"], b["state"])
    for k in b["metrics"]:
        _close(a["metrics"][k], b["metrics"][k])


def test_binary_and_segmentation_trainers_match_reference(runs):
    ours, ref = runs
    for tag in ("binary", "segmentation"):
        a, b = ours[tag], ref[tag]
        _same_state(a["state"], b["state"])
        assert set(a["metrics"]) == set(b["metrics"])
        for k in b["metrics"]:
            _close(a["metrics"][k], b["metrics"][k])
        assert a["msg"] == b["msg"]


def test_detection_trainer_and_assign_iou_match_reference(runs):
    ours, ref = runs
    a, b = ours["detection"], ref["detection"]
    _close(a["w"], b["w"])
    assert set(a["metrics"]) == set(b["metrics"]) == {"loc_err", "clf_err", "det_err", "val_loss"}
    for k in b["metrics"]:
        _close(a["metrics"][k], b["metrics"][k])
    assert a["assign"] == b["assign"] and a["msg"] == b["msg"] and a["msg_none"] == b["msg_none"]


def test_lr_finder_and_check_setup_match_reference(runs):
    ours, ref = runs
    a, b = ours["find_lr"], ref["find_lr"]
    assert len(a["lrs"]) == len(b["lrs"]) == len(a["losses"]) == 6
    for x, y in zip(a["lrs"] + a["losses"], b["lrs"] + b["losses"]):
        _close(x, y)
    _same_state(a["state_after_check"], b["state_after_check"])
    assert a["too_many"] == b["too_many"] is not None


def test_trainer_errors_and_checkpoint_round_trip(tmp_path):
    model = cases.cls_model()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    tr = hb.trainer.ClassificationTrainer(model, cases.cls_batches(2, 1), cases.cls_batches(1, 2), torch.nn.CrossEntropyLoss(), opt,
                                          gpu=None, output_file=str(tmp_path / "ckpt.pth"))
    with pytest.raises(ValueError):
        tr.fit_n_epochs(1, 1e-3, sched_type="linear")
    with pytest.raises(AssertionError):
        tr.plot_recorder()
    for p in model.parameters():
        p.requires_grad_(False)
    with pytest.raises(AssertionError):
        tr._reset_opt(1e-3)
    for p in model.parameters():
        p.requires_grad_(True)
    tr.epoch, tr.step, tr.min_loss = 3, 17, 0.25
    tr.save(str(tmp_path / "ckpt.pth"))
    other = hb.trainer.ClassificationTrainer(cases.cls_model(), [], [], torch.nn.CrossEntropyLoss(),
                                             torch.optim.Adam(model.parameters(), lr=1e-3), gpu=None)
    other.load(torch.load(tmp_path / "ckpt.pth", map_location="cpu"))
    assert (other.start_epoch, other.epoch, other.step, other.min_loss) == (3, 3, 17, 0.25)
    if not torch.cuda.is_available():
        with pytest.raises(AssertionError):
            hb.trainer.ClassificationTrainer(model, [], [], torch.nn.CrossEntropyLoss(), opt, gpu=0)
    # NaN tolerance of the host-driven path (reference core.py:153-159)
    flaky = cases.FlakyCrossEntropy(bad=1)
    flaky.forward = lambda out, target: torch.nn.functional.cross_entropy(out, target) * float("nan")
    tr = hb.trainer.ClassificationTrainer(cases.cls_model(), cases.cls_batches(4, 1), cases.cls_batches(1, 2), flaky,
                                          torch.optim.SGD(model.parameters(), lr=1e-3), gpu=None, skip_nan_loss=True, nan_tolerance=2)
    tr._reset_scheduler(1e-3, 1, "cosine")
    with pytest.raises(ValueError, match="NaN or inf for more than 2 steps"):
        tr._fit_epoch()


# ------------------------------------------------------------------------------------------------------------------------
# The flow of the reference's own trainer test (tests/test_trainer.py:79-147 `_test_trainer`, :150-270) on this package's classes,
# with real DataLoaders over the reference's mock datasets (host-driven path: stock model and optimizer on the CPU).
class _MockCls(torch.utils.data.Dataset):
    def __init__(self, n, target=0):
        self.n, self.target = n, target

    def __getitem__(self, idx):
        return torch.rand((3, 32, 32)), self.target

    def __len__(self):
        return self.n


class _MockSeg(_MockCls):
    def __getitem__(self, idx):
        return torch.rand((3, 32, 32)), torch.zeros((32, 32), dtype=torch.long)


def _reference_trainer_flow(learner, num_it, ref_param, freeze_until=None, lr=1e-3):
    T = hb.trainer
    T.freeze_model(learner.model.train(), freeze_until)
    learner._reset_opt(lr)
    learner.save(learner.output_file)
    checkpoint = torch.load(learner.output_file, map_location="cpu")
    model_w = learner.model.state_dict()[ref_param].clone()
    learner.check_setup(freeze_until, num_it=num_it, block=False)
    learner.load(checkpoint)
    with pytest.raises(AssertionError):
        learner.plot_recorder(block=False)
    with pytest.raises(ValueError):
        learner.find_lr(freeze_until, num_it=num_it + 1)
    for p in learner.model.parameters():
        p.requires_grad_(False)
    with pytest.raises(AssertionError):
        learner._set_params()
    for p in learner.model.parameters():
        p.requires_grad_(True)
    learner.find_lr(freeze_until, norm_weight_decay=5e-4, num_it=num_it)
    assert len(learner.lr_recorder) == len(learner.loss_recorder) > 0
    learner.load(checkpoint)
    with pytest.raises(ValueError):
        learner.fit_n_epochs(1, 1e-3, freeze_until, sched_type="my_scheduler")
    learner.fit_n_epochs(1, 1e-3, freeze_until)
    assert not torch.equal(learner.model.state_dict()[ref_param], model_w)
    learner.load(checkpoint)
    learner.fit_n_epochs(1, 1e-3, freeze_until, sched_type="cosine")
    assert not torch.equal(learner.model.state_dict()[ref_param], model_w)
    # gradient accumulation: the update happens every second batch
    learner.load(checkpoint)
    assert torch.equal(learner.model.state_dict()[ref_param], model_w)
    learner.model.train()
    learner.gradient_acc = 2
    learner._reset_opt(lr)
    it = iter(learner.train_loader)
    assert all(torch.all(p.grad == 0) for p in learner.model.parameters() if p.requires_grad and p.grad is not None)
    x, target = learner.to_cuda(*next(it))
    learner._backprop_step(learner._get_loss(x, target))
    assert torch.equal(learner.model.state_dict()[ref_param], model_w)
    assert all(torch.any(p.grad != 0) for p in learner.model.parameters() if p.requires_grad and p.grad is not None)
    x, target = learner.to_cuda(*next(it))
    learner._backprop_step(learner._get_loss(x, target))
    assert not torch.equal(learner.model.state_dict()[ref_param], model_w)
    assert all(torch.all(p.grad == 0) for p in learner.model.parameters() if p.requires_grad and p.grad is not None)


@pytest.mark.parametrize("amp", [False, True])
def test_reference_trainer_test_flow_classification(tmp_path, amp):
    from torch import nn
    from torch.utils.data import DataLoader
    torch.manual_seed(0)
    num_it, batch_size = 10, 8
    model = nn.Sequential(nn.Conv2d(3, 32, 3), nn.ReLU(inplace=True), nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(32, 5))
    loader = DataLoader(_MockCls(num_it * batch_size), batch_size=batch_size)
    opt = torch.optim.Adam(model.parameters())
    with pytest.raises(ValueError if torch.cuda.is_available() else AssertionError):
        hb.trainer.ClassificationTrainer(model, loader, loader, nn.CrossEntropyLoss(), opt, gpu=7)
    learner = hb.trainer.ClassificationTrainer(model, loader, loader, nn.CrossEntropyLoss(), opt, output_file=str(tmp_path / "tmp.pt"),
                                               gpu=None, amp=amp)
    learner.plot_top_losses((0, 0, 0), (1, 1, 1), [str(i) for i in range(5)], num_samples=6, block=False)
    top = learner.top_losses
    assert top["images"].shape == (6, 3, 32, 32) and torch.all(top["losses"][:-1] >= top["losses"][1:]) and set(top) >= {"preds", "probs", "targets"}
    with pytest.raises(AssertionError):
        learner.plot_top_losses((0, 0, 0), (1, 1, 1))
    assert learner.criterion.reduction == "mean"
    _reference_trainer_flow(learner, num_it, "4.weight")
    # fewer than 5 classes: no top-5 accuracy (reference tests/test_trainer.py:192-202)
    few = nn.Sequential(nn.Conv2d(3, 8, 3), nn.ReLU(inplace=True), nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(8, 3))
    assert hb.trainer.ClassificationTrainer(few, loader, loader, nn.CrossEntropyLoss(), torch.optim.Adam(few.parameters())).evaluate()["acc5"] == 0


def test_reference_trainer_test_flow_segmentation_and_binary(tmp_path):
    from torch import nn
    from torch.utils.data import DataLoader
    torch.manual_seed(0)
    model = nn.Sequential(nn.Conv2d(3, 16, 3, padding=1), nn.ReLU(inplace=True), nn.Conv2d(16, 5, 3, padding=1))
    loader = DataLoader(_MockSeg(6 * 4), batch_size=4)
    learner = hb.trainer.SegmentationTrainer(model, loader, loader, nn.CrossEntropyLoss(), torch.optim.Adam(model.parameters()),
                                             num_classes=5, output_file=str(tmp_path / "tmp.pt"), gpu=None)
    _reference_trainer_flow(learner, 6, "2.weight")
    # binary targets given as (N, 1) float columns or as plain integers (reference tests/test_trainer.py:205-230)
    bmodel = nn.Sequential(nn.Conv2d(3, 8, 3), nn.ReLU(inplace=True), nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(8, 1))
    for target in (torch.zeros((1,)), 0):
        loader = DataLoader(_MockCls(16, target), batch_size=8)
        tr = hb.trainer.BinaryClassificationTrainer(bmodel, loader, loader, nn.BCEWithLogitsLoss(), torch.optim.Adam(bmodel.parameters()),
                                                    amp=True)
        assert 0 <= tr.evaluate()["acc"] <= 1
    tr.plot_top_losses((0, 0, 0), (1, 1, 1), num_samples=4, block=False)
    assert tr.top_losses["losses"].shape == (4,)
