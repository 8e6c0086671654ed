"""On-disk / wire formats of SURVEY §8 f4 on the CPU (no kernels involved: pure host logic):

  * the HF-hub repository layout of reference models/utils.py:146-175 (config.json + pytorch_model.bin), written by
    ``save_hf_hub_folder`` and read back by ``model_from_hf_hub`` through a stubbed ``hf_hub_download`` (no network);
    the same two files match what the UNMODIFIED reference's ``model_from_hf_hub`` reads (tests/golden/cross_checks.pt);
  * ``load_pretrained_params`` (reference models/utils.py:89-113) from a ``file://`` URL incl. key filter / replacement, and
    the factories' ``checkpoint=Checkpoint(...)`` argument;
  * ``clean_checkpoint`` (reference references/clean_checkpoint.py): Trainer checkpoint -> bare legacy-serialised state_dict."""
import hashlib
import json
import zipfile

import pytest
import torch

import holocron_b200 as hb
from holocron_b200.models import checkpoints as CK
from holocron_b200.models import utils as U
from conftest import load_golden


def _stub_hub(monkeypatch, folder, repo):
    import huggingface_hub

    def fake_download(repo_id, filename, **kwargs):
        assert repo_id == repo
        return str(folder / filename)
    monkeypatch.setattr(huggingface_hub, "hf_hub_download", fake_download)


def test_hf_hub_folder_round_trip(tmp_path, monkeypatch):
    torch.manual_seed(3)
    model = hb.models.repvgg_a0(num_classes=10)
    classes = [f"class_{i}" for i in range(10)]
    folder = U.save_hf_hub_folder(model, tmp_path / "hub", "repvgg_a0", classes)
    cfg = json.loads((folder / "config.json").read_text())
    assert cfg == {"arch": "repvgg_a0", "classes": classes, "input_shape": [3, 224, 224], "mean": [0.485, 0.456, 0.406],
                   "std": [0.229, 0.224, 0.225]}
    _stub_hub(monkeypatch, folder, "frgfm/repvgg_a0")
    loaded = U.model_from_hf_hub("frgfm/repvgg_a0")
    assert type(loaded) is type(model) and loaded.default_cfg == cfg
    sd, sl = model.state_dict(), loaded.state_dict()
    assert list(sd) == list(sl) and all(torch.equal(sd[k], sl[k]) for k in sd)


def test_hf_hub_folder_is_readable_by_the_reference(tmp_path, monkeypatch):
    """Interoperability both ways, against the reference's hub loader as recorded in tests/golden/cross_checks.pt
    (make_golden.py --cross): a folder written here names an architecture the reference registers and holds exactly the
    parameter names, shapes and dtypes its strict ``load_state_dict`` accepts, and a folder holding a state_dict in the
    reference's layout loads here."""
    ref = load_golden("cross_checks")["hub"]
    torch.manual_seed(4)
    ours = hb.models.rexnet1_0x(num_classes=ref["num_classes"])
    classes = [str(i) for i in range(ref["num_classes"])]
    folder = U.save_hf_hub_folder(ours, tmp_path / "hub", "rexnet1_0x", classes)
    # what the reference's model_from_hf_hub reads: cfg["arch"] from its registry, len(cfg["classes"]), the state_dict
    cfg = json.loads((folder / "config.json").read_text())
    assert cfg["arch"] == ref["arch"] and cfg["arch"] in ref["registry"] and len(cfg["classes"]) == ref["num_classes"]
    sd = torch.load(folder / "pytorch_model.bin", map_location="cpu")
    assert [(k, tuple(v.shape), v.dtype) for k, v in sd.items()] == ref["layout"]
    # and back: a state_dict in the reference's layout, seeded values
    g = torch.Generator().manual_seed(5)
    theirs = {k: (torch.rand(shape, generator=g) * 2 - 1).to(dtype) if dtype.is_floating_point else
              torch.randint(0, 100, shape, generator=g).to(dtype) for k, shape, dtype in ref["layout"]}
    torch.save(theirs, folder / "pytorch_model.bin")
    _stub_hub(monkeypatch, folder, "frgfm/rexnet1_0x")
    back = U.model_from_hf_hub("frgfm/rexnet1_0x")
    assert all(torch.equal(v, back.state_dict()[k]) for k, v in theirs.items())


def _checkpoint(url, arch):
    return CK.Checkpoint(
        evaluation=CK.Evaluation(dataset=CK.Dataset.IMAGENETTE, results={CK.Metric.TOP1_ACC: 0.9, CK.Metric.TOP5_ACC: 0.99}),
        meta=CK.LoadingMeta(url=url, sha256="0" * 64, size=0, num_params=0, arch=arch, categories=[str(i) for i in range(10)]),
        pre_processing=CK.PreProcessing(input_shape=(3, 224, 224), mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)),
        recipe=CK.TrainingRecipe(commit=None, script="references/classification/train.py", args=None))


def test_factories_load_a_checkpoint_from_a_file_url(tmp_path, monkeypatch):
    monkeypatch.setenv("TORCH_HOME", str(tmp_path / "torch_home"))
    torch.manual_seed(5)
    src = hb.models.resnet18(num_classes=10)
    path = tmp_path / "resnet18_224-deadbeef.pth"
    torch.save(src.state_dict(), path)
    ckpt = _checkpoint(path.as_uri(), "resnet18")
    torch.manual_seed(6)
    model = hb.models.resnet18(checkpoint=ckpt, num_classes=10)
    assert model.default_cfg is ckpt
    assert all(torch.equal(v, model.state_dict()[k]) for k, v in src.state_dict().items())
    # pretrained without a checkpoint: the released-checkpoint table is not shipped (no network)
    with pytest.raises(NotImplementedError):
        hb.models.resnet18(pretrained=True)
    with pytest.raises(TypeError):
        hb.models.repvgg_a0(checkpoint="repvgg_a0.pth")
    assert hb.models.darknet19(num_classes=10).default_cfg is None
    assert CK._handle_legacy_pretrained(True, None, ckpt) is ckpt and CK._handle_legacy_pretrained(False, None, ckpt) is None


def test_load_pretrained_params_filters_and_renames_keys(tmp_path, monkeypatch, caplog):
    """The detectors' backbone loading path (reference yolo.py:381-392): classification checkpoint -> 'features.' keys only,
    prefix stripped."""
    monkeypatch.setenv("TORCH_HOME", str(tmp_path / "torch_home"))
    torch.manual_seed(7)
    clf = hb.models.darknet19(num_classes=10)
    path = tmp_path / "darknet19.pth"
    torch.save(clf.state_dict(), path)
    det = hb.models.yolov2(num_classes=20)
    before = det.backbone.state_dict()["stem.0.weight"].clone()
    U.load_pretrained_params(det.backbone, path.as_uri(), progress=False, key_replacement=("features.", ""),
                             key_filter="features.")
    assert not torch.equal(before, det.backbone.state_dict()["stem.0.weight"])
    assert all(torch.equal(v, clf.features.state_dict()[k]) for k, v in det.backbone.state_dict().items())
    with caplog.at_level("WARNING"):
        U.load_pretrained_params(det.backbone, None)
    assert "Invalid model URL" in caplog.text


def test_clean_checkpoint_writes_the_released_format(tmp_path):
    torch.manual_seed(8)
    model = hb.models.repvgg_a0(num_classes=10)
    train_ckpt = {"epoch": 3, "step": 120, "min_loss": 0.5, "model": model.state_dict(), "optimizer": {"state": {}},
                  "scheduler": None}
    src, dst = tmp_path / "checkpoint.pth", tmp_path / "repvgg_a0.pth"
    torch.save(train_ckpt, src)
    sha = U.clean_checkpoint(src, dst)
    assert sha == hashlib.sha256(dst.read_bytes()).hexdigest()
    assert not zipfile.is_zipfile(dst)                       # legacy serialisation, like the reference's releases
    state = torch.load(dst, map_location="cpu")
    assert list(state) == list(model.state_dict()) and all(torch.equal(v, model.state_dict()[k]) for k, v in state.items())
