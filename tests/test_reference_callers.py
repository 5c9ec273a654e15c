"""The drop-in boundary under the reference's OWN callers.  Applies the swap of INTEGRATION.md --
`yolov6_b200.build_model` where the reference calls `yolov6.models.yolo.build_model` -- and checks the result against
what those callers saw of the reference's models (tests/golden/callers.json, minted from the unmodified reference by
tests/golden/make_golden_callers.py): the configs/*.py that `Config.fromfile` reads, the state_dict layout, the parameter
groups of `build_optimizer` (solver/build.py:10-33), the decay of `ModelEMA` (utils/ema.py) and the layouts of
pickled-module checkpoints (utils/checkpoint.py:22-32).  CPU only: nothing here runs a network forward (that needs the
CUDA engine; see tests/test_gpu_*.py)."""
import copy
import types

import pytest
import torch
import torch.nn as nn

from conftest import golden_json


@pytest.fixture(scope="module")
def ref():
    return golden_json("callers.json")


def load_cfg(ref, name):
    """The golden config in the shape of the reference's `Config`: attributes at the top, dicts below."""
    c = ref[name]["config"]
    return types.SimpleNamespace(model=copy.deepcopy(c["model"]), solver=types.SimpleNamespace(**c["solver"]),
                                 training_mode=c["training_mode"])


def optimizer_groups(model):
    """The grouping rule of the reference's `build_optimizer`, walking `model.modules()`: every module's bias Parameter
    goes to the bias group; a BatchNorm2d's weight to the BN group; any other module's weight Parameter to the decayed
    group."""
    bnw, w, b = [], [], []
    for v in model.modules():
        if isinstance(getattr(v, "bias", None), nn.Parameter):
            b.append(v.bias)
        if isinstance(v, nn.BatchNorm2d):
            bnw.append(v.weight)
        elif isinstance(getattr(v, "weight", None), nn.Parameter):
            w.append(v.weight)
    return bnw, w, b


def build_optimizer(cfg, model):
    """SGD-nesterov over the three groups with the solver's hyper-parameters, as the reference builds it."""
    bnw, w, b = optimizer_groups(model)
    s = cfg.solver
    opt = torch.optim.SGD(bnw, lr=s.lr0, momentum=s.momentum, nesterov=True)
    opt.add_param_group({"params": w, "weight_decay": s.weight_decay})
    opt.add_param_group({"params": b})
    return opt


@pytest.mark.parametrize("name", ["yolov6n", "yolov6s", "yolov6m", "yolov6l6"])
def test_build_model_from_reference_config_and_optimizer_groups(ref, name):
    from yolov6_b200.model import build_model
    cfg = load_cfg(ref, name)
    ours = build_model(cfg, 80, torch.device("cpu"))
    theirs = ref[name]["state"]
    sd_o = ours.state_dict()
    assert sorted(sd_o) == sorted(k for k, *_ in theirs)   # same keys (registration order differs, loading is by key)
    assert all(list(sd_o[k].shape) == shape and str(sd_o[k].dtype) == f"torch.{dt}" for k, shape, dt, _ in theirs)
    params_o = {n for n, _ in ours.named_parameters()}
    assert params_o == {k for k, _, _, is_param in theirs if is_param}
    assert ours.stride.float().tolist() == ref[name]["stride"]
    # the reference's optimizer builder sees the same three parameter groups on our model as on its own
    name_of = {id(p): n for n, p in ours.named_parameters()}
    opt = build_optimizer(cfg, ours)
    want = [sorted(theirs[i][0] for i in g["params"]) for g in ref[name]["groups"]]
    assert [sorted(name_of[id(p)] for p in g["params"]) for g in opt.param_groups] == want
    for g, gw in zip(opt.param_groups, ref[name]["groups"]):
        assert (g["lr"], g["momentum"], g["nesterov"], g["weight_decay"]) == (gw["lr"], gw["momentum"], gw["nesterov"], gw["weight_decay"])
    if name == "yolov6s":
        print("yolov6s parameter groups (bn weights, weights, biases):", [len(g["params"]) for g in opt.param_groups])
    # an optimizer step over zero gradients is a weight-decay-only update and runs through the views of the flat state
    for p in ours.parameters():
        if p.requires_grad:
            p.grad = torch.zeros_like(p)
    key = "backbone.ERBlock_2.0." + ("rbr_dense" if name != "yolov6l6" else "block") + ".conv.weight"
    before = ours.state_dict()[key].clone()
    opt.step()
    after = ours.state_dict()[key]
    # nesterov, first step: g = wd*p, buf = g, p -= lr * (g + momentum * buf)
    s = cfg.solver
    assert torch.allclose(after, before * (1 - s.lr0 * s.weight_decay * (1 + s.momentum)), rtol=1e-5, atol=1e-9)


def test_model_ema_over_the_drop_in_model(ref):
    """`ModelEMA` keeps `deepcopy(model).eval()` and, per update, blends every floating-point state_dict entry in place;
    `update_attr` copies plain attributes over."""
    from yolov6_b200.model import build_model
    m = build_model(load_cfg(ref, "yolov6n"), 80, torch.device("cpu"))
    ema = copy.deepcopy(m).eval()
    for p in ema.parameters():
        p.requires_grad_(False)
    assert type(ema) is type(m) and not ema.training
    with torch.no_grad():
        for p in m.parameters():
            p.add_(1.0)
    d = ref["ema_decay_first_update"]
    with torch.no_grad():
        msd = m.state_dict()
        for k, item in ema.state_dict().items():
            if item.dtype.is_floating_point:
                item *= d
                item += (1 - d) * msd[k].detach()
    k = "backbone.stem.rbr_dense.conv.weight"
    want = (m.state_dict()[k] - 1.0) * d + (1 - d) * m.state_dict()[k]
    assert torch.allclose(ema.state_dict()[k], want, rtol=1e-6, atol=1e-8)
    for a in ("nc", "names", "stride"):                    # core/engine.py:186
        if a in m.__dict__:
            setattr(ema, a, m.__dict__[a])


class RefLayout(nn.Module):
    """A module with the reference's state_dict layout (parameters and buffers under the same dotted keys) and its
    `detect.nc`: what `from_reference` reads of an unpickled `yolov6.models.yolo.Model`."""

    def __init__(self, rows, nc=80):
        super().__init__()
        for key, shape, dt, is_param in rows:
            *path, leaf = key.split(".")
            mod = self
            for p in path:
                if not hasattr(mod, p):
                    mod.add_module(p, nn.Module())
                mod = getattr(mod, p)
            t = torch.zeros(shape, dtype=getattr(torch, dt))
            if is_param:
                mod.register_parameter(leaf, nn.Parameter(t))
            else:
                mod.register_buffer(leaf, t)
        self.detect.nc = nc


def test_pickled_reference_checkpoint_converts(ref, tmp_path):
    """checkpoint.py:22-32 unpickles a module of the reference; `yolov6_b200.checkpoint` turns it into the kernel-backed model."""
    from yolov6_b200.checkpoint import from_reference, load_checkpoint
    from yolov6_b200.model import Model
    theirs = RefLayout(ref["yolov6s"]["state"])
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for k, v in theirs.state_dict().items():
            if v.dtype.is_floating_point:
                v.copy_(torch.rand(v.shape, generator=g) * 1.01)
    path = tmp_path / "last_ckpt.pt"
    torch.save({"model": copy.deepcopy(theirs).half(), "ema": None, "epoch": 3}, path)   # Trainer saves half (engine.py:185)
    m = load_checkpoint(str(path), map_location="cpu")
    assert isinstance(m, Model) and not m.training
    sd_t = theirs.state_dict()
    for k, a in m.state_dict().items():
        assert torch.allclose(a.float(), sd_t[k].half().float()), k
    m2 = from_reference(theirs.train())
    assert m2.training and m2.detect.nc == 80
    deployed = RefLayout(ref["yolov6s"]["deploy"]).eval()   # fuse_model + switch_to_deploy: BN folded, rbr_reparam
    with pytest.raises(RuntimeError):
        from_reference(deployed)
