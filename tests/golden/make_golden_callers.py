"""tests/golden/make_golden_callers.py -- what the reference's own callers see of its models, for
tests/test_reference_callers.py.

Runs the UNMODIFIED reference (read-only, never copied) on CPU and stores, per configuration, in
tests/golden/callers.json:
  config  the model / solver part of configs/<name>.py as `Config.fromfile` reads it (plus training_mode)
  state   [key, shape, dtype, is_parameter] of `build_model(cfg, 80, cpu).state_dict()`, in its order
  stride  `model.stride`
  groups  the optimizer `build_optimizer(cfg, model)` (solver/build.py) makes: per parameter group the indices of its
          parameters into `state` and its hyper-parameters
  deploy  (yolov6s) the `state` rows after `fuse_model` + `switch_to_deploy` (the inferer's deploy order)
and the decay `ModelEMA` (utils/ema.py) applies at its first update.

    PYTHONPATH=tests/golden/refshim:<reference checkout>:. python tests/golden/make_golden_callers.py <reference checkout>
"""
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.abspath(sys.argv[1])
sys.path[:0] = [os.path.join(HERE, "refshim"), REF]
torch.cuda.is_available = lambda: False

from yolov6.models.yolo import build_model  # noqa: E402
from yolov6.solver.build import build_optimizer  # noqa: E402
from yolov6.utils.config import Config  # noqa: E402
from yolov6.utils.ema import ModelEMA  # noqa: E402
from yolov6.utils.torch_utils import fuse_model  # noqa: E402

NAMES = ["yolov6n", "yolov6s", "yolov6m", "yolov6l6"]
SOLVER_KEYS = ["optim", "lr0", "momentum", "weight_decay"]


def plain(v):
    if isinstance(v, dict):
        return {k: plain(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [plain(x) for x in v]
    return v


def state_rows(model):
    params = {n for n, _ in model.named_parameters()}
    return [[k, list(v.shape), str(v.dtype).replace("torch.", ""), k in params] for k, v in model.state_dict().items()]


def main():
    torch.manual_seed(0)
    out = {}
    for name in NAMES:
        cfg = Config.fromfile(os.path.join(REF, "configs", f"{name}.py"))
        mode = getattr(cfg, "training_mode", "repvgg")          # tools/train.py:99-100
        if not hasattr(cfg, "training_mode"):
            setattr(cfg, "training_mode", mode)
        model = build_model(cfg, 80, torch.device("cpu"))
        state = state_rows(model)
        index = {k: i for i, (k, *_rest) in enumerate(state)}
        name_of = {id(p): n for n, p in model.named_parameters()}
        opt = build_optimizer(cfg, model)
        groups = [{"params": [index[name_of[id(p)]] for p in g["params"]], "lr": g["lr"], "momentum": g["momentum"],
                   "nesterov": g["nesterov"], "weight_decay": g["weight_decay"]} for g in opt.param_groups]
        rec = {"config": {"training_mode": mode, "model": plain(dict(cfg.model)),
                          "solver": {k: cfg.solver[k] for k in SOLVER_KEYS}},
               "state": state, "stride": [float(s) for s in model.stride], "groups": groups}
        if name == "yolov6s":
            deployed = fuse_model(model.eval())
            for layer in deployed.modules():
                if hasattr(layer, "switch_to_deploy"):
                    layer.switch_to_deploy()
            rec["deploy"] = state_rows(deployed)
        out[name] = rec
    out["ema_decay_first_update"] = ModelEMA(torch.nn.Linear(1, 1)).decay(1)
    with open(os.path.join(HERE, "callers.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote", os.path.join(HERE, "callers.json"), os.path.getsize(os.path.join(HERE, "callers.json")), "bytes")


if __name__ == "__main__":
    main()
