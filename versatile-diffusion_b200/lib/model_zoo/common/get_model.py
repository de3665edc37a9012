"""Model registry with the reference's surface: get_model()(cfg) and @register(name)
(reference lib/model_zoo/common/get_model.py:37-104)."""
import importlib

import torch

from ...log_service import print_log

_TYPE_TO_MODULE = (("autoencoderkl", "autokl"), ("clip", "clip"), ("vd", "vd"), ("openai_unet", "openaimodel"),
                   ("optimus", "optimus"))


class _Registry(object):
    def __init__(self):
        self.model = {}

    def register(self, model, name):
        self.model[name] = model

    def __call__(self, cfg, verbose=True):
        t = cfg["type"] if isinstance(cfg, dict) else cfg.type
        for prefix, module in _TYPE_TO_MODULE:
            if t.startswith(prefix):
                importlib.import_module("lib.model_zoo." + module)
                break
        if t not in self.model:
            raise KeyError(f"model type '{t}' is outside the B200 hot-path build (registered: {sorted(self.model)})")
        args = cfg["args"] if isinstance(cfg, dict) else cfg.args
        net = self.model[t](**dict(args))
        get = cfg.get if hasattr(cfg, "get") else (lambda k, d=None: getattr(cfg, k, d))
        strict_sd = get("strict_sd", True)
        for key in ("ckpt", "pth"):
            path = get(key, None)
            if path is not None:
                sd = torch.load(path, map_location=get("map_location", "cpu"))
                net.load_state_dict(sd["state_dict"] if key == "ckpt" else sd, strict=strict_sd)
                if verbose:
                    print_log("Load {} from {}".format(key, path))
        if verbose:
            n = sum(p.numel() for p in net.parameters())
            print_log("Load {} with total {} parameters".format(t, n))
        return net


_instance = _Registry()


def get_model():
    """Singleton accessor, called as get_model()(cfg) like the reference."""
    return _instance


def register(name):
    def wrapper(class_):
        _instance.register(class_, name)
        return class_
    return wrapper
