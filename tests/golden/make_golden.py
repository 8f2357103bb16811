"""Pins the oracle against the reference itself and writes the golden fixtures replayed by tests/test_oracle_golden.py.

Run in the build container (needs /root/reference, which does NOT exist on the GPU box):
    python tests/golden/make_golden.py
For every model it (1) builds the *reference* module under a fixed seed, (2) checks that the host-side mirror constructor
of deeplearning_b200 produces a bit-identical state_dict under the same seed, (3) checks that the oracle restatement gives
bit-identical logits / loss / gradients / buffer updates on the same weights and input, and (4) stores small outputs.
"""
import importlib.util
import json
import os
import sys
import types

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)


def _shim(name, **attrs):
    if name not in sys.modules:
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _grad_norms(named_params):
    return {n: float(p.grad.double().norm()) for n, p in named_params}


def resnet50_fixture():
    from deeplearning_b200.classification.resnet.models.networks import resnet50 as mine_ctor
    from oracle.resnet import resnet_forward, train_step_grads

    ref_mod = _load(f"{REF}/classification/resnet/models/networks.py", "ref_resnet_networks")
    torch.manual_seed(0)
    ref = ref_mod.resnet50()
    torch.manual_seed(0)
    mine = mine_ctor()
    sr = {k: v.clone() for k, v in ref.state_dict().items()}  # frozen copy of the initial state
    sm = mine.state_dict()
    assert list(sr.keys()) == list(sm.keys()) and all(torch.equal(sr[k], sm[k]) for k in sr), "ctor init differs"
    x_eval = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
    ref.eval()
    with torch.no_grad():
        le = ref(x_eval)
        lo = resnet_forward({k: v.clone() for k, v in sr.items()}, x_eval, False)
    assert torch.equal(le, lo), "oracle eval forward differs from the reference"
    x = torch.randn(4, 3, 64, 64, generator=torch.Generator().manual_seed(2))
    y = torch.randint(0, 1000, (4,), generator=torch.Generator().manual_seed(3))
    st = {k: v.clone() for k, v in sr.items()}  # snapshot before the reference's train-mode forward updates the buffers
    ref.train()
    out = ref(x)
    loss = F.cross_entropy(out, y)
    loss.backward()
    lg, lo_loss, grads = train_step_grads(st, x, y)
    assert torch.equal(lg, out.detach()) and float(lo_loss) == float(loss.detach())
    for n, p in ref.named_parameters():
        assert torch.equal(p.grad, grads[n]), n
    s2 = ref.state_dict()
    for k in s2:
        if "running" in k or "num_batches" in k:
            assert torch.equal(s2[k], st[k]), k
    return {"init_abs_sum": {k: float(v.double().abs().sum()) for k, v in sr.items() if v.is_floating_point()},
            "eval_logits": le.clone(), "train_logits": out.detach().clone(), "train_loss": float(loss.detach()),
            "grad_norms": _grad_norms(ref.named_parameters()),
            "running_mean_bn1": s2["bn1.running_mean"].clone(), "running_var_layer4": s2["layer4.2.bn3.running_var"].clone(),
            "seeds": {"init": 0, "x_eval": 1, "x_train": 2, "labels": 3}, "shapes": {"x_eval": [2, 3, 64, 64], "x_train": [4, 3, 64, 64]}}


def mnist_fixture():
    from deeplearning_b200.classification.mnist.models.network import mnist_cnn, mnist_fcn
    from oracle.mnist import mnist_cnn_forward, mnist_fcn_forward

    _shim("torchsummary", summary=lambda *a, **k: None)
    ref_mod = _load(f"{REF}/classification/mnist/models/network.py", "ref_mnist_network")
    out = {}
    for name, ctor, ref_ctor, fwd in (("mnist_fcn", mnist_fcn, ref_mod.mnist_fcn, mnist_fcn_forward),
                                      ("mnist_cnn", mnist_cnn, ref_mod.mnist_cnn, mnist_cnn_forward)):
        torch.manual_seed(0)
        ref = ref_ctor(10)
        torch.manual_seed(0)
        mine = ctor(10)
        sr, sm = ref.state_dict(), mine.state_dict()
        assert list(sr.keys()) == list(sm.keys()) and all(torch.equal(sr[k], sm[k]) for k in sr), name
        x = torch.randn(64, 3, 28, 28, generator=torch.Generator().manual_seed(1))  # SURVEY D1: 3x28x28, not 1x28x28
        y = torch.randint(0, 10, (64,), generator=torch.Generator().manual_seed(2))
        lg = ref(x)
        loss = F.cross_entropy(lg, y)
        loss.backward()
        assert torch.equal(lg.detach(), fwd(sr, x)), name
        assert torch.equal(lg.detach(), mine(x).detach()), name
        out[name] = {"logits": lg.detach().clone(), "loss": float(loss.detach()), "grad_norms": _grad_norms(ref.named_parameters())}
    return out


def vit_fixture():
    from deeplearning_b200.classification.vision_transformer.vit_model import vit_base_patch16_224_in21k as mine_ctor
    from oracle.vit import train_step_grads, vit_forward

    ref_mod = _load(f"{REF}/classification/vision_transformer/vit_model.py", "ref_vit_model")
    out = {}
    for has_logits in (False, True):
        torch.manual_seed(0)
        ref = ref_mod.vit_base_patch16_224_in21k(num_classes=1000, has_logits=has_logits)
        torch.manual_seed(0)
        mine = mine_ctor(num_classes=1000, has_logits=has_logits)
        sr = {k: v.clone() for k, v in ref.state_dict().items()}
        sm = mine.state_dict()
        assert list(sr) == list(sm) and all(torch.equal(sr[k], sm[k]) for k in sr), "ViT ctor init differs"
        x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
        y = torch.randint(0, 1000, (2,), generator=torch.Generator().manual_seed(2))
        ref.eval()
        with torch.no_grad():
            le = ref(x)
            assert torch.equal(le, vit_forward(sr, x)), "oracle ViT forward differs from the reference"
        ref.train()
        lt = ref(x)
        loss = F.cross_entropy(lt, y)
        loss.backward()
        lg, lo, grads = train_step_grads(sr, x, y)
        assert torch.equal(lg, lt.detach()) and float(lo) == float(loss.detach())
        for n, p in ref.named_parameters():
            assert torch.equal(p.grad, grads[n]), n
        out[f"has_logits={has_logits}"] = {"init_abs_sum": {k: float(v.double().abs().sum()) for k, v in sr.items()},
                                           "eval_logits": le.clone(), "train_loss": float(loss.detach()),
                                           "grad_norms": _grad_norms(ref.named_parameters())}
    return out


def convnext_fixture():
    from deeplearning_b200.classification.convNext.models.networks import convnext_tiny as mine_ctor
    from oracle.convnext import convnext_forward, train_step_grads

    ref_mod = _load(f"{REF}/classification/convNext/models/networks.py", "ref_convnext_networks")
    torch.manual_seed(0)
    ref = ref_mod.convnext_tiny(1000)
    torch.manual_seed(0)
    mine = mine_ctor(1000)
    sr = {k: v.clone() for k, v in ref.state_dict().items()}
    sm = mine.state_dict()
    assert list(sr) == list(sm) and all(torch.equal(sr[k], sm[k]) for k in sr), "ConvNeXt ctor init differs"
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    y = torch.randint(0, 1000, (2,), generator=torch.Generator().manual_seed(2))
    ref.eval()
    with torch.no_grad():
        le = ref(x)
        assert torch.equal(le, convnext_forward(sr, x)), "oracle ConvNeXt forward differs from the reference"
    for mod in ref.modules():  # parity protocol (SURVEY 8c): stochastic depth off
        if hasattr(mod, "drop_path"):
            mod.drop_path = torch.nn.Identity()
    ref.train()
    lt = ref(x)
    loss = F.cross_entropy(lt, y)
    loss.backward()
    lg, lo, grads = train_step_grads(sr, x, y)
    assert torch.equal(lg, lt.detach()) and float(lo) == float(loss.detach())
    for n, p in ref.named_parameters():
        assert torch.equal(p.grad, grads[n]), n
    return {"init_abs_sum": {k: float(v.double().abs().sum()) for k, v in sr.items()}, "eval_logits": le.clone(),
            "train_loss": float(loss.detach()), "grad_norms": _grad_norms(ref.named_parameters())}


def swin_fixture():
    from deeplearning_b200.classification.swin_transformer.models.swin_transformer import SwinTransformer as mine_ctor
    from oracle.swin import swin_forward, train_step_grads

    class _DropPath(torch.nn.Module):  # timm is not installed: the three names the reference file imports from it
        def __init__(self, p=None):
            super().__init__()
            self.drop_prob = p

        def forward(self, x):
            return x

    _shim("timm")
    _shim("timm.models")
    _shim("timm.models.layers", DropPath=_DropPath, trunc_normal_=torch.nn.init.trunc_normal_,
          to_2tuple=lambda x: tuple(x) if isinstance(x, (tuple, list)) else (x, x))
    ref_mod = _load(f"{REF}/classification/swin_transformer/models/swin_transformer.py", "ref_swin_transformer")
    torch.manual_seed(0)
    ref = ref_mod.SwinTransformer(drop_path_rate=0.0)   # Swin-T defaults; parity protocol (SURVEY 8c): stochastic depth off
    torch.manual_seed(0)
    mine = mine_ctor(drop_path_rate=0.0)
    sr = {k: v.clone() for k, v in ref.state_dict().items()}
    sm = mine.state_dict()
    assert list(sr) == list(sm) and all(torch.equal(sr[k], sm[k]) for k in sr), "Swin ctor init differs"
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    y = torch.randint(0, 1000, (2,), generator=torch.Generator().manual_seed(2))
    ref.eval()
    with torch.no_grad():
        le = ref(x)
        assert torch.equal(le, swin_forward(sr, x)), "oracle Swin forward differs from the reference"
    ref.train()
    lt = ref(x)
    loss = F.cross_entropy(lt, y)
    loss.backward()
    lg, lo, grads = train_step_grads(sr, x, y)
    assert torch.equal(lg, lt.detach()) and float(lo) == float(loss.detach())
    for n, p in ref.named_parameters():
        assert torch.equal(p.grad, grads[n]), n
    return {"init_abs_sum": {k: float(v.double().abs().sum()) for k, v in sr.items()}, "eval_logits": le.clone(),
            "train_loss": float(loss.detach()), "grad_norms": _grad_norms(ref.named_parameters())}


class _ScriptedRand:
    """Replays a fixed sequence of uniforms through ``torch.rand`` (the only RNG call of the reference's drop_path)."""

    def __init__(self, us):
        self.us, self.i = us, 0

    def __enter__(self):
        self._orig = torch.rand

        def fake(*shape, **kw):
            shape = shape[0] if len(shape) == 1 and isinstance(shape[0], (tuple, list, torch.Size)) else shape
            u = self.us[self.i]
            self.i += 1
            return u.to(kw.get("dtype") or torch.float32).view(*shape)

        torch.rand = fake
        return self

    def __exit__(self, *exc):
        torch.rand = self._orig


def drop_entries(blocks_probs, us, per_block):
    """Oracle ``drop`` list for blocks with the given drop probabilities (``per_block`` drop_path applications each)."""
    out, i = [], 0
    for p in blocks_probs:
        for _ in range(per_block):
            if p and p > 0:
                keep = 1.0 - p
                out.append(((keep + us[i]).floor(), keep))
                i += 1
            else:
                out.append(None)
    return out, i


def _timm_drop_path_shim():
    """timm 0.4.12 ``DropPath`` (the version classification/swin_transformer/README.md:7-13 pins): the published rand/floor
    algorithm, identical to the drop_path function the ConvNeXt / ViT sub-projects carry."""

    class DropPath(torch.nn.Module):
        def __init__(self, drop_prob=None):
            super().__init__()
            self.drop_prob = drop_prob

        def forward(self, x):
            if self.drop_prob == 0. or not self.training:
                return x
            keep_prob = 1 - self.drop_prob
            shape = (x.shape[0],) + (1,) * (x.ndim - 1)
            random_tensor = keep_prob + torch.rand(shape, dtype=x.dtype, device=x.device)
            random_tensor.floor_()
            return x.div(keep_prob) * random_tensor

    return DropPath


def droppath_fixture():
    """Stochastic depth ON (the reference's real recipes: convnext_tiny 0.2, SwinTransformer() 0.1, ViT 0.1): the reference's
    train-mode forward/backward with torch.rand scripted == the oracle fed the same per-sample masks, bit for bit."""
    from oracle import convnext as oc, swin as osw, vit as ov

    B = 4
    x = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(11))
    y = torch.randint(0, 1000, (B,), generator=torch.Generator().manual_seed(12))
    us = [torch.rand(B, generator=torch.Generator().manual_seed(100 + i)) for i in range(64)]
    out = {"seeds": {"x": 11, "labels": 12, "u0": 100}, "batch": B}

    def run(ref, probs, per_block, oracle_grads, **kw):
        sr = {k: v.clone() for k, v in ref.state_dict().items()}
        ref.train()
        with _ScriptedRand(us) as sc:
            lt = ref(x)
            used = sc.i
        loss = F.cross_entropy(lt, y)
        loss.backward()
        drop, n = drop_entries(probs, us, per_block)
        assert n == used and used > 0, (n, used)
        assert any(e is not None and float(e[0].min()) == 0.0 for e in drop), "no sample was dropped: pick other seeds"
        lg, lo, grads = oracle_grads(sr, x, y, drop=drop, **kw)
        assert torch.equal(lg, lt.detach()) and float(lo) == float(loss.detach())
        for n_, p in ref.named_parameters():
            assert torch.equal(p.grad, grads[n_]), n_
        return {"train_loss": float(loss.detach()), "train_logits": lt.detach().clone(), "grad_norms": _grad_norms(ref.named_parameters()),
                "rand_calls": used}

    ref_mod = _load(f"{REF}/classification/convNext/models/networks.py", "ref_convnext_networks_dp")
    torch.manual_seed(0)
    ref = ref_mod.convnext_tiny(1000)          # drop_path_rate 0.2 hard-coded (networks.py:178)
    probs = [getattr(b.drop_path, "drop_prob", 0.0) for st in ref.stages for b in st]
    out["convnext_tiny"] = run(ref, probs, 1, oc.train_step_grads)

    ref_mod = _load(f"{REF}/classification/vision_transformer/vit_model.py", "ref_vit_model_dp")
    torch.manual_seed(0)
    ref = ref_mod.VisionTransformer(img_size=224, patch_size=16, embed_dim=768, depth=12, num_heads=12, representation_size=768,
                                    num_classes=1000, drop_path_ratio=0.1)
    probs = [getattr(b.drop_path, "drop_prob", 0.0) for b in ref.blocks]
    out["vit_b16"] = run(ref, probs, 2, ov.train_step_grads)

    sys.modules.pop("timm.models.layers", None)
    _shim("timm")
    _shim("timm.models")
    _shim("timm.models.layers", DropPath=_timm_drop_path_shim(), trunc_normal_=torch.nn.init.trunc_normal_,
          to_2tuple=lambda v: tuple(v) if isinstance(v, (tuple, list)) else (v, v))
    ref_mod = _load(f"{REF}/classification/swin_transformer/models/swin_transformer.py", "ref_swin_transformer_dp")
    torch.manual_seed(0)
    ref = ref_mod.SwinTransformer()            # class default drop_path_rate 0.1
    probs = [getattr(b.drop_path, "drop_prob", 0.0) for l in ref.layers for b in l.blocks]
    out["swin_tiny"] = run(ref, probs, 2, osw.train_step_grads)
    sys.modules.pop("timm.models.layers", None)
    return out


def resnet50_loops_fixture():
    """The reference's own ``evaluate`` and ``train_one_epoch`` (classification/resnet/utils.py) on its resnet50(), CPU fp32,
    with the running statistics calibrated on one batch first: their return values, and the check that the restated loops
    of oracle/train_loop.py return the same numbers bit for bit."""
    from oracle.resnet import resnet_forward
    from oracle.train_loop import evaluate, train_one_epoch

    _shim("matplotlib")
    _shim("matplotlib.pyplot")
    utils = _load(f"{REF}/classification/resnet/utils.py", "ref_resnet_utils")
    ref_mod = _load(f"{REF}/classification/resnet/models/networks.py", "ref_resnet_networks_loops")
    seeds = {"init": 0, "calib": 3, "batches": 5}
    torch.manual_seed(seeds["init"])
    state = {k: v.clone() for k, v in ref_mod.resnet50().state_dict().items()}
    xc = torch.randn(32, 3, 224, 224, generator=torch.Generator().manual_seed(seeds["calib"]))
    with torch.no_grad():
        resnet_forward(state, xc, train=True, momentum=1.0)
    g = torch.Generator().manual_seed(seeds["batches"])
    batches = [(torch.randn(8, 3, 224, 224, generator=g), torch.randint(0, 1000, (8,), generator=g)) for _ in range(2)]
    cpu, loss_fn = torch.device("cpu"), torch.nn.CrossEntropyLoss()
    out = {"seeds": seeds, "calib_batch": 32, "batch": 8, "steps": 2, "lr": 0.01, "momentum": 0.9, "weight_decay": 5e-5}
    loops = {"reference": (lambda m: utils.evaluate(m, batches, cpu, loss_fn, 0),
                           lambda m, opt: utils.train_one_epoch(m, batches, cpu, opt, loss_fn, 0)),
             "oracle": (lambda m: evaluate(m, batches, cpu, loss_fn),
                        lambda m, opt: train_one_epoch(m, batches, cpu, opt, loss_fn))}
    for which, (ev, tr) in loops.items():
        model = ref_mod.resnet50()
        model.load_state_dict(state)
        e = ev(model)
        opt = torch.optim.SGD(model.parameters(), lr=out["lr"], momentum=out["momentum"], weight_decay=out["weight_decay"])
        t = tr(model, opt)
        res = {"eval_loss": e[0], "eval_acc": e[1], "train_loss": t[0], "train_acc": t[1],
               "fc_weight_norm_after": float(model.fc.weight.detach().double().norm())}
        if which == "reference":
            out.update(res)
        else:
            assert res == {k: out[k] for k in res}, ("oracle loops differ from the reference's", res)
    return out


FIXTURES = {"resnet50": resnet50_fixture, "mnist": mnist_fixture, "vit_b16": vit_fixture, "convnext_tiny": convnext_fixture,
            "swin_tiny": swin_fixture, "droppath": droppath_fixture}
# plain numbers, kept in a JSON file of their own: {name: (fixture, file name)}
JSON_FIXTURES = {"resnet50_loops": (resnet50_loops_fixture, "resnet50_loops.json")}

if __name__ == "__main__":
    torch.set_num_threads(8)
    only = sys.argv[1:]   # e.g. `make_golden.py swin_tiny` refreshes one entry and keeps the others
    for name, (fn, fname) in JSON_FIXTURES.items():
        if not only or name in only:
            with open(os.path.join(HERE, fname), "w") as f:
                json.dump(fn(), f, indent=1)
                f.write("\n")
            print("golden fixture written:", os.path.join(HERE, fname))
    if not only or set(only) & set(FIXTURES):
        path = os.path.join(HERE, "classification_golden.pt")
        fx = torch.load(path, weights_only=False) if only else {}
        for name, fn in FIXTURES.items():
            if not only or name in only:
                fx[name] = fn()
        fx["torch"] = torch.__version__
        torch.save(fx, path)
        print("golden fixtures written:", path, os.path.getsize(path), "bytes")
