"""The oracle replayed against the golden fixtures generated from the reference itself (tests/golden/make_golden.py).

The weights are re-created by the host-side mirror constructors under the recorded seed, so these tests pin three things at
once without /root/reference: constructor init == reference init, oracle forward/backward == reference, fixtures unchanged.
"""
import json
import os

import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
FX = torch.load(os.path.join(HERE, "golden", "classification_golden.pt"), weights_only=False)


def _close(a, b, tol=2e-4):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    assert float((a - b).abs().max()) <= tol * (1.0 + float(b.abs().max())), float((a - b).abs().max())


def test_resnet50_init_matches_reference():
    from deeplearning_b200.classification.resnet.models.networks import resnet50

    fx = FX["resnet50"]
    torch.manual_seed(fx["seeds"]["init"])
    sd = resnet50().state_dict()
    for k, v in fx["init_abs_sum"].items():
        assert abs(float(sd[k].double().abs().sum()) - v) <= 1e-9 * (1 + abs(v)), k


def test_resnet50_oracle_matches_reference_outputs():
    from deeplearning_b200.classification.resnet.models.networks import resnet50
    from oracle.resnet import resnet_forward, train_step_grads

    fx = FX["resnet50"]
    torch.manual_seed(fx["seeds"]["init"])
    state = {k: v.clone() for k, v in resnet50().state_dict().items()}
    x_eval = torch.randn(*fx["shapes"]["x_eval"], generator=torch.Generator().manual_seed(fx["seeds"]["x_eval"]))
    with torch.no_grad():
        _close(resnet_forward({k: v.clone() for k, v in state.items()}, x_eval, False), fx["eval_logits"])
    x = torch.randn(*fx["shapes"]["x_train"], generator=torch.Generator().manual_seed(fx["seeds"]["x_train"]))
    y = torch.randint(0, 1000, (x.shape[0],), generator=torch.Generator().manual_seed(fx["seeds"]["labels"]))
    logits, loss, grads = train_step_grads(state, x, y)
    _close(logits, fx["train_logits"])
    assert abs(float(loss) - fx["train_loss"]) < 1e-4
    for n, g in grads.items():
        ref = fx["grad_norms"][n]
        assert abs(float(g.double().norm()) - ref) <= 2e-3 * (ref + 1e-6), n
    _close(state["bn1.running_mean"], fx["running_mean_bn1"])
    _close(state["layer4.2.bn3.running_var"], fx["running_var_layer4"])


@pytest.mark.parametrize("name", ["mnist_fcn", "mnist_cnn"])
def test_mnist_plumbing_config(name):
    """BASELINE config 0: mnist net on CPU, synthetic 3x28x28 (SURVEY D1), bs=64 - constructor, oracle and a full step."""
    from deeplearning_b200.classification.mnist.models import network
    from oracle import mnist as om

    fx = FX["mnist"][name]
    torch.manual_seed(0)
    model = getattr(network, name)(10)
    x = torch.randn(64, 3, 28, 28, generator=torch.Generator().manual_seed(1))
    y = torch.randint(0, 10, (64,), generator=torch.Generator().manual_seed(2))
    fwd = om.mnist_fcn_forward if name == "mnist_fcn" else om.mnist_cnn_forward
    _close(fwd(model.state_dict(), x), fx["logits"])
    out = model(x)
    _close(out.detach(), fx["logits"])
    loss = F.cross_entropy(out, y)
    assert abs(float(loss.detach()) - fx["loss"]) < 1e-4
    loss.backward()
    for n, p in model.named_parameters():
        ref = fx["grad_norms"][n]
        assert abs(float(p.grad.double().norm()) - ref) <= 2e-3 * (ref + 1e-6), n
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-5)
    opt.step()
    assert float(F.cross_entropy(model(x), y)) < float(loss.detach())


@pytest.mark.parametrize("has_logits", [False, True])
def test_vit_b16_init_and_oracle_match_reference(has_logits):
    from deeplearning_b200.classification.vision_transformer.vit_model import vit_base_patch16_224_in21k
    from oracle.vit import train_step_grads, vit_forward

    fx = FX["vit_b16"][f"has_logits={has_logits}"]
    torch.manual_seed(0)
    state = {k: v.clone() for k, v in vit_base_patch16_224_in21k(num_classes=1000, has_logits=has_logits).state_dict().items()}
    for k, v in fx["init_abs_sum"].items():
        assert abs(float(state[k].double().abs().sum()) - v) <= 1e-9 * (1 + abs(v)), k
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    y = torch.randint(0, 1000, (2,), generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        _close(vit_forward(state, x), fx["eval_logits"])
    _, loss, grads = train_step_grads(state, x, y)
    assert abs(float(loss) - fx["train_loss"]) < 1e-4
    for n, g in grads.items():
        ref = fx["grad_norms"][n]
        assert abs(float(g.double().norm()) - ref) <= 2e-3 * (ref + 1e-6), n


def test_convnext_tiny_init_and_oracle_match_reference():
    from deeplearning_b200.classification.convNext.models.networks import convnext_tiny
    from oracle.convnext import convnext_forward, train_step_grads

    fx = FX["convnext_tiny"]
    torch.manual_seed(0)
    state = {k: v.clone() for k, v in convnext_tiny(1000).state_dict().items()}
    for k, v in fx["init_abs_sum"].items():
        assert abs(float(state[k].double().abs().sum()) - v) <= 1e-9 * (1 + abs(v)), k
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    y = torch.randint(0, 1000, (2,), generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        _close(convnext_forward(state, x), fx["eval_logits"])
    _, loss, grads = train_step_grads(state, x, y)
    assert abs(float(loss) - fx["train_loss"]) < 1e-3
    for n, g in grads.items():
        ref = fx["grad_norms"][n]
        assert abs(float(g.double().norm()) - ref) <= 2e-3 * (ref + 1e-6), n


def test_swin_tiny_init_and_oracle_match_reference():
    from deeplearning_b200.classification.swin_transformer.models.swin_transformer import SwinTransformer
    from oracle.swin import swin_forward, train_step_grads

    fx = FX["swin_tiny"]
    torch.manual_seed(0)
    state = {k: v.clone() for k, v in SwinTransformer(drop_path_rate=0.0).state_dict().items()}
    for k, v in fx["init_abs_sum"].items():
        assert abs(float(state[k].double().abs().sum()) - v) <= 1e-9 * (1 + abs(v)), k
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    y = torch.randint(0, 1000, (2,), generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        _close(swin_forward(state, x), fx["eval_logits"])
    _, loss, grads = train_step_grads(state, x, y)
    assert abs(float(loss) - fx["train_loss"]) < 1e-4
    for n, g in grads.items():
        ref = fx["grad_norms"][n]
        assert abs(float(g.double().norm()) - ref) <= 2e-3 * (ref + 1e-6), n


def _drop_entries(probs, per_block, batch, u0):
    """The oracle's ``drop`` list from the scripted uniforms of make_golden.droppath_fixture (seed u0 + call index)."""
    out, i = [], 0
    for p in probs:
        for _ in range(per_block):
            if p and p > 0:
                keep = 1.0 - p
                u = torch.rand(batch, generator=torch.Generator().manual_seed(u0 + i))
                out.append(((keep + u).floor(), keep))
                i += 1
            else:
                out.append(None)
    return out, i


@pytest.mark.parametrize("name", ["convnext_tiny", "vit_b16", "swin_tiny"])
def test_droppath_oracle_matches_reference(name):
    """Stochastic depth at the reference's own default rates (convnext_tiny 0.2, VisionTransformer(drop_path_ratio=0.1) with
    pre_logits, SwinTransformer() 0.1): the oracle fed the scripted per-sample masks reproduces the reference's loss /
    logits / gradient norms recorded by make_golden.py (there: bit-identical to the reference with torch.rand scripted)."""
    fx = FX["droppath"]
    B = fx["batch"]
    x = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(fx["seeds"]["x"]))
    y = torch.randint(0, 1000, (B,), generator=torch.Generator().manual_seed(fx["seeds"]["labels"]))
    torch.manual_seed(0)
    if name == "convnext_tiny":
        from deeplearning_b200.classification.convNext.models.networks import convnext_tiny
        from oracle.convnext import train_step_grads

        m = convnext_tiny(1000)
        probs, per = [getattr(b.drop_path, "drop_prob", 0.0) for st in m.stages for b in st], 1
    elif name == "vit_b16":
        from deeplearning_b200.classification.vision_transformer.vit_model import VisionTransformer
        from oracle.vit import train_step_grads

        m = VisionTransformer(img_size=224, patch_size=16, embed_dim=768, depth=12, num_heads=12, representation_size=768,
                              num_classes=1000, drop_path_ratio=0.1)
        probs, per = [getattr(b.drop_path, "drop_prob", 0.0) for b in m.blocks], 2
    else:
        from deeplearning_b200.classification.swin_transformer.models.swin_transformer import SwinTransformer
        from oracle.swin import train_step_grads

        m = SwinTransformer()
        probs, per = [getattr(b.drop_path, "drop_prob", 0.0) for l in m.layers for b in l.blocks], 2
    drop, calls = _drop_entries(probs, per, B, fx["seeds"]["u0"])
    assert calls == fx[name]["rand_calls"]
    state = {k: v.clone() for k, v in m.state_dict().items()}
    logits, loss, grads = train_step_grads(state, x, y, drop=drop)
    _close(logits, fx[name]["train_logits"])
    assert abs(float(loss) - fx[name]["train_loss"]) < 1e-3
    for n, g in grads.items():
        ref = fx[name]["grad_norms"][n]
        assert abs(float(g.double().norm()) - ref) <= 2e-3 * (ref + 1e-6), n


class _OracleResNet(torch.nn.Module):
    """The fp32 oracle ResNet as a module: parameters registered for an optimizer, running statistics updated in place."""

    def __init__(self, state):
        super().__init__()
        self.state = dict(state)
        self.params = torch.nn.ParameterList()
        for k, v in state.items():
            if v.is_floating_point() and "running_" not in k:
                self.state[k] = torch.nn.Parameter(v.clone())
                self.params.append(self.state[k])

    def forward(self, x):
        from oracle.resnet import resnet_forward

        return resnet_forward(self.state, x, train=self.training)


def test_resnet50_epoch_loops_match_reference():
    """oracle/train_loop.py's evaluate / train_one_epoch (the loops tests/test_gpu_resnet.py drives the drop-in module with)
    return what the reference's own loops returned on the same weights and batches (make_golden.py, there bit for bit)."""
    from deeplearning_b200.classification.resnet.models.networks import resnet50
    from oracle.resnet import resnet_forward
    from oracle.train_loop import evaluate, train_one_epoch

    with open(os.path.join(HERE, "golden", "resnet50_loops.json")) as f:
        fx = json.load(f)
    torch.manual_seed(fx["seeds"]["init"])
    state = {k: v.clone() for k, v in resnet50().state_dict().items()}
    xc = torch.randn(fx["calib_batch"], 3, 224, 224, generator=torch.Generator().manual_seed(fx["seeds"]["calib"]))
    with torch.no_grad():
        resnet_forward(state, xc, train=True, momentum=1.0)
    g = torch.Generator().manual_seed(fx["seeds"]["batches"])
    batches = [(torch.randn(fx["batch"], 3, 224, 224, generator=g), torch.randint(0, 1000, (fx["batch"],), generator=g))
               for _ in range(fx["steps"])]
    model, cpu, loss_fn = _OracleResNet(state), torch.device("cpu"), torch.nn.CrossEntropyLoss()
    loss, acc = evaluate(model, batches, cpu, loss_fn)
    assert abs(loss - fx["eval_loss"]) < 1e-4 and acc == fx["eval_acc"], (loss, acc)
    opt = torch.optim.SGD(model.parameters(), lr=fx["lr"], momentum=fx["momentum"], weight_decay=fx["weight_decay"])
    loss, acc = train_one_epoch(model, batches, cpu, opt, loss_fn)
    assert abs(loss - fx["train_loss"]) < 1e-4 and acc == fx["train_acc"], (loss, acc)
    norm = float(model.state["fc.weight"].detach().double().norm())
    assert abs(norm - fx["fc_weight_norm_after"]) <= 1e-5 * fx["fc_weight_norm_after"], norm
