"""Oracle: the reference's epoch loop restated (classification/resnet/utils.py:28-57 ``train_one_epoch``):
for each (images, labels): pred = model(images); acc += (argmax == labels); loss = CE(pred, labels); loss.backward();
optimizer.step(); optimizer.zero_grad().  The optimizer is SGD(momentum 0.9, weight_decay 5e-5) as built at
classification/resnet/train.py:96.  Runs on CPU in fp32 on the oracle's functional models; used as the parity checker of the
trainer tests and as bench.py's CPU baseline / ``--impl reference`` arm (kind "port": the reference's Python modules cannot
travel to the GPU box, and ``tests/golden/make_golden.py`` shows this restatement is bit-identical to them).
"""
import torch
import torch.nn.functional as F


class CpuSgdTrainer:
    def __init__(self, forward_fn, state, lr=0.01, momentum=0.9, weight_decay=5e-5):
        self.forward_fn = forward_fn
        self.state = state
        self.param_names = [k for k, v in state.items() if v.is_floating_point() and "running_" not in k]
        for k in self.param_names:
            state[k] = state[k].detach().clone().requires_grad_(True)
        self.opt = torch.optim.SGD([state[k] for k in self.param_names], lr=lr, momentum=momentum,
                                   weight_decay=weight_decay)

    def step(self, images, labels):
        pred = self.forward_fn(self.state, images, train=True)
        correct = int((pred.argmax(1) == labels).sum())
        loss = F.cross_entropy(pred, labels)
        loss.backward()
        self.opt.step()
        self.opt.zero_grad()
        return float(loss.detach()), correct


def train_one_epoch(model, data_loader, device, optimizer, loss_function):
    """The reference's ``train_one_epoch`` protocol (classification/resnet/utils.py:28-57) on any module, without its
    per-step prints: the loss is summed in an fp32 tensor on ``device``.  Returns (mean loss per step, accuracy over the
    samples seen), as the reference does.  ``tests/golden/make_golden.py`` checks that this loop and ``evaluate`` return
    exactly what the reference's own loops return; ``tests/golden/resnet50_loops.json`` keeps those values."""
    model.train()
    loss_sum = torch.zeros(1, device=device)
    correct = torch.zeros(1, device=device)
    optimizer.zero_grad()
    seen = steps = 0
    for images, labels in data_loader:
        images, labels = images.to(device), labels.to(device)
        seen += images.shape[0]
        steps += 1
        pred = model(images)
        correct += (pred.argmax(1) == labels).sum()
        loss = loss_function(pred, labels)
        loss.backward()
        loss_sum += loss.detach()
        if not torch.isfinite(loss):
            raise FloatingPointError(f"non-finite training loss {float(loss)}")
        optimizer.step()
        optimizer.zero_grad()
    return loss_sum.item() / steps, correct.item() / seen


@torch.no_grad()
def evaluate(model, data_loader, device, loss_function):
    """The reference's ``evaluate`` protocol (classification/resnet/utils.py:60-83): eval mode, no autograd, same return."""
    model.eval()
    loss_sum = torch.zeros(1, device=device)
    correct = torch.zeros(1, device=device)
    seen = steps = 0
    for images, labels in data_loader:
        images, labels = images.to(device), labels.to(device)
        seen += images.shape[0]
        steps += 1
        pred = model(images)
        correct += (pred.argmax(1) == labels).sum()
        loss_sum += loss_function(pred, labels)
    return loss_sum.item() / steps, correct.item() / seen
