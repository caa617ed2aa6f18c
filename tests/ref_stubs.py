"""Test infrastructure: import the reference's model/runner.py (build container only - needs /root/reference) with
stand-ins for the third-party modules that are not installed here (SURVEY.md 8(c): torch_ema, tensorboardX, imageio,
open3d; lpips / skimage are only needed by utils/metrics.py, which the Trainer class itself does not import) and for
the chamfer extension wrapper, whose module-level `importlib.find_loader` no longer exists in Python 3.12."""
import sys
import types

import torch

REF = "/root/reference"


class _CpuChamferFn(torch.autograd.Function):
    """chamfer_3DFunction's contract (dist_chamfer_3D.py:31-73) in plain torch, for CPU runs of the reference Trainer."""

    @staticmethod
    def forward(ctx, a, b):
        d = ((a.unsqueeze(2) - b.unsqueeze(1)) ** 2).sum(-1)
        d1, i1 = d.min(2)
        d2, i2 = d.min(1)
        ctx.save_for_backward(a, b, i1, i2)
        return d1, d2, i1.int(), i2.int()

    @staticmethod
    def backward(ctx, g1, g2, *_):
        a, b, i1, i2 = ctx.saved_tensors
        ga, gb = torch.zeros_like(a), torch.zeros_like(b)
        for bi in range(a.shape[0]):
            diff1 = a[bi] - b[bi][i1[bi]]
            ga[bi] += 2 * g1[bi].unsqueeze(-1) * diff1
            gb[bi].index_add_(0, i1[bi], -2 * g1[bi].unsqueeze(-1) * diff1)
            diff2 = b[bi] - a[bi][i2[bi]]
            gb[bi] += 2 * g2[bi].unsqueeze(-1) * diff2
            ga[bi].index_add_(0, i2[bi], -2 * g2[bi].unsqueeze(-1) * diff2)
        return ga, gb


class CpuChamferDist(torch.nn.Module):
    def forward(self, a, b):
        return _CpuChamferFn.apply(a.contiguous(), b.contiguous())


def install_reference_stubs():
    from trainer_mirror import MirrorEMA

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    class ExponentialMovingAverage(MirrorEMA):
        def __init__(self, parameters, decay, use_num_updates=True):
            super().__init__(list(parameters), decay)

    mod("torch_ema", ExponentialMovingAverage=ExponentialMovingAverage)
    mod("tensorboardX", SummaryWriter=lambda *a, **k: None)
    mod("imageio")
    mod("open3d")
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import utils  # noqa: F401  (the reference's package)
    mod("utils.chamfer3D.dist_chamfer_3D", chamfer_3DDist=CpuChamferDist)


def import_reference_runner():
    sys.dont_write_bytecode = True
    install_reference_stubs()
    import model.runner as runner
    return runner
