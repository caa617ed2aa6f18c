"""Drop-in of lidar4d_b200.LiDAR4D under the reference's Trainer (VERDICT r1 #7, SURVEY.md 8(b)).

The reference's `Trainer` (model/runner.py) is not part of this repository, and it cannot drive the CUDA module itself
(it needs the reference's tiny-cuda-nn model code).  So the chain is:
  (CPU)         tests/trainer_mirror.py returns the loss and predictions of the unmodified Trainer.train_step / eval_step
                when it gets the same model answers: tests/golden/trainer_replay.npz holds the Trainer's results and every
                call it made into the reference model-on-shim (written by tests/golden/make_golden.py)
  (GPU)         the mirror drives lidar4d_b200.LiDAR4D + lidar4d_b200.chamfer + lidar4d_b200.optim.Adam through
                train iterations with autocast + GradScaler + flow loss, EMA evaluate (copy_to / restore through .data),
                a checkpoint round trip, and reproduces the loss the REAL Trainer computed on the CPU on the same parameters
                (tests/golden/trainer_step.npz, written by tests/golden/make_golden.py)."""
import io
import os

import numpy as np
import pytest
import torch

import ref_stubs
from trainer_mirror import MirrorTrainer, default_opt, synthetic_batch
from parity_util import small_config, cuda_model_from_oracle, rel_err
from oracle import lidar4d_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
S_SMALL = 48


def _opt():
    return default_opt(num_frames=6, num_steps=S_SMALL, near_lidar=0.0105, far_lidar=0.851, fp16=False)


class ReplayModel:
    """Stands in for the reference model-on-shim: answers the k-th render / flow call with what the model returned to
    the real Trainer on its k-th call (tests/golden/trainer_replay.npz), after checking that the call carries the same
    arguments, and leaves the torch RNG where that call left it."""

    def __init__(self, fx):
        self.fx, self.n = fx, 0

    def _call(self, kind, args, kw):
        i, fx = self.n, self.fx
        self.n += 1
        assert i < int(fx["n_calls"]) and str(fx[f"call{i}:kind"]) == kind, f"call {i}: unexpected {kind}"
        assert repr(sorted(kw.items())) == str(fx[f"call{i}:kw"]), f"call {i} ({kind}): keyword arguments differ"
        for j, a in enumerate(args):
            assert torch.equal(a.detach().cpu(), torch.from_numpy(fx[f"call{i}:arg{j}"])), f"call {i} ({kind}): argument {j} differs"
        torch.set_rng_state(torch.from_numpy(fx[f"call{i}:rng"]))
        pre = f"call{i}:out:"
        return {k[len(pre):]: torch.from_numpy(fx[k]) for k in fx.keys() if k.startswith(pre)}

    def render(self, rays_o, rays_d, time, **kw):
        return self._call("render", (rays_o, rays_d, time), kw)

    def flow(self, x, time):
        return self._call("flow", (x, time), {})


def test_mirror_reproduces_reference_trainer():
    """The mirror's train_step / eval_step return the loss and predictions of the UNMODIFIED Trainer, given the same
    model answers (the recorded calls of the Trainer into the reference model-on-shim, make_golden.py)."""
    from trainer_mirror import MirrorEMA
    fx = np.load(os.path.join(GOLD, "trainer_replay.npz"), allow_pickle=False)
    opt = _opt()
    train, ev, pcs, ground = synthetic_batch(64, frame=2, num_frames=6, seed=1)
    model = ReplayModel(fx)
    mirror = MirrorTrainer(opt, model, ref_stubs.CpuChamferDist(), pc_list=pcs, pc_ground_list=ground, device=torch.device("cpu"))
    torch.manual_seed(3)
    b = mirror.train_step(train)
    assert float(fx["train:loss"]) == pytest.approx(float(b[4]), rel=1e-6)
    assert torch.allclose(torch.from_numpy(fx["train:pred_depth"]), b[2])
    assert torch.allclose(torch.from_numpy(fx["train:pred_intensity"]), b[0])
    with torch.no_grad():
        eb = mirror.eval_step(ev)
    assert float(fx["eval:loss"]) == pytest.approx(float(eb[6]), rel=1e-6)
    assert torch.allclose(torch.from_numpy(fx["eval:pred_depth"]), eb[1])
    assert model.n == int(fx["n_calls"]), "the mirror made fewer model calls than the Trainer"
    # the EMA stand-in the Trainer used (runner.py:98-101 through ref_stubs); its arithmetic against the closed form
    orc = O.build_seeded(small_config(), 31, flow_last_std=0.02)
    ema = MirrorEMA(orc.parameters(), 0.95)
    ema.update()
    d = min(0.95, 2 / 11)
    p0 = next(p for p in orc.parameters() if p.requires_grad)
    assert torch.allclose(ema.shadow[0], p0.detach())                 # shadow == param while param has not moved
    assert d == pytest.approx(2 / 11)


@pytest.mark.gpu
def test_trainer_mirror_drives_cuda_model():
    from lidar4d_b200.chamfer import chamfer_3DDist
    from lidar4d_b200.optim import Adam
    dev = torch.device("cuda:0")
    fx = np.load(os.path.join(GOLD, "trainer_step.npz"), allow_pickle=False)
    orc = O.build_seeded(small_config(), int(fx["seed"]), flow_last_std=0.02)
    model = cuda_model_from_oracle(orc)                       # fp32 MLP weights, as the reference-on-shim run of the fixture
    model.jitter_seed = int(fx["seed"])
    opt = _opt()
    train, ev, pcs, ground = synthetic_batch(64, frame=2, num_frames=6, seed=1, device=dev)
    tr = MirrorTrainer(opt, model, chamfer_3DDist(), pc_list=pcs, pc_ground_list=ground, device=dev, ema_decay=0.95,
                       optimizer=lambda m: Adam(m, m.get_params(1e-2), betas=(0.9, 0.99), eps=1e-15),
                       lr_scheduler=lambda o: torch.optim.lr_scheduler.LambdaLR(o, lambda it: 0.1 ** min(it / 100, 1)))
    # ---- the loss of the REAL Trainer.train_step (reference model-on-shim, CPU) on the same parameters and batch ----
    torch.manual_seed(3)
    model._jitter_calls = 0
    out = tr.train_step(train)
    assert float(out[4]) == pytest.approx(float(fx["train_loss"]), rel=2e-4)
    assert rel_err(out[2], fx["pred_depth"]) < 1e-4
    model._jitter_calls = 0
    with torch.no_grad():
        e = tr.eval_step(ev)
    assert float(e[6]) == pytest.approx(float(fx["eval_loss"]), rel=2e-4)
    # ---- training iterations exactly as runner.py:491-511, now with fp16 autocast + GradScaler ----
    tr.fp16 = True
    tr.scaler = torch.amp.GradScaler("cuda", enabled=True)
    losses = [tr.train_iteration(train) for _ in range(3)]
    assert all(np.isfinite(losses)) and tr.scaler.get_scale() == 65536.0
    assert losses[-1] < losses[0]
    tr.end_epoch()                                            # ema.update()
    losses.append(tr.train_iteration(train))
    tr.end_epoch()
    # ---- evaluate with EMA weights: copy_to()/restore() write through .data (no version bump) ----
    with torch.no_grad():
        raw = tr.eval_step(ev)[1].clone()
    ema = tr.evaluate(ev)[1].clone()
    assert not torch.allclose(raw, ema), "the EMA weights were not picked up by the kernels"
    with torch.no_grad():
        again = tr.eval_step(ev)[1]
    assert torch.equal(raw, again), "restore() was not picked up"
    # ---- checkpoint: save, keep training, load, and the next step repeats ----
    buf = io.BytesIO()
    torch.save(tr.checkpoint(), buf)
    calls = model._jitter_calls
    l_a = tr.train_iteration(train)
    buf.seek(0)
    res = tr.load_checkpoint(torch.load(buf, weights_only=False))
    assert not res.missing_keys and not res.unexpected_keys
    model._jitter_calls = calls
    l_b = tr.train_iteration(train)
    assert l_b == pytest.approx(l_a, rel=1e-4)
    # torch.optim.Adam works unchanged as well (main_lidar4d.py:298-300 as written)
    tr2 = MirrorTrainer(opt, model, chamfer_3DDist(), pc_list=pcs, pc_ground_list=ground, device=dev, fp16=True,
                        optimizer=lambda m: torch.optim.Adam(m.get_params(1e-2), betas=(0.9, 0.99), eps=1e-15))
    l0 = tr2.train_iteration(train)
    l1 = tr2.train_iteration(train)
    assert np.isfinite(l0) and np.isfinite(l1)
