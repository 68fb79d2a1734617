"""Checkpoint payload compatibility with the reference (SURVEY 8f-4): torch.optim.Adam-format optimizer state, StepLR
state, tolerant resume; device metrics against numpy restatements of the reference's formulas."""
import numpy as np
import pytest
import torch

import graph_neural_cellular_automata_b200 as G
from graph_neural_cellular_automata_b200.training.optim import FusedNormalizedAdam
from graph_neural_cellular_automata_b200.utils import checkpoint as CK
from graph_neural_cellular_automata_b200.utils import metrics as M


def _model():
    return G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                           graph_zero_padded_shift=False)


def test_optimizer_state_round_trips_through_torch_adam(tmp_path):
    torch.manual_seed(0)
    m = _model()
    opt = FusedNormalizedAdam(m, lr=3e-4, weight_decay=1e-5)
    opt.exp_avg.normal_(); opt.exp_avg_sq.uniform_(); opt.step_count = 17
    sd = opt.torch_state_dict()
    # a stock Adam over the same module accepts it, and holds the same moments per parameter
    ref = torch.optim.Adam(m.parameters(), lr=1.0)
    ref.load_state_dict(sd)
    params = list(m.parameters())
    names = [n for n, _ in m.named_parameters()]
    owned = 0
    for i, p in enumerate(params):
        st = ref.state.get(p)
        if "gate_mlp" in names[i] or "perception" in names[i]:
            assert not st
            continue
        owned += 1
        assert float(st["step"]) == 17 and st["exp_avg"].shape == p.shape
    assert owned == 12 and ref.param_groups[0]["lr"] == 3e-4
    # payload on disk -> fresh model + optimiser
    path = str(tmp_path / "nca_epoch3.pt")
    CK.save_checkpoint(path, m, opt, epoch=3, config={"x": 1}, scheduler_state=CK.steplr_state(3e-4, 150, 0.85, 2))
    m2 = _model()
    opt2 = FusedNormalizedAdam(m2, lr=1.0)
    payload, missing, unexpected = CK.load_checkpoint(path, m2, opt2)
    assert not missing and not unexpected and payload["epoch"] == 3 and payload["param_count"] == 10753
    assert torch.equal(opt2.exp_avg, opt.exp_avg) and torch.equal(opt2.exp_avg_sq, opt.exp_avg_sq)
    assert opt2.step_count == 17 and opt2.lr == 3e-4
    assert torch.equal(opt2.flat, opt.flat)
    assert CK.pick_resume(str(tmp_path))[0] == path
    sch = torch.optim.lr_scheduler.StepLR(torch.optim.Adam(m.parameters(), lr=3e-4), step_size=150, gamma=0.85)
    sch.load_state_dict(payload["scheduler_state"])


def test_resume_in_stock_adam_steplr_after_a_decay_boundary(tmp_path):
    """A checkpoint written here AFTER the first StepLR boundary resumes in the reference's trainer (stock Adam + StepLR,
    train_graph_augmented_nca.py:143-158,405-416) at the DECAYED rate: StepLR is chainable and continues from
    `param_groups[0]["lr"]`, so the payload must carry base*gamma**(last_epoch//step_size) there, `initial_lr` = base."""
    base, step_size, gamma = 2e-4, 150, 0.85
    m = _model()
    opt = FusedNormalizedAdam(m, lr=base, weight_decay=1e-5)
    opt.exp_avg.normal_(); opt.exp_avg_sq.uniform_(); opt.step_count = 5
    for last_epoch in (149, 150, 301, 449):
        path = str(tmp_path / f"nca_epoch{last_epoch}.pt")
        CK.save_checkpoint(path, m, opt, epoch=last_epoch, scheduler_state=CK.steplr_state(base, step_size, gamma, last_epoch))
        payload = torch.load(path, map_location="cpu", weights_only=False)
        ref_opt = torch.optim.Adam(_model().parameters(), lr=base, weight_decay=1e-5)
        ref_sch = torch.optim.lr_scheduler.StepLR(ref_opt, step_size=step_size, gamma=gamma)
        ref_opt.load_state_dict(payload["optimizer_state"])
        ref_sch.load_state_dict(payload["scheduler_state"])
        want = base * gamma ** (last_epoch // step_size)
        assert ref_opt.param_groups[0]["lr"] == pytest.approx(want, rel=1e-12)
        assert ref_opt.param_groups[0]["initial_lr"] == base
        ref_opt.step(); ref_sch.step()                         # one more epoch in the reference's loop
        assert ref_opt.param_groups[0]["lr"] == pytest.approx(base * gamma ** ((last_epoch + 1) // step_size), rel=1e-12)
        # and back: the base rate, not the decayed one, is what this optimiser keeps (the trainer decays per step)
        opt2 = FusedNormalizedAdam(_model(), lr=1.0)
        opt2.load_torch_state_dict(payload["optimizer_state"])
        assert opt2.lr == base


def test_device_metrics_match_the_reference_formulas():
    torch.manual_seed(1)
    state = torch.rand(3, 16, 40, 40)
    target = torch.rand(4, 40, 40)
    pp, ps = M.pixel_perfect(state, target), M.psnr_rgb(state, target)
    for b in range(3):
        pred = state[b, :4]
        rgba = torch.cat([pred[:3] * pred[3:4], pred[3:4]], 0).numpy()
        diff = np.abs(rgba - target.numpy())
        assert abs(float(pp[b]) - float((diff < 0.05).all(axis=0).mean())) < 1e-6
        a, t = rgba[:3].clip(0, 1), target.numpy()[:3].clip(0, 1)
        assert abs(float(ps[b]) - 10 * np.log10(1.0 / ((a - t) ** 2).mean())) < 1e-4
