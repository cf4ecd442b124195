"""The optimizer reference of the GPU optimizer tests, pinned against torch on the CPU: ``oracle/prior_oracle.py``'s
``adam_step`` / ``adamax_step`` (float64, step count held by the caller per parameter group) and ``Plateau`` against
``torch.optim.Adam`` / ``Adamax`` and ``ReduceLROnPlateau`` in float64, with groups of different lr and weight decay, a
group that joins late and one that sits out some steps and rejoins, and a scripted loss sequence that drives the
scheduler through patience, the threshold equality, ``min_lr`` and the eps-suppressed reduction.

It also pins the libawb kernels' per-group step semantics on the host: they count the steps a group sat out
(``OptScal.group_start``) and bias-correct a group with ``step + 1 - skipped``, which must equal torch's per-parameter
step count."""
import pytest
import torch

from oracle import prior_oracle as O

STEPS = 50
PATIENCE, FACTOR, THRESHOLD, MIN_LR, PLATEAU_EPS = 3, 0.5, 1e-4, 1e-3, 1e-8
# group lr / weight decay; group 2's lr sits 5e-9 above min_lr: its first reduction is suppressed by the scheduler's eps
GROUPS = [dict(lr=1e-2, weight_decay=0.0), dict(lr=3e-3, weight_decay=1e-2), dict(lr=MIN_LR + 5e-9, weight_decay=1e-3)]


def _group_active(g: int, k: int) -> bool:
    """Group 2 joins late (step 6) and sits out steps 20..27; group 1 sits out step 40 only."""
    if g == 2:
        return k >= 6 and not 20 <= k < 28
    if g == 1:
        return k != 40
    return True


def _losses():
    """Decreasing, then flat (patience runs out again and again until min_lr), an exact threshold equality (not an
    improvement), a real improvement that resets the counter, and flat again."""
    out = [1.0 / (1 + k) for k in range(6)]
    best = out[-1]
    out += [best * 1.5] * 14                                    # 14 bad steps: reductions after 4, 8, 12
    out.append(best * (1.0 - THRESHOLD))                        # equality: counts as bad
    out.append(best * 0.5)                                      # improvement
    out += [best * 0.6] * (STEPS - len(out))
    return out


@pytest.mark.parametrize("kind", ["adam", "adamax"])
def test_oracle_matches_torch_with_per_group_steps_and_plateau(kind):
    gen = torch.Generator().manual_seed(3)
    shapes = [[(5, 3), (7,)], [(4, 4), (1,)], [(2, 9)]]
    init = [[torch.randn(s, generator=gen, dtype=torch.float64) for s in grp] for grp in shapes]
    tp = [[t.clone().requires_grad_(True) for t in grp] for grp in init]
    cls = torch.optim.Adam if kind == "adam" else torch.optim.Adamax
    opt = cls([dict(params=tp[g], **GROUPS[g]) for g in range(3)], betas=(0.9, 0.999), eps=1e-8, foreach=False)
    sched = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, mode="min", factor=FACTOR, patience=PATIENCE,
                                                       threshold=THRESHOLD, threshold_mode="rel", cooldown=0,
                                                       min_lr=MIN_LR, eps=PLATEAU_EPS)
    op = [[t.clone() for t in grp] for grp in init]
    om = [[torch.zeros_like(t) for t in grp] for grp in init]
    ov = [[torch.zeros_like(t) for t in grp] for grp in init]
    plateau = O.Plateau([g["lr"] for g in GROUPS], patience=PATIENCE, factor=FACTOR, threshold=THRESHOLD,
                        min_lr=MIN_LR, eps=PLATEAU_EPS)
    own = [0, 0, 0]            # the oracle's per-group step counts
    skipped = [0, 0, 0]        # the kernels' OptScal.group_start
    step = 0                   # the kernels' OptScal.step
    step_fn = O.adam_step if kind == "adam" else O.adamax_step
    reductions, suppressed_seen = 0, False
    for k, loss in enumerate(_losses()):
        opt.zero_grad(set_to_none=True)
        for g in range(3):
            if not _group_active(g, k):
                continue
            own[g] += 1
            for i, t in enumerate(tp[g]):
                grad = torch.randn(t.shape, generator=gen, dtype=torch.float64) * (1.0 + i)
                t.grad = grad
                step_fn(op[g][i], grad, om[g][i], ov[g][i], own[g], plateau.lrs[g], weight_decay=GROUPS[g]["weight_decay"])
        opt.step()
        lrs_before = list(plateau.lrs)
        sched.step(loss)
        plateau.step(loss)
        if plateau.lrs != lrs_before:
            reductions += 1
        if plateau.lrs[2] == lrs_before[2] and plateau.lrs[1] != lrs_before[1]:
            suppressed_seen = True
        # the kernels' counters: every group's bias correction uses step + 1 - skipped
        for g in range(3):
            if _group_active(g, k):
                assert step + 1 - skipped[g] == own[g] == int(opt.state[tp[g][0]]["step"]), (k, g)
            else:
                skipped[g] += 1
        step += 1
        for g in range(3):
            for i, t in enumerate(tp[g]):
                torch.testing.assert_close(op[g][i], t.detach(), rtol=1e-13, atol=1e-15, msg=lambda s: f"step {k} p[{g}][{i}]: {s}")
                st = opt.state.get(t)
                if st:
                    torch.testing.assert_close(om[g][i], st["exp_avg"], rtol=1e-13, atol=1e-16)
                    torch.testing.assert_close(ov[g][i], st["exp_avg_sq" if kind == "adam" else "exp_inf"],
                                               rtol=1e-13, atol=1e-16)
                else:
                    assert not own[g]
        assert plateau.lrs == [float(pg["lr"]) for pg in opt.param_groups], k
        assert plateau.best == sched.best and plateau.num_bad == sched.num_bad_epochs, k
    # the script reached what it is there for
    assert reductions >= 3 and suppressed_seen
    assert plateau.lrs[1] == MIN_LR and plateau.lrs[2] == GROUPS[2]["lr"] and plateau.lrs[0] < GROUPS[0]["lr"] / 4
    assert own == [STEPS, STEPS - 1, STEPS - 6 - 8]
