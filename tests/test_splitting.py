"""Multilevel splitting (cavgym_b200.splitting) without a GPU: the estimator against the exact hitting probability of a
random walk run by a torch-CPU stand-in for the engine, its work-normalised variance against crude Monte Carlo's, and
the C-ABI entry's refusal of a NULL engine."""
import ctypes
import math

import numpy as np
import pytest
import torch

from cavgym_b200 import _native, splitting

# Gambler's ruin with jumps: from X0, steps +1, +2, -1, -2 with these probabilities; a tester "wins" at X >= TOP, the
# episode ends otherwise at X <= 0 or after HORIZON steps.  Jumps of 2 skip levels.
STEPS = np.array([1, 2, -1, -2])
PROBS = np.array([0.3, 0.1, 0.4, 0.2])
X0, TOP, HORIZON = 2, 42, 400


def exact_probability():
    """P(X reaches TOP within HORIZON steps), by dynamic programming over the states 1..TOP-1 (exact up to rounding)."""
    win = np.zeros(TOP + 2)   # win[x] for x in 0..TOP+1 at the remaining horizon; x >= TOP counts as won
    win[TOP:] = 1.0
    for _ in range(HORIZON):
        nxt = win.copy()
        for x in range(1, TOP):
            nxt[x] = sum(p * win[min(max(x + s, 0), TOP + 1)] for s, p in zip(STEPS, PROBS))
        win = nxt
    return win[X0]


class WalkEnv:
    """The methods splitting.estimate uses, on a batch of independent walks.  Danger = position; status as
    cavgym_rollout_until's.  salt = 0 draws from the env's own generator, another salt from a generator seeded with it."""

    dtype, device, max_timesteps = torch.float64, torch.device("cpu"), HORIZON

    def __init__(self, n, seed=0):
        self.num_envs = n
        self.rng = torch.Generator().manual_seed(seed)
        self.x = torch.zeros(n, dtype=torch.int64)
        self.timestep = torch.zeros(n, dtype=torch.int32)
        self.done = torch.zeros(n, dtype=torch.uint8)
        self.winner = torch.full((n,), -1, dtype=torch.int32)

    def reset(self):
        self.x.fill_(X0)
        self.timestep.zero_()
        self.done.zero_()
        self.winner.fill_(-1)

    def fork(self, src, dst):
        for a in (self.x, self.timestep, self.done, self.winner):
            a[dst] = a[src].clone()

    def rollout_until(self, n_steps, level, score, salt=0, status=None):
        rng = self.rng if salt == 0 else torch.Generator().manual_seed(salt & ((1 << 63) - 1))
        status = torch.zeros(self.num_envs, dtype=torch.uint8) if status is None else status
        won = (self.done != 0) & (self.winner > 0)
        score[won] = math.inf
        status[:] = torch.where(self.done != 0, torch.where(won, 1, 2), torch.where(score >= level, 1, 0)).to(torch.uint8)
        steps, probs = torch.as_tensor(STEPS), torch.as_tensor(PROBS)
        for _ in range(n_steps):
            live = status == 0
            if not live.any():
                break
            move = steps[torch.multinomial(probs, self.num_envs, replacement=True, generator=rng)]
            self.x += torch.where(live, move, 0)
            self.timestep += live.to(torch.int32)
            win, lose = live & (self.x >= TOP), live & (self.x <= 0)
            cut = live & ~win & ~lose & (self.timestep >= HORIZON)
            self.done[win | lose] = 1
            self.done[cut] = 2
            self.winner[win] = 1
            score[win] = math.inf
            status[win] = 1
            status[lose | cut] = 2
            rest = live & ~win & ~lose & ~cut
            score[rest] = torch.maximum(score[rest], self.x[rest].to(score.dtype))
            status[rest & (score >= level)] = 1
        return status


LEVELS = tuple(range(4, TOP - 1, 3))


def test_splitting_agrees_with_the_exact_hitting_probability_and_beats_crude_monte_carlo():
    p = exact_probability()
    assert 1e-7 < p < 1e-5
    result = splitting.estimate(WalkEnv(2000, seed=1), LEVELS, repetitions=40, seed=3)
    est = np.array(result.estimates)
    se = est.std(ddof=1) / math.sqrt(len(est))
    assert abs(est.mean() - p) <= 4 * se, (est.mean(), p, se)
    assert result.interval.value == pytest.approx(est.mean()) and result.levels[-1] == math.inf
    assert all(len(f) == len(LEVELS) + 1 for f in result.fractions)
    # work-normalised relative variance: (variance / p^2) x steps per estimate.  Crude Monte Carlo's estimate from one
    # episode is a Bernoulli(p) draw: relative variance (1 - p) / p, at the walk's mean episode length in steps.
    walk = WalkEnv(20000, seed=2)
    walk.reset()
    walk.rollout_until(HORIZON, math.inf, torch.full((20000,), -math.inf, dtype=torch.float64))
    crude = (1 - p) / p * walk.timestep.double().mean().item()
    split = est.var(ddof=1) / p ** 2 * (result.env_steps / len(est))
    assert split * 100 < crude, (split, crude)


def test_no_parked_env_gives_zero():
    result = splitting.estimate(WalkEnv(50, seed=4), (TOP - 0.5,), repetitions=3, seed=0)
    assert result.estimates == [0.0, 0.0, 0.0] and result.mean == 0.0
    assert all(f == [0.0] for f in result.fractions)


def test_resample_keeps_the_parked_slots_and_spreads_the_rest():
    parked = torch.tensor([3, 7, 8])
    src, dst = splitting.resample(parked, 10, torch.Generator().manual_seed(0))
    assert dst.tolist() == [0, 1, 2, 4, 5, 6, 9]
    counts = torch.bincount(torch.cat([parked, src]), minlength=10)[parked]
    assert sorted(counts.tolist()) == [3, 3, 4]   # floor(10 / 3) each, the one left over to a single parked env


def test_levels_and_salts():
    with pytest.raises(ValueError):
        splitting.estimate(WalkEnv(4), (3, 2), repetitions=1)
    salts = {splitting.stage_salt(s, r, j) for s in range(3) for r in range(3) for j in range(3)}
    assert len(salts) == 27 and 0 not in salts


def test_rollout_until_refuses_a_null_engine():
    lib = _native.load()
    score = (ctypes.c_double * 4)()
    status = (ctypes.c_uint8 * 4)()
    assert lib.cavgym_rollout_until(None, 4, 1.0, 0, score, status, None) == -22   # CAV_EINVAL
    assert b"NULL" in lib.cavgym_last_error()
