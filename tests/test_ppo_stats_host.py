"""CPU checks of the host side of the PPO training diagnostics (PpoUpdateStats) on synthetic records: per-key means over the
minibatches that ran, epochs_run, and the epoch-granular early-stop rule on the approximate KL."""
import math

import pytest
import torch

from ppo_rl_satellite_b200 import _lib as L
from ppo_rl_satellite_b200.dropin.ppo_continuous import PpoUpdateStats


def _records(K, per_epoch_kl, mbs=4):
    """K epochs of `mbs` minibatches; actor term k of epoch e sums to mbs * (e + 1) * (k + 1), the KL to mbs * per_epoch_kl[e]"""
    rec = torch.zeros((K, 2, L.PPO_STATS_DOUBLES), dtype=torch.float64)
    for e in range(K):
        for net in range(2):
            for k in range(L.PPO_STAT_COUNT):
                rec[e, net, k] = mbs * (e + 1) * (k + 1) * (1 if net == 0 else 10)
            rec[e, net, L.PPO_STAT_COUNT] = mbs
        rec[e, 0, L.PPO_STAT_APPROX_KL] = mbs * per_epoch_kl[e]
    return rec


def test_layout_matches_header():
    import os
    import re
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "satb200.h")).read()
    vals = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define SAT_PPO_STAT(?:S)?_([A-Z_]+)\s+(\d+)", hdr)}
    assert vals == {"LOSS": L.PPO_STAT_LOSS, "SURROGATE": L.PPO_STAT_SURROGATE, "ENTROPY": L.PPO_STAT_ENTROPY,
                    "APPROX_KL": L.PPO_STAT_APPROX_KL, "CLIP_FRAC": L.PPO_STAT_CLIP_FRAC, "GRAD_NORM": L.PPO_STAT_GRAD_NORM,
                    "CLIP_COEF": L.PPO_STAT_CLIP_COEF, "COUNT": L.PPO_STAT_COUNT, "DOUBLES": L.PPO_STATS_DOUBLES}
    assert L.ppo_grad_floats_stats(3) == L.ppo_param_floats(3) + 6


def test_means_over_all_epochs_without_target():
    kl = [0.01, 0.02, 0.04]
    st = PpoUpdateStats(_records(3, kl), minibatches=4)
    assert [st.end_epoch(e) for e in range(3)] == [False, False, False]
    d = st.as_dict()
    assert d["epochs_run"] == 3 and d["early_stopped"] is False
    # mean over the 12 minibatches of sums 4 (e + 1) (k + 1): (k + 1) * (1 + 2 + 3) / 3
    assert d["policy_loss"] == pytest.approx(2 * 2.0) and d["entropy"] == pytest.approx(3 * 2.0)
    assert d["clip_fraction"] == pytest.approx(5 * 2.0) and d["actor_grad_norm"] == pytest.approx(6 * 2.0)
    assert d["value_loss"] == pytest.approx(1 * 2.0 * 10) and d["critic_grad_norm"] == pytest.approx(6 * 2.0 * 10)
    assert d["approx_kl"] == pytest.approx(sum(kl) / 3)
    assert d["approx_kl_per_epoch"] == pytest.approx(kl)


def test_early_stop_after_the_epoch_whose_mean_kl_exceeds_the_target():
    kl = [0.005, 0.03, 0.5, 0.5]
    rec = _records(4, kl)
    st = PpoUpdateStats(rec, minibatches=4, target_kl=0.02)
    ran = []
    for e in range(4):
        ran.append(e)
        if st.end_epoch(e):
            break
    assert ran == [0, 1]
    d = st.as_dict()
    assert d["epochs_run"] == 2 and d["early_stopped"] is True
    assert d["approx_kl_per_epoch"] == pytest.approx(kl[:2])
    assert d["approx_kl"] == pytest.approx(sum(kl[:2]) / 2)          # only the minibatches that ran
    assert d["policy_loss"] == pytest.approx(2 * 1.5)


def test_target_equal_to_the_kl_does_not_stop_and_last_epoch_is_not_an_early_stop():
    st = PpoUpdateStats(_records(2, [0.25, 0.75]), minibatches=4, target_kl=0.25)   # exact in binary
    assert st.end_epoch(0) is False
    assert st.end_epoch(1) is False                  # nothing left to skip
    assert st.as_dict()["early_stopped"] is False and st.epochs_run == 2


def test_extra_scalars_and_empty_epochs():
    st = PpoUpdateStats(_records(2, [0.1, 0.1]), minibatches=4)
    st.extra["explained_variance"] = torch.tensor(0.25, dtype=torch.float32)
    d = st.as_dict()                                  # nothing ran yet: means are NaN, extras still reported
    assert d["epochs_run"] == 0 and math.isnan(d["approx_kl"]) and d["approx_kl_per_epoch"] == []
    assert d["explained_variance"] == 0.25
