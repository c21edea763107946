"""-m "not gpu": the early-stopping rule, the validation schedule and metrics, the argument checks of spVIPES.train's validation
options, and the binding of spv_elbo_accumulate."""
import math
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

from spvipes_b200.trainer import EarlyStopping, elbo_metrics, is_validation_epoch, validation_interval

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(values, **kw):
    """index of the value that stops training, or None"""
    es = EarlyStopping(**kw)
    for i, v in enumerate(values):
        if es.update(v):
            return i
    return None


def test_patience_counts_runs_without_improvement():
    assert _run([5.0, 4.0, 4.0, 4.0], patience=2) == 3
    assert _run([5.0, 4.0, 4.5, 3.0, 3.5, 3.5], patience=2) == 5  # the improvement at index 3 resets the count
    assert _run([5.0, 4.0, 3.0, 2.0], patience=1) is None
    assert _run([5.0, 5.0], patience=1) == 1


def test_first_value_is_an_improvement():
    es = EarlyStopping(patience=1, min_delta=1e9)
    assert not es.update(123.0)
    assert es.best == 123.0 and es.wait == 0
    assert es.update(-1e6)  # not below best - 1e9
    # max mode as well
    es = EarlyStopping(patience=1, min_delta=1e9, mode="max")
    assert not es.update(-5.0) and es.best == -5.0


def test_min_delta_min_mode():
    # improvement only when value < best - min_delta
    assert _run([10.0, 9.6, 9.5, 9.55], patience=3, min_delta=0.5) == 3  # none is below 10 - 0.5
    assert _run([10.0, 9.4, 8.8, 8.2], patience=1, min_delta=0.5) is None
    es = EarlyStopping(patience=5, min_delta=0.5)
    for v in (10.0, 9.4, 9.0):
        es.update(v)
    assert es.best == 9.4 and es.wait == 1


def test_min_delta_max_mode():
    assert _run([1.0, 1.4, 1.5, 1.45], patience=3, min_delta=0.5, mode="max") == 3  # none is above 1 + 0.5
    assert _run([1.0, 1.6, 2.2], patience=1, min_delta=0.5, mode="max") is None
    # a decrease is never an improvement in max mode
    assert _run([1.0, 0.0], patience=1, mode="max") == 1


def test_non_finite_stops_at_once():
    assert _run([3.0, float("nan")], patience=45) == 1
    assert _run([float("inf")], patience=45) == 0
    assert _run([3.0, float("-inf")], patience=45, mode="max") == 1


def test_validation_schedule():
    assert validation_interval(None, False) is None
    assert validation_interval(None, True) == 1
    assert validation_interval(3, False) == 3
    assert [e for e in range(10) if is_validation_epoch(e, 3)] == [2, 5, 8]
    assert [e for e in range(4) if is_validation_epoch(e, 1)] == [0, 1, 2, 3]
    assert not any(is_validation_epoch(e, None) for e in range(10))
    for bad in (0, -1, 1.5):
        with pytest.raises(ValueError):
            validation_interval(bad, True)


def test_unknown_monitor_or_mode():
    with pytest.raises(ValueError, match="monitor"):
        EarlyStopping(monitor="elbo_train")
    with pytest.raises(ValueError, match="mode"):
        EarlyStopping(mode="minimum")


def test_elbo_metrics_from_sums():
    # [rec0, rec1, klp0, klq0, klp1, klq1, n_obs, weighted loss]
    acc = np.array([100.0, 50.0, 3.0, 4.0, 5.0, 6.0, 10.0, 150.0 + 0.5 * 18.0])
    m = elbo_metrics(acc)
    assert math.isclose(m["reconstruction_loss_validation"], 15.0)
    assert math.isclose(m["kl_local_validation"], 1.8)
    assert math.isclose(m["elbo_validation"], 16.8)
    assert math.isclose(m["validation_loss"], 15.9)
    assert set(elbo_metrics(acc, "train")) == {"elbo_train", "reconstruction_loss_train", "kl_local_train"}


def _bare_model(n=(10, 12)):
    """a spVIPES without device state: the argument checks of train() run before any device work"""
    from spvipes_b200.model import spVIPES
    m = object.__new__(spVIPES)
    m.adata = SimpleNamespace(X=np.zeros((sum(n), 3), dtype=np.float32))
    m.history = {"train_loss_epoch": []}
    gil = [list(range(n[0])), list(range(n[0], n[0] + n[1]))]
    return m, gil


def test_train_argument_errors():
    m, gil = _bare_model()
    with pytest.raises(ValueError, match="validation split"):
        m.train(gil, max_epochs=1, train_size=1.0, early_stopping=True)
    with pytest.raises(ValueError, match="validation split"):
        m.train(gil, max_epochs=1, train_size=1.0, check_val_every_n_epoch=2)
    with pytest.raises(ValueError, match="monitor"):
        m.train(gil, max_epochs=1, early_stopping=True, early_stopping_monitor="train_loss_epoch")
    with pytest.raises(ValueError, match="mode"):
        m.train(gil, max_epochs=1, early_stopping=True, early_stopping_mode="lowest")
    with pytest.raises(ValueError, match="check_val_every_n_epoch"):
        m.train(gil, max_epochs=1, check_val_every_n_epoch=0)


def test_elbo_accumulate_binding_matches_header():
    from spvipes_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "spvipes_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+spv_elbo_accumulate\s*\((.*?)\)\s*;", src, flags=re.S)
    assert m
    assert len(m.group(1).split(",")) == len(_lib._SIGS["spv_elbo_accumulate"]) == 11
