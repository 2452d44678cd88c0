"""
The builder / serializer seam against what the original gordo does with the gordo_b200 classes (SURVEY.md §8b.2,
§8b.5): gordo/serializer/from_definition.py:176-191 resolving ``gordo_b200.*`` class paths, into_definition round
trips, and gordo/builder/build_model.py:192-339 (``ModelBuilder._build``, inherited by FleetModelBuilder when gordo
is installed) driving the mirror up to its first device call.

tests/golden/seam_golden.json holds what gordo's own code produced, recorded by tests/golden/make_seam_golden.py
(which executes the reference modules unmodified, third-party dependencies stubbed): the object graph its
``from_definition`` builds for each definition below, what its ``into_definition`` writes for it, and, for the
builder, the definition ``_build`` resolves, the estimator it builds and the keyword arguments of its
``model.cross_validate(...)`` call.  These tests check gordo_b200's own serializer, redirect, metrics, split
metadata and estimator signatures against that record, with no GPU and without gordo installed.
"""
import inspect
import json
import os

import numpy as np
import pandas as pd
import yaml

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "seam_golden.json")

DEFINITIONS = {
    "detector": yaml.safe_load("""
        gordo_b200.machine.model.anomaly.diff.DiffBasedAnomalyDetector:
          require_thresholds: false
          base_estimator:
            sklearn.pipeline.Pipeline:
              steps:
                - sklearn.preprocessing.MinMaxScaler
                - gordo_b200.machine.model.models.KerasAutoEncoder:
                    kind: feedforward_hourglass
                    encoding_layers: 2
                    epochs: 3
                    batch_size: 64
        """),
    # LSTM estimators: lookback_window / batch_size survive the codec
    "lstm": {"gordo_b200.machine.model.models.KerasLSTMAutoEncoder": {"kind": "lstm_hourglass", "lookback_window": 12}},
    # the raw-Keras regressor: its `kind` (a spec holding tensorflow.keras.* paths) must reach the class untouched --
    # gordo's from_definition hands it over through the from_definition hook instead of importing the paths
    "raw": {"gordo_b200.machine.model.models.KerasRawModelRegressor": {"kind": {
        "compile": {"loss": "mse", "optimizer": "adam"},
        "spec": {"tensorflow.keras.models.Sequential": {"layers": [
            {"tensorflow.keras.layers.Dense": {"units": 4, "input_shape": [4], "activation": "tanh"}},
            {"tensorflow.keras.layers.Dense": {"units": 1}}]}}}, "epochs": 2}},
}

# an unmodified project's model block: gordo.machine.model.* paths, which FleetModelBuilder redirects to the mirror
BUILDER_MODEL = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": {
    "sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler",
                                            {"gordo.machine.model.models.KerasAutoEncoder": {"kind": "feedforward_hourglass"}}]}}}}

BUILDER_EVALUATIONS = {
    "r2_only": {"cv_mode": "full_build", "seed": 3, "metrics": ["sklearn.metrics.r2_score"],
                "scoring_scaler": "sklearn.preprocessing.MinMaxScaler"},
    "default_metrics": {"cv_mode": "full_build", "seed": 3,
                        "metrics": ["explained_variance_score", "r2_score", "mean_squared_error", "mean_absolute_error"],
                        "scoring_scaler": "sklearn.preprocessing.MinMaxScaler"},
}


def builder_frame():
    return pd.DataFrame(np.random.default_rng(0).random((200, 4)), columns=list("abcd"),
                        index=pd.date_range("2020-01-01", periods=200, freq="10min", tz="UTC"))


def describe(obj):
    """An estimator graph as plain JSON data: class path and constructor parameters, recursively."""
    if isinstance(obj, (list, tuple)):
        return [describe(v) for v in obj]
    if isinstance(obj, dict):
        return {str(k): describe(v) for k, v in obj.items()}
    if hasattr(type(obj), "get_params"):
        return {"class": f"{type(obj).__module__}.{type(obj).__qualname__}",
                "params": describe(obj.get_params(deep=False))}
    if obj is None or isinstance(obj, (bool, int, float, str)):
        return obj
    return repr(obj)


def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


def test_reference_serializer_resolves_and_round_trips_the_mirror():
    from gordo_b200 import serializer as ours
    import gordo_b200.machine.model.anomaly.diff as d
    import gordo_b200.machine.model.models as m
    from sklearn.pipeline import Pipeline
    golden = _golden()["serializer"]
    assert sorted(golden) == sorted(DEFINITIONS)
    for name, definition in DEFINITIONS.items():
        want = golden[name]
        model = ours.from_definition(definition)
        # the same object graph gordo's from_definition built from this definition
        assert describe(model) == want["built"], name
        # into_definition writes what gordo's into_definition wrote, and both read back to the same graph
        assert json.loads(json.dumps(ours.into_definition(model))) == want["into_definition"], name
        assert describe(ours.from_definition(want["into_definition"])) == want["read_back"], name
        assert want["read_back"] == want["built"], name

    model = ours.from_definition(DEFINITIONS["detector"])
    assert type(model) is d.DiffBasedAnomalyDetector and model.require_thresholds is False
    assert isinstance(model.base_estimator, Pipeline)
    est = model.base_estimator.steps[1][1]
    assert type(est) is m.KerasAutoEncoder and est.kind == "feedforward_hourglass"
    assert est.kwargs == {"encoding_layers": 2, "epochs": 3, "batch_size": 64}      # models.py:146-159 hook used
    lstm = ours.from_definition(DEFINITIONS["lstm"])
    assert lstm.lookback_window == 12 and ours.from_definition(ours.into_definition(lstm)).lookback_window == 12
    reg = ours.from_definition(DEFINITIONS["raw"])
    assert type(reg) is m.KerasRawModelRegressor and reg.kwargs == {"epochs": 2}
    assert reg._topology().widths == [4, 4, 1] and reg._topology().acts == ["tanh", "linear"]
    assert ours.from_definition(ours.into_definition(reg)).kind == reg.kind


def test_fleet_model_builder_is_a_reference_model_builder_and_drives_the_mirror():
    from sklearn.model_selection import TimeSeriesSplit
    from gordo_b200 import serializer
    from gordo_b200.builder import FleetModelBuilder, _metrics_dict, build_split_dict, redirect_definition
    golden = _golden()["builder"]
    # ModelBuilder's constructor and build() take what FleetModelBuilder takes (builder/utils.py:8-17 hands it the same
    # arguments: the standalone class keeps gordo's public contract)
    assert list(inspect.signature(FleetModelBuilder.__init__).parameters) == golden["signatures"]["__init__"]
    assert list(inspect.signature(FleetModelBuilder.build).parameters) == golden["signatures"]["build"]
    X = builder_frame()
    assert sorted(golden["cases"]) == sorted(BUILDER_EVALUATIONS)
    for name, evaluation in BUILDER_EVALUATIONS.items():
        want = golden["cases"][name]
        # the redirect maps the unmodified project YAML onto the mirror before _build resolves it
        resolved = redirect_definition(BUILDER_MODEL)
        assert json.loads(json.dumps(resolved)) == want["resolved_model"], name
        model = serializer.from_definition(resolved)
        assert describe(model) == want["model"], name
        # _build's model.cross_validate(X=X, y=y, scoring=..., return_estimator=True, cv=split_obj) (:272) binds
        call = {k: None for k in want["kwargs"]}
        inspect.signature(type(model).cross_validate).bind(model, **call)
        assert want["return_estimator"] is True and want["X_is_the_dataset"], name
        assert want["cv"] == describe(TimeSeriesSplit(n_splits=3)), name
        metrics = [m.rsplit(".", 1)[-1] for m in evaluation["metrics"]]
        scorers = {k for k in _metrics_dict(X, evaluation["scoring_scaler"])
                   if any(k == mm.replace("_", "-") or k.startswith(mm.replace("_", "-") + "-") for mm in metrics)}
        assert sorted(scorers) == want["scoring"], name
    got = build_split_dict(X, TimeSeriesSplit(n_splits=3))
    assert {k: str(v) for k, v in got.items()} == golden["split_metadata"]
