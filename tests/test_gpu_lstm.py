"""
-m gpu parity tests of the LSTM path (gb200_lstm_predict / gb200_lstm_fit through gordo_b200.lstm
and the KerasLSTM* estimators) against the oracle on the same seeded inputs and weights.
fp32 kernels: |yhat - oracle| <= 3e-5 abs; after the primer + a few Adam steps weights <= 3e-4 abs.
"""
import numpy as np
import pandas as pd
import pytest
import torch

from oracle import factories, lstm as olstm
from oracle.scaler import MinMaxScaler as OMinMax

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _spec(T, L, enc=(6, 3), dec=(3, 5), funcs=("tanh", "tanh"), T_out=None, out_func="linear"):
    return factories.lstm_model(T, T_out, lookback_window=L, encoding_dim=enc, encoding_func=funcs,
                                decoding_dim=dec, decoding_func=funcs, out_func=out_func)


def _topo(spec):
    from gordo_b200.lstm import LSTMTopology
    return LSTMTopology(spec["n_features"], spec["n_features_out"], spec["units"], spec["acts"], spec["out_func"],
                        spec["lookback_window"])


@pytest.mark.parametrize("lookahead,L,funcs", [(0, 5, ("tanh", "tanh")), (1, 4, ("relu", "tanh")), (0, 1, ("tanh", "sigmoid"))])
def test_lstm_predict_matches_oracle(lookahead, L, funcs):
    from gordo_b200.fleet import Schedule
    from gordo_b200.lstm import LSTMFleet
    rng = np.random.default_rng(3)
    T, rows = 4, [60, 37, 90]
    spec = _spec(T, L, funcs=funcs)
    topo = _topo(spec)
    Xs = [rng.random((n, T)).astype(np.float32) * 4 - 1 for n in rows]
    P = [olstm.lstm_init(spec, rng) for _ in rows]
    scal = [OMinMax().fit(X) for X in Xs]
    fl = LSTMFleet(topo, len(rows), lookahead, DEV)
    fl.set_params(torch.from_numpy(np.stack([olstm.lstm_flatten(p) for p in P])))
    fl.in_scale = torch.from_numpy(np.stack([s.scale_ for s in scal]).astype(np.float32)).to(DEV)
    fl.in_min = torch.from_numpy(np.stack([s.min_ for s in scal]).astype(np.float32)).to(DEV)
    out, off = fl.predict(Schedule(rows), torch.from_numpy(np.concatenate(Xs)).to(DEV), max_windows=40)   # forces chunking
    torch.cuda.synchronize()
    for m, (X, p, s) in enumerate(zip(Xs, P, scal)):
        want = olstm.lstm_predict(spec, p, s.transform(X).astype(np.float32), L, lookahead)
        got = out[off[m]:off[m + 1]].cpu().numpy()
        assert got.shape == want.shape == (rows[m] - L + 1 - lookahead, T)          # models.py:618-660
        np.testing.assert_allclose(got, want, atol=3e-5)


def test_lstm_predict_wider_layers_and_tile_edges():
    from gordo_b200.fleet import Schedule
    from gordo_b200.lstm import LSTMFleet
    rng = np.random.default_rng(4)
    T, L, n = 20, 6, 150
    spec = factories.lstm_hourglass(T, lookback_window=L)            # units 17-13-10-10-13-17 (> one 16-unit tile)
    X = rng.random((n, T)).astype(np.float32)
    p = olstm.lstm_init(spec, rng)
    fl = LSTMFleet(_topo(spec), 1, 0, DEV)
    fl.set_params(torch.from_numpy(olstm.lstm_flatten(p)[None]))
    out, _ = fl.predict(Schedule([n]), torch.from_numpy(X).to(DEV))
    np.testing.assert_allclose(out.cpu().numpy(), olstm.lstm_predict(spec, p, X, L, 0), atol=3e-5)


@pytest.mark.parametrize("lookahead", [0, 1])
def test_lstm_fit_matches_oracle(lookahead):
    from gordo_b200.lstm import LSTMFleet
    rng = np.random.default_rng(5)
    T, L, B, epochs = 3, 4, 8, 2
    spec = _spec(T, L, enc=(5,), dec=(4,), funcs=("tanh",))
    rows = [45, 30]
    X = rng.random((sum(rows), T)).astype(np.float32)
    Y = rng.random((sum(rows), T)).astype(np.float32)
    lo = np.array([0, rows[0]]); hi = np.array([rows[0], sum(rows)])
    inits = [olstm.lstm_init(spec, rng) for _ in rows]
    want, hist = [], []
    for j in range(2):
        p = olstm.lstm_unflatten(olstm.lstm_flatten(inits[j]), spec)
        hp, hm, _ = olstm.lstm_fit(spec, p, X[lo[j]:hi[j]], Y[lo[j]:hi[j]], lookback_window=L, lookahead=lookahead,
                                   batch_size=B, epochs=epochs)
        want.append(olstm.lstm_flatten(p)); hist.append((hp, hm))
    fl = LSTMFleet(_topo(spec), 2, lookahead, DEV)
    params = torch.from_numpy(np.stack([olstm.lstm_flatten(p) for p in inits])).to(DEV)
    hl, pl = fl.fit_jobs(torch.from_numpy(X).to(DEV), torch.from_numpy(Y).to(DEV), lo, hi, params, epochs=epochs, batch_size=B)
    torch.cuda.synchronize()
    for j in range(2):
        np.testing.assert_allclose(params[j].cpu().numpy(), want[j], atol=3e-4, err_msg=f"job {j}")
        np.testing.assert_allclose(float(pl[j]), hist[j][0]["loss"][0], rtol=1e-4)
        np.testing.assert_allclose(hl[j].cpu().numpy(), hist[j][1]["loss"], rtol=1e-3)


def test_lstm_estimators_surface():
    """tests/gordo/machine/model/test_model.py:161-236, 324-338; test_builder.py:99-115 offsets."""
    from gordo_b200.machine.model.models import KerasLSTMAutoEncoder, KerasLSTMForecast
    rng = np.random.default_rng(6)
    xTrain, yTrain = rng.random((5, 3)), rng.random((5, 3))
    model = KerasLSTMAutoEncoder(kind="lstm_model", lookback_window=3, encoding_dim=(4,), encoding_func=("tanh",),
                                 decoding_dim=(4,), decoding_func=("tanh",)).fit(xTrain, yTrain)
    assert model.predict(rng.random((4, 3))).shape == (2, 3)             # test_lstmae_predict_output
    with pytest.raises(ValueError):                                      # lookback_window >= rows
        model.predict(xTrain[-3:-1, :])
    with pytest.raises(ValueError):
        KerasLSTMAutoEncoder(kind="lstm_model", lookback_window=11).fit(rng.random(10), rng.random(10))
    for lb in (5, 6):
        with pytest.raises(ValueError):
            KerasLSTMForecast(kind="lstm_model", lookback_window=lb).fit(rng.random((5, 2)), rng.random((5, 2)))
    # 1-D arrays are reshaped (test_keras_ae_reshapes_array / forecast)
    X1 = rng.random(100)
    small = dict(encoding_dim=(3,), encoding_func=("tanh",), decoding_dim=(3,), decoding_func=("tanh",))
    KerasLSTMAutoEncoder(kind="lstm_model", **small).fit(X1, X1).predict(X1)
    f = KerasLSTMForecast(kind="lstm_symmetric", lookback_window=13, dims=(4,), funcs=("tanh",)).fit(rng.random((100, 2)), rng.random((100, 2)))
    X = rng.random((100, 2))
    assert len(X) - len(f.predict(X)) == 13                              # Forecast L=13 -> offset 13
    a = KerasLSTMAutoEncoder(kind="lstm_hourglass", lookback_window=10, epochs=2).fit(X, X)
    assert len(X) - len(a.predict(X)) == 9                               # LSTM-AE L=10 -> offset 9
    md = a.get_metadata()
    assert md["forecast_steps"] == 0 and len(md["history"]["loss"]) == 1 and len(a.history_main_["loss"]) == 2
    assert a.score(X, X) <= 1.0
    import pickle
    b = pickle.loads(pickle.dumps(a))
    assert np.allclose(b.predict(X), a.predict(X))


def test_lstm_detector_offsets_in_anomaly_frame():
    from gordo_b200.machine.model.anomaly.diff import DiffBasedAnomalyDetector
    from gordo_b200.machine.model.models import KerasLSTMAutoEncoder
    rng = np.random.default_rng(7)
    X = pd.DataFrame(rng.random((120, 3)), columns=list("abc"), index=pd.date_range("2021-01-01", periods=120, freq="1min"))
    np.random.seed(0)
    det = DiffBasedAnomalyDetector(base_estimator=KerasLSTMAutoEncoder(kind="lstm_hourglass", lookback_window=6), require_thresholds=False)
    det.fit(X, X)
    f = det.anomaly(X, X)
    assert len(f) == 115 and f.index[0] == X.index[5]                    # aligned to the LAST len(output) rows
    np.testing.assert_array_equal(f["model-input"].to_numpy(), X.to_numpy()[5:])
    d = np.abs(f["model-output"].to_numpy() - X.to_numpy()[5:])
    np.testing.assert_allclose(f["tag-anomaly-unscaled"].to_numpy(), d, rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("T,L,units,funcs", [(20, 6, None, "tanh"), (7, 9, (40, 18), "tanh"), (5, 4, (3,), "relu")])
def test_lstm_predict_tensor_core_path(T, L, units, funcs):
    """
    tcgen05 step kernel (bf16 operands, fp32 accumulate + cell state, tanh.approx gates) against the
    fp32 oracle.  Stated tolerance: 3e-2 abs on O(1) outputs after L recurrent steps through the stack
    (bf16 rounding of h at every step); mean error <= 5e-3.
    """
    from gordo_b200.fleet import Schedule
    from gordo_b200.lstm import LSTMFleet
    rng = np.random.default_rng(40 + T)
    rows = [300, 129, 140 + L]
    if units is None:
        spec = factories.lstm_hourglass(T, lookback_window=L, func=funcs)
    else:
        spec = factories.lstm_symmetric(T, lookback_window=L, dims=units, funcs=tuple([funcs] * len(units)))
    Xs = [rng.random((n, T)).astype(np.float32) * 3 - 1 for n in rows]
    P = [olstm.lstm_init(spec, rng) for _ in rows]
    scal = [OMinMax().fit(X) for X in Xs]
    fl = LSTMFleet(_topo(spec), len(rows), 0, DEV)
    assert fl.tc_eligible()
    fl.set_params(torch.from_numpy(np.stack([olstm.lstm_flatten(p) for p in P])))
    fl.in_scale = torch.from_numpy(np.stack([s.scale_ for s in scal]).astype(np.float32)).to(DEV)
    fl.in_min = torch.from_numpy(np.stack([s.min_ for s in scal]).astype(np.float32)).to(DEV)
    X = torch.from_numpy(np.concatenate(Xs)).to(DEV)
    out, off = fl.predict(Schedule(rows), X, max_windows=256, precision="bf16")      # 300 rows -> 2 chunks
    ref, _ = fl.predict(Schedule(rows), X, precision="f32")
    torch.cuda.synchronize()
    for m, (Xm, p, s) in enumerate(zip(Xs, P, scal)):
        want = olstm.lstm_predict(spec, p, s.transform(Xm).astype(np.float32), L, 0)
        got = out[off[m]:off[m + 1]].cpu().numpy()
        assert got.shape == want.shape
        scale = max(1.0, float(np.abs(want).max()))
        np.testing.assert_allclose(got, want, atol=3e-2 * scale, err_msg=f"machine {m}")
        assert float(np.abs(got - want).mean()) < 5e-3 * scale
    assert float((out - ref).abs().max()) < 3e-2 * max(1.0, float(ref.abs().max()))


def test_lstm_detector_fused_scoring_matches_generic_path():
    """Pipeline[MinMaxScaler, KerasLSTMAutoEncoder]: GPU predict + gb200_score_outputs == host arithmetic."""
    from sklearn.pipeline import Pipeline
    from sklearn.preprocessing import MinMaxScaler, RobustScaler
    from gordo_b200.machine.model.anomaly.diff import DiffBasedAnomalyDetector
    from gordo_b200.machine.model.models import KerasLSTMAutoEncoder
    rng = np.random.default_rng(8)
    X = pd.DataFrame(rng.random((150, 4)) * [1, 10, 100, 0.1], columns=list("abcd"))
    np.random.seed(1)
    det = DiffBasedAnomalyDetector(base_estimator=Pipeline([("s", MinMaxScaler()), ("m", KerasLSTMAutoEncoder(
        kind="lstm_hourglass", lookback_window=5))]))
    det.cross_validate(X=X, y=X); det.fit(X, X)
    assert det._fused_plan() is not None
    f = det.anomaly(X, X)
    assert len(f) == 146
    out = det.predict(X)                                          # generic path pieces on the host
    np.testing.assert_allclose(f["model-output"].to_numpy(), out, atol=1e-6)
    d = np.abs(out.astype(np.float64) - X.to_numpy()[4:])
    s = np.abs(det.scaler.transform(pd.DataFrame(out, columns=X.columns)) - det.scaler.transform(X)[4:])
    np.testing.assert_allclose(f["tag-anomaly-unscaled"].to_numpy(), d, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(f["tag-anomaly-scaled"].to_numpy(), s, rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(f["total-anomaly-scaled"].to_numpy().ravel(), (s ** 2).mean(1), rtol=1e-4, atol=1e-8)
    np.testing.assert_allclose(f["anomaly-confidence"].to_numpy(), d / det.feature_thresholds_.to_numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(f["total-anomaly-confidence"].to_numpy().ravel(), (s ** 2).mean(1) / det.aggregate_threshold_, rtol=1e-4, atol=1e-7)
    # bf16 tensor-core inference selectable from the model kwargs
    det.base_estimator.steps[1][1].kwargs["precision"] = "bf16"
    fb = det.anomaly(X, X)
    assert float(np.abs(fb["model-output"].to_numpy() - f["model-output"].to_numpy()).max()) < 3e-2


def test_fleet_builder_lstm_bucket_matches_oracle():
    """Batched LSTM build (all folds + final fits in one gb200_lstm_fit, fold scoring on the device) vs the oracle."""
    from gordo_b200.builder import FleetBuild, FleetMachine, FleetModelBuilder
    from gordo_b200.lstm import LSTMTopology
    from oracle.anomaly import DiffDetector, LSTMBase
    T, L, rows = 3, 4, [120, 96]
    rng = np.random.default_rng(50)
    Xs = [rng.random((n, T)).astype(np.float32) * [1, 5, 0.2] for n in rows]
    defn = {"gordo_b200.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": {
        "sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler",
            {"gordo_b200.machine.model.models.KerasLSTMAutoEncoder": {
                "kind": "lstm_symmetric", "lookback_window": L, "batch_size": 16, "dims": [4], "funcs": ["tanh"]}}]}}}}
    mcs = [FleetMachine(f"m{i}", pd.DataFrame(X, columns=list("abc")), model=defn, evaluation={"seed": 9}) for i, X in enumerate(Xs)]
    built = FleetBuild(mcs).build()
    spec = factories.lstm_symmetric(T, lookback_window=L, dims=(4,), funcs=("tanh",))
    topo = LSTMTopology(T, T, spec["units"], spec["acts"], "linear", L)
    from tests.test_gpu_estimators import _builder_init
    init = _builder_init(topo.init_params, 9, len(rows), 4)
    for m, ((model, meta), X) in enumerate(zip(built, Xs)):
        Xd = X.astype(np.float64)
        det = DiffDetector(lambda tag, m=m: LSTMBase(spec, olstm.lstm_unflatten(
            init[m * 4 + (3 if tag == "final" else int(tag[-1]))], spec), lookback_window=L, batch_size=16))
        det.cross_validate(Xd, Xd); det.fit(Xd, Xd)
        est = model.base_estimator.steps[1][1]
        np.testing.assert_allclose(est.model.params, olstm.lstm_flatten(det.base.params), atol=3e-4)
        np.testing.assert_allclose(model.feature_thresholds_.to_numpy(), det.feature_thresholds_, rtol=5e-3, atol=1e-5)
        np.testing.assert_allclose(model.aggregate_threshold_, det.aggregate_threshold_, rtol=5e-3)
        assert meta["model_offset"] == L - 1 and meta["fleet"]["fit_jobs"] == 8
        f = model.anomaly(mcs[m].X, mcs[m].X)
        want = det.anomaly(Xd, Xd)
        assert len(f) == rows[m] - L + 1
        np.testing.assert_allclose(f["total-anomaly-confidence"].to_numpy().ravel(), want["total-anomaly-confidence"], rtol=2e-2, atol=1e-4)


def test_lstm_fit_on_a_side_stream_stops_finished_jobs():
    """A fit on a non-default stream: jobs of different lengths share the steps of one launch, and the device-side
    batch cursor stops each job stepping when it runs out of windows."""
    from gordo_b200.lstm import LSTMFleet
    rng = np.random.default_rng(15)
    T, L, B = 4, 5, 8
    spec = _spec(T, L, enc=(6,), dec=(5,), funcs=("tanh",))
    rows = [120, 61, 90]
    X = torch.from_numpy(rng.random((sum(rows), T)).astype(np.float32)).to(DEV)
    lo = np.concatenate([[0], np.cumsum(rows)[:-1]]); hi = np.cumsum(rows)
    init = torch.from_numpy(np.stack([olstm.lstm_flatten(olstm.lstm_init(spec, rng)) for _ in rows])).to(DEV)
    fl = LSTMFleet(_topo(spec), 3, 0, DEV)
    side = torch.cuda.Stream()
    p = init.clone()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        fl.fit_jobs(X, X, lo, hi, p, epochs=2, batch_size=B)
    side.synchronize()
    got = p.cpu().numpy()
    # the shortest job equals the oracle (it must not keep stepping after its last batch)
    pj = olstm.lstm_unflatten(init[1].cpu().numpy(), spec)
    Xj = X[lo[1]:hi[1]].cpu().numpy()
    olstm.lstm_fit(spec, pj, Xj, Xj, lookback_window=L, lookahead=0, batch_size=B, epochs=2)
    np.testing.assert_allclose(got[1], olstm.lstm_flatten(pj), atol=3e-4)
