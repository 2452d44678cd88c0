"""
-m gpu tests of the round-2 work, all through the C-ABI / the plugin surface:
  * ff_fit on the topologies the advisor found rejected (feedforward_symmetric default dims, batch 128 at T >= 100)
    and batches larger than the thread block (accuracy history);
  * FleetBuild: a Machine's model is bit-identical whether it is built alone through the estimator API, in a
    bucket, or in a bucket that shares the device with other buckets on concurrent streams; equal to the
    per-Machine estimator-API build up to the float32 input scaling;
  * FleetModelBuilder seam: (model, machine) + the reference's BuildMetadata record, computed offsets;
  * FleetAnomalyServer: every transfer plan returns the same host columns as model.anomaly() per Machine;
  * two host threads hammering one model's .anomaly() (gordo.server's gthread workers share the model);
  * the bench's own data: Machine 0 of bench.py against the oracle, and the error distribution of the bf16 columns.
"""
import threading

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import dense, factories
from oracle.scaler import MinMaxScaler as OMinMax
from tests.gpu_util import make_fleet_case, oracle_score, fleet_from_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _i64(a):
    return torch.tensor(np.asarray(a, np.int64), device=DEV)


def _defn(est_kw=None, det="DiffBasedAnomalyDetector", det_kw=None, prefix="gordo_b200"):
    kw = {"kind": "feedforward_hourglass"}
    kw.update(est_kw or {})
    return {f"{prefix}.machine.model.anomaly.diff.{det}": dict(det_kw or {}, base_estimator={
        "sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler",
                                                {f"{prefix}.machine.model.models.KerasAutoEncoder": kw}]}})}


# ----------------------------------------------------------------------------- ff_fit: wide topologies, big batches
@pytest.mark.parametrize("kind,T,batch,kw", [
    ("feedforward_symmetric", 20, 32, {}),                       # default dims (256, 128, 64): 269 KB of activations
    ("feedforward_hourglass", 100, 128, {}),                     # examples/model-configuration.yaml batch_size at 100 tags
    ("feedforward_model", 12, 32, {}),                           # default encoding_dim / decoding_dim
])
def test_ff_fit_topologies_beyond_shared_memory_match_oracle(kind, T, batch, kw):
    from gordo_b200.fleet import FFFleet, FFTopology
    rng = np.random.default_rng(7 + T)
    spec = getattr(factories, kind)(T, **kw)
    topo = FFTopology(spec["widths"], spec["acts"], spec["l1"])
    fl = FFFleet(topo, 1, DEV)
    rows = [3 * batch + 5, 2 * batch]
    X = rng.random((sum(rows), T)).astype(np.float32)
    lo = np.concatenate([[0], np.cumsum(rows)[:-1]]); hi = np.cumsum(rows)
    inits = [dense.ff_flatten(dense.ff_init(spec, rng)) for _ in rows]
    perms = [[rng.permutation(r)] for r in rows]
    want, want_h = [], []
    for j, r in enumerate(rows):
        p = dense.ff_unflatten(inits[j], spec["widths"])
        h, _ = dense.ff_fit(spec, p, X[lo[j]:hi[j]], X[lo[j]:hi[j]], epochs=1, batch_size=batch, perms=perms[j])
        want.append(dense.ff_flatten(p)); want_h.append(h)
    params = torch.from_numpy(np.stack(inits)).to(DEV)
    pool = torch.from_numpy(np.concatenate([p[0] for p in perms]).astype(np.int32)).to(DEV)
    hl, ha, _, t = fl.fit_jobs(torch.from_numpy(X).to(DEV), None, _i64(lo), _i64(hi), params, epochs=1, batch_size=batch,
                               perm_pool=pool, perm_off=_i64(lo))
    torch.cuda.synchronize()
    for j in range(len(rows)):
        # Adam normalises every gradient to ~lr: a near-zero gradient whose fp32 summation order differs moves a weight
        # by a visible fraction of lr per step; a handful of 37 422 weights lands between 3e-4 and 6e-4
        np.testing.assert_allclose(params[j].cpu().numpy(), want[j], rtol=0, atol=6e-4, err_msg=f"job {j}")
        assert float(np.mean(np.abs(params[j].cpu().numpy() - want[j]))) < 2e-5
        np.testing.assert_allclose(hl[j].cpu().numpy(), want_h[j]["loss"], rtol=3e-4)
        np.testing.assert_allclose(ha[j].cpu().numpy(), want_h[j]["accuracy"], atol=2.0 / rows[j])


def test_ff_fit_accuracy_history_with_batch_larger_than_the_block():
    from gordo_b200.fleet import FFFleet, FFTopology
    rng = np.random.default_rng(3)
    spec = factories.feedforward_hourglass(3)
    topo = FFTopology(spec["widths"], spec["acts"], spec["l1"])
    fl = FFFleet(topo, 1, DEV)
    n, batch = 1500, 700                                          # > 512 threads per fit CTA
    X = rng.random((n, 3)).astype(np.float32)
    init = dense.ff_flatten(dense.ff_init(spec, rng))
    p = dense.ff_unflatten(init, spec["widths"])
    h, _ = dense.ff_fit(spec, p, X, X, epochs=2, batch_size=batch, perms=None)          # None = no shuffle
    params = torch.from_numpy(init[None].copy()).to(DEV)
    hl, ha, _, _ = fl.fit_jobs(torch.from_numpy(X).to(DEV), None, _i64([0]), _i64([n]), params, epochs=2, batch_size=batch)
    torch.cuda.synchronize()
    np.testing.assert_allclose(ha[0].cpu().numpy(), h["accuracy"], atol=2.0 / n)
    np.testing.assert_allclose(hl[0].cpu().numpy(), h["loss"], rtol=3e-4)


# ----------------------------------------------------------------------------- builder: seeds, streams, seam
def _machines(n, T, rows, seed0, est_kw=None, frame=True):
    from gordo_b200.builder import FleetMachine
    out = []
    for i in range(n):
        X = np.random.default_rng(seed0 + i).random((rows, T)).astype(np.float32)
        Xf = pd.DataFrame(X, columns=[f"t{j}" for j in range(T)]) if frame else X
        out.append(FleetMachine(f"m{i}", Xf, model=_defn(est_kw), evaluation={"seed": 11 + i}))
    return out


def _params(model):
    return model.base_estimator.steps[1][1].model.params


def test_batched_build_equals_the_per_machine_build():
    """
    The bucket a Machine shares must not change its model: same seeds, same draws, same kernel arithmetic --
    bit-identical between bucket compositions.  Against the per-Machine path through the estimator API the
    only difference is the input scaling (sklearn scales in float64 on the host and casts, the batched path
    fuses x * scale + min in float32 on the device): same initial weights and permutations, weights equal to ~1e-6.
    """
    from gordo_b200 import serializer
    from gordo_b200.builder import FleetBuild
    mcs = _machines(3, 6, 400, 50)
    batched = FleetBuild(mcs).build()
    assert all(meta["fleet"]["machines_in_launch"] == 3 for _, meta in batched)
    for mc, (model, meta) in zip(mcs, batched):
        alone_model, alone_meta = FleetBuild([mc])._build_one(serializer.from_definition(mc.definition()), mc)
        np.testing.assert_allclose(_params(model), _params(alone_model), rtol=0, atol=2e-5)
        np.testing.assert_allclose(model.feature_thresholds_.to_numpy(), alone_model.feature_thresholds_.to_numpy(), rtol=1e-3)
        np.testing.assert_allclose(model.aggregate_threshold_, alone_model.aggregate_threshold_, rtol=1e-3)
        assert meta["model_offset"] == alone_meta["model_offset"] == 0
    # another bucket composition, same Machine 1
    again = FleetBuild([mcs[1]]).build()
    np.testing.assert_array_equal(_params(again[0][0]), _params(batched[1][0]))


def test_concurrent_stream_buckets_equal_the_sequential_build():
    from gordo_b200.builder import FleetBuild
    mcs = []
    for T in (4, 5, 6, 7, 9):                                     # five topologies = five buckets
        mcs += _machines(2, T, 300, 100 + T)
    seq = FleetBuild(mcs, streams=1).build()
    par_builder = FleetBuild(mcs, streams=4)
    par = par_builder.build()
    assert par_builder.last_bucket_count == 5
    for (a, ma), (b, mb) in zip(seq, par):
        np.testing.assert_array_equal(_params(a), _params(b))
        np.testing.assert_array_equal(a.feature_thresholds_.to_numpy(), b.feature_thresholds_.to_numpy())
        assert a.aggregate_threshold_ == b.aggregate_threshold_
        assert ma["cross_validation"]["scores"].keys() == mb["cross_validation"]["scores"].keys()


def test_fleet_model_builder_seam_contract():
    """ModelBuilder's contract (build_model.py:104-190, 313-337): (model, machine), BuildMetadata layout, offsets."""
    from gordo_b200.builder import FleetMachine, FleetModelBuilder
    from gordo_b200.machine.model.anomaly.diff import DiffBasedAnomalyDetector
    X = pd.DataFrame(np.random.default_rng(1).random((300, 4)).astype(np.float32), columns=list("abcd"),
                     index=pd.date_range("2020-01-01", periods=300, freq="10min", tz="UTC"))
    # an UNMODIFIED gordo project definition (gordo.machine.model.* paths) builds on the mirror
    mc = FleetMachine("single", X, model=_defn(prefix="gordo"), evaluation={"seed": 2})
    model, machine = FleetModelBuilder(mc).build()
    assert type(model) is DiffBasedAnomalyDetector and machine.name == "single"
    bm = machine.build_metadata
    assert set(bm) == {"model", "dataset"}
    assert set(bm["model"]) == {"model_offset", "model_creation_date", "model_builder_version", "model_training_duration_sec",
                                "cross_validation", "model_meta"}
    assert bm["model"]["model_offset"] == 0 and bm["model"]["model_training_duration_sec"] > 0
    cv = bm["model"]["cross_validation"]
    assert set(cv) == {"cv_duration_sec", "scores", "splits"} and cv["cv_duration_sec"] > 0
    assert {"r2-score", "explained-variance-score-a", "mean-absolute-error-d"} <= set(cv["scores"])
    assert set(cv["scores"]["r2-score"]) == {"fold-mean", "fold-std", "fold-max", "fold-min", "fold-1", "fold-2", "fold-3"}
    assert "history" in bm["model"]["model_meta"] and "feature-thresholds" in bm["model"]["model_meta"]
    frame = model.anomaly(X, X, frequency=pd.Timedelta("10min"))
    assert ("total-anomaly-confidence", "") in frame.columns and len(frame) == 300
    # the fleet twin returns one (model, machine) per Machine, LSTM offsets computed from the output length
    lstm_def = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": {
        "sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler",
            {"gordo.machine.model.models.KerasLSTMAutoEncoder": {"kind": "lstm_hourglass", "lookback_window": 5}}]}}}}
    fleet = [FleetMachine(f"f{i}", X.iloc[:200 + 10 * i], model=_defn(prefix="gordo"), evaluation={"seed": i}) for i in range(3)]
    fleet.append(FleetMachine("l0", X.iloc[:120], model=lstm_def, evaluation={"seed": 4}))
    built = FleetModelBuilder.build_fleet(fleet, streams=2)
    assert [m.name for _, m in built] == ["f0", "f1", "f2", "l0"]
    assert [m.build_metadata["model"]["model_offset"] for _, m in built] == [0, 0, 0, 4]
    assert built[0][1].fleet_metadata["fleet"]["machines_in_launch"] == 3
    single_again, _ = FleetModelBuilder(fleet[1]).build()
    np.testing.assert_allclose(_params(single_again), _params(built[1][0]), rtol=0, atol=2e-5)      # seam single build == fleet build


# ----------------------------------------------------------------------------- serving
def test_fleet_anomaly_server_plans_match_per_machine_anomaly():
    from gordo_b200.builder import FleetBuild
    from gordo_b200.serving import FleetAnomalyServer
    T, rows = 6, [700, 333, 512, 129]
    mcs = []
    for i, n in enumerate(rows):
        m = _machines(1, T, n, 200 + i)[0]; m.name = f"s{i}"
        mcs.append(m)
    models = [m for m, _ in FleetBuild(mcs).build()]
    Xs = [np.random.default_rng(900 + i).random((n, T)).astype(np.float32) for i, n in enumerate(rows)]
    want = [mdl.anomaly(pd.DataFrame(X, columns=mc.X.columns), pd.DataFrame(X, columns=mc.X.columns))
            for mdl, mc, X in zip(models, mcs, Xs)]
    assert FleetAnomalyServer.group_by_topology(models).keys().__len__() == 1
    for plan in (0, 1, 1.5, 2, 3, "auto"):
        srv = FleetAnomalyServer.from_models(models, rows, precision="f32", n_chunks=3, plan=plan, n_threads=3)
        res = srv.anomaly(Xs)                                    # list of per-Machine host arrays (staged to pinned memory)
        if plan == "auto":
            assert 0 <= srv.plan <= 3 and len(srv.plan_timings) >= 4
        for m in range(len(rows)):
            c = res.machine(m)
            for name in ("model-output", "tag-anomaly-scaled", "tag-anomaly-unscaled", "anomaly-confidence"):
                np.testing.assert_allclose(c[name], want[m][name].to_numpy(), rtol=2e-5, atol=2e-6, err_msg=f"plan {plan} {name}")
            for name in ("total-anomaly-scaled", "total-anomaly-unscaled", "total-anomaly-confidence"):
                np.testing.assert_allclose(c[name], want[m][name].to_numpy().ravel(), rtol=2e-5, atol=1e-7, err_msg=f"plan {plan} {name}")
        frame = res.frame(1, tags=list(mcs[1].X.columns))
        assert list(frame.columns) == list(want[1].columns)
        np.testing.assert_allclose(frame["anomaly-confidence"].to_numpy(), want[1]["anomaly-confidence"].to_numpy(), rtol=2e-5, atol=2e-6)
        by = srv.bytes_per_call()
        k = srv.plan
        if float(k).is_integer():
            assert by["d2h"] == sum(rows) * ((4 - int(k)) * T + 3) * 4
        else:       # x.5: odd chunks derive one matrix more than even ones
            assert sum(rows) * ((4 - int(k) - 1) * T + 3) * 4 < by["d2h"] < sum(rows) * ((4 - int(k)) * T + 3) * 4
        assert by["h2d"] == sum(rows) * T * 4 and by["d2h"] + by["host_derived_bytes"] == sum(rows) * (4 * T + 3) * 4
        srv.close()
    # pinned input: zero-copy path, bf16 tensor-core scorer, device columns == host columns
    big = FleetAnomalyServer.from_models(models, rows, precision="bf16", n_chunks=2, plan=3)
    xp = torch.empty((sum(rows), T), dtype=torch.float32, pin_memory=True)
    xp.numpy()[:] = np.concatenate(Xs)
    r2 = big.anomaly(xp)
    assert r2.model_input is xp
    np.testing.assert_allclose(r2.columns["tag-anomaly-unscaled"].numpy(),
                               np.abs(r2.columns["model-output"].numpy() - xp.numpy()), rtol=0, atol=0)
    big.close()


def test_two_threads_share_one_model():
    """gordo.server: one lru-cached model object, gthread workers call .anomaly() concurrently (server/utils.py:334-335)."""
    from gordo_b200.builder import FleetBuild
    mcs = _machines(1, 8, 600, 321, est_kw={"precision": "bf16"})
    model = FleetBuild(mcs).build()[0][0]
    cols = list(mcs[0].X.columns)
    frames = [pd.DataFrame(np.random.default_rng(5000 + i).random((100 + 37 * (i % 5), 8)).astype(np.float32), columns=cols)
              for i in range(24)]
    want = [model.anomaly(f, f) for f in frames]
    for attr in ("_gb200_serving",):                               # cold caches: both threads race to create them
        model.__dict__.pop(attr, None)
        model.base_estimator.steps[1][1].__dict__.pop(attr, None)
    from gordo_b200.fleet import Schedule
    Schedule._single.clear()
    errors, got = [], [None] * len(frames)

    def worker(idxs):
        try:
            torch.cuda.set_device(0)
            for _ in range(3):
                for i in idxs:
                    got[i] = model.anomaly(frames[i], frames[i])
                    model.predict(frames[i])
        except Exception as e:            # noqa: BLE001
            errors.append(e)
    ts = [threading.Thread(target=worker, args=(range(k, len(frames), 2),)) for k in range(2)]
    [t.start() for t in ts]; [t.join() for t in ts]
    assert not errors, errors
    for g, w in zip(got, want):
        pd.testing.assert_frame_equal(g, w)


# ----------------------------------------------------------------------------- the bench's own data
def test_bench_machine_zero_against_the_oracle_and_bf16_error_distribution():
    """Machine 0 of bench.py's c2 workload (same bytes): fp32 columns vs the oracle on a 2 000-row slice; the bf16
    headline path's error on yhat and on the confidence columns as a distribution (p50 / p99 / max), not one bound."""
    import bench
    from gordo_b200.fleet import FFFleet, FFTopology, Schedule
    T, rows = 50, 100_000
    rng, X = bench.machine_data(0, rows, T)
    widths = bench.hourglass_widths(T)
    spec = factories.feedforward_hourglass(T)
    assert spec["widths"] == widths
    flat = bench.machine_params(rng, widths)
    ft, at = bench.machine_thresholds(rng, T)
    topo = FFTopology(spec["widths"], spec["acts"], spec["l1"])
    fl = FFFleet(topo, 1, DEV)
    fl.set_params(torch.from_numpy(flat[None]))
    xd = torch.from_numpy(X).to(DEV)
    fl.in_scale, fl.in_min = FFFleet.minmax_fit(xd, _i64([0]), _i64([rows]))
    fl.err_scale = fl.in_scale.clone()
    fl.feat_thr = torch.from_numpy(ft.astype(np.float32)[None]).to(DEV); fl.agg_thr = torch.tensor([at], dtype=torch.float32, device=DEV)
    sched = Schedule([rows])
    r32 = {k: v.cpu().numpy() for k, v in fl.score(sched, xd, precision="f32").items()}
    r16 = {k: v.cpu().numpy() for k, v in fl.score(sched, xd, precision="bf16").items()}
    sl = slice(40_000, 42_000)
    sx = OMinMax().fit(X)
    case = dict(spec=spec, X=[X[sl]], Y=[X[sl]], params=flat[None], in_scale=sx.scale_.astype(np.float32)[None],
                in_min=sx.min_.astype(np.float32)[None], err_scale=sx.scale_.astype(np.float32)[None],
                feat_thr=ft.astype(np.float32)[None], agg_thr=np.asarray([at], np.float32), row_counts=[2000])
    want = oracle_score(case, 0)
    for key, w in want.items():
        tol = dict(rtol=0, atol=2e-5) if key == "model-output" else dict(rtol=3e-4, atol=3e-6)
        np.testing.assert_allclose(r32[key][sl], w, err_msg=f"fp32 {key}", **tol)
    # bf16 tensor-core path vs the fp32 path over ALL 100 000 rows
    dist = {}
    for key in ("model-output", "anomaly-confidence", "total-anomaly-confidence"):
        e = np.abs(r16[key].astype(np.float64) - r32[key].astype(np.float64)).ravel()
        dist[key] = (float(np.percentile(e, 50)), float(np.percentile(e, 99)), float(e.max()))
    print("bf16 vs fp32 |error| p50 / p99 / max:", dist)
    assert dist["model-output"][0] < 4e-3 and dist["model-output"][1] < 1.5e-2 and dist["model-output"][2] < 3e-2
    # confidence = |yhat - y| / threshold with thresholds in [0.1, 0.5]: the yhat error divided by >= 0.1
    assert dist["anomaly-confidence"][1] < 0.15 and dist["anomaly-confidence"][2] < 0.3
    rel = np.abs(r16["total-anomaly-confidence"] - r32["total-anomaly-confidence"]) / np.abs(r32["total-anomaly-confidence"])
    assert float(np.percentile(rel, 99)) < 0.05


# ----------------------------------------------------------------------------- fp32-grade tensor-core scorer (f16x3)
X3_CASES = {
    "c1_1x10x1000": dict(seed=1, row_counts=[1000], T=10),
    "ragged_small_T9": dict(seed=2, row_counts=[1, 127, 128, 129, 0, 1000, 5], T=9),
    "c2_shape_3x50": dict(seed=3, row_counts=[4096, 1003, 2500], T=50),
    "sigmoid_T33_E2": dict(seed=6, row_counts=[513], T=33, func="sigmoid", encoding_layers=2),
    "separate_y_T12_to_4": dict(seed=7, row_counts=[400, 333], T=12, T_out=4),
    "T64": dict(seed=12, row_counts=[700, 300], T=64),
    "no_thresholds_T20": dict(seed=13, row_counts=[640, 64], T=20, thresholds=False),
}


@pytest.mark.parametrize("name", list(X3_CASES))
def test_ff_score_f16x3_is_fp32_grade(name):
    """GB200_PREC_F16X3_TC (hi + lo fp16 operands, 3 MMAs per K step) against the fp32 oracle at the fp32 kernel's
    own tolerance: 2e-5 abs on yhat -- 1 000x tighter than the bf16 path's bound."""
    from tests.test_gpu_ff_score import _compare
    case = make_fleet_case(**X3_CASES[name])
    fl, sched, X, Y = fleet_from_case(case)
    assert fl.tc_eligible("f16x3") and fl.auto_precision("f16x3") == "f16x3"
    res = fl.score(sched, X, Y, precision="f16x3")
    torch.cuda.synchronize()
    _compare(res, case, None, 2e-5, 2e-4, 2e-6)
    r32 = fl.score(sched, X, Y, precision="f32")
    e = (res["model-output"] - r32["model-output"]).abs()
    if e.numel():
        print(name, "f16x3 vs fp32 kernel |yhat err| max / mean:", float(e.max()), float(e.mean()))
        assert float(e.max()) < 2e-5 * max(1.0, float(r32["model-output"].abs().max()))


def test_ff_score_f16x3_eligibility_and_input_range():
    from gordo_b200.fleet import FFFleet, FFTopology, Schedule
    relu = make_fleet_case(seed=5, row_counts=[64], T=20, func="relu")
    fl, _, _, _ = fleet_from_case(relu)
    assert not fl.tc_eligible("f16x3") and fl.auto_precision("f16x3") == "f32" and fl.tc_eligible("bf16")
    wide = make_fleet_case(seed=5, row_counts=[64], T=100)          # hi + lo images of 100 tags exceed shared memory
    fw, _, _, _ = fleet_from_case(wide)
    assert not fw.tc_eligible("f16x3") and fw.auto_precision("f16x3") == "f32" and fw.tc_eligible("bf16")
    # inputs far outside fp16 range and NaNs: the per-row power-of-two scale keeps every finite row equal to the
    # fp32 kernel; a NaN input poisons its own row only
    case = make_fleet_case(seed=21, row_counts=[256], T=10)
    fl, sched, X, Y = fleet_from_case(case)
    Xb = X.clone()
    Xb[3] = 1e9; Xb[7, 2] = float("nan"); Xb[11] = -3e7
    a = fl.score(sched, Xb, None, precision="f16x3")["model-output"]
    b = fl.score(sched, Xb, None, precision="f32")["model-output"]
    ok = torch.ones(256, dtype=torch.bool, device=X.device); ok[[3, 7, 11]] = False
    np.testing.assert_allclose(a[ok].cpu().numpy(), b[ok].cpu().numpy(), rtol=0, atol=2e-5)
    assert bool(torch.isnan(a[7]).all()) and bool(torch.isfinite(a[3]).all()) and bool(torch.isfinite(a[11]).all())
    np.testing.assert_allclose(a[[3, 11]].cpu().numpy(), b[[3, 11]].cpu().numpy(), rtol=0, atol=2e-5)
    Xc = X.clone(); Xc[5] *= 4e5; Xc[9, 3] = 7e4                    # just past fp16's range, mixed magnitudes in one row
    a2 = fl.score(sched, Xc, None, precision="f16x3")["model-output"]
    b2 = fl.score(sched, Xc, None, precision="f32")["model-output"]
    np.testing.assert_allclose(a2.cpu().numpy(), b2.cpu().numpy(), rtol=0, atol=2e-5)


def test_estimator_and_detector_with_f16x3_precision():
    """precision="f16x3" from the Machine YAML: predict / anomaly agree with the exact fp32 path to 2e-5."""
    from gordo_b200.builder import FleetBuild
    frames = {}
    for prec in ("f32", "f16x3"):
        mcs = _machines(1, 12, 500, 77, est_kw={"precision": prec})
        model = FleetBuild(mcs).build()[0][0]
        frames[prec] = model.anomaly(mcs[0].X, mcs[0].X)
    for col in ("model-output", "tag-anomaly-unscaled", "anomaly-confidence", "total-anomaly-confidence"):
        np.testing.assert_allclose(frames["f16x3"][col].to_numpy(), frames["f32"][col].to_numpy(), rtol=2e-4, atol=3e-5, err_msg=col)


def test_anomaly_response_bodies_equal_the_frame_codecs():
    """model.anomaly_response (column groups -> parquet bytes / JSON dict) == the server codecs applied to model.anomaly's
    frame (gordo/server/blueprints/anomaly.py:57-72), incl. the smooth-* columns the view drops by default."""
    import json
    from gordo_b200.builder import FleetBuild
    from gordo_b200.server import utils as su
    from gordo_b200.builder import FleetMachine
    X = pd.DataFrame(np.random.default_rng(3).random((400, 5)).astype(np.float32), columns=[f"tag {j}" for j in range(5)],
                     index=pd.date_range("2020-01-01", periods=400, freq="10min", tz="UTC"))
    model = FleetBuild([FleetMachine("m", X, model=_defn(det_kw={"window": 12}), evaluation={"seed": 1})]).build()[0][0]
    req = X.iloc[:100]
    freq = pd.Timedelta("10min")
    frame = model.anomaly(req, req, frequency=freq)
    assert any(c[0].startswith("smooth-") for c in frame.columns)
    dropped = frame.drop(columns=[c for c in frame.columns if c[0].startswith("smooth-")])
    got = su.dataframe_from_parquet_bytes(model.anomaly_response(req, req, frequency=freq, fmt="parquet"))
    pd.testing.assert_frame_equal(got, su.dataframe_from_parquet_bytes(su.dataframe_into_parquet_bytes(dropped)))
    full = su.dataframe_from_parquet_bytes(model.anomaly_response(req, req, frequency=freq, fmt="parquet", all_columns=True))
    pd.testing.assert_frame_equal(full, su.dataframe_from_parquet_bytes(su.dataframe_into_parquet_bytes(frame)))
    d = model.anomaly_response(req, req, frequency=freq, fmt="json")
    assert json.dumps(d, sort_keys=True, default=str) == json.dumps(su.dataframe_to_dict(dropped), sort_keys=True, default=str)


def test_fleet_anomaly_server_with_separate_targets():
    """model.anomaly(X, y) with y != X (target tags differ from the input tags, T_out != T): host targets are staged and
    copied per chunk, the host expansion uses them; every plan equals the device-resident columns."""
    from gordo_b200.serving import FleetAnomalyServer
    case = make_fleet_case(seed=7, row_counts=[400, 333, 129], T=12, T_out=4)
    fl, sched, X, Y = fleet_from_case(case)
    want = fl.score(sched, X, Y, precision="f32")
    Xh = [x for x in case["X"]]; Yh = [y for y in case["Y"]]
    for plan in (0, 2, 3):
        srv = FleetAnomalyServer(fl, case["row_counts"], precision="f32", n_chunks=2, plan=plan, n_threads=2)
        res = srv.anomaly(Xh, Yh)
        for k, w in want.items():
            np.testing.assert_allclose(res.columns[k].numpy(), w.cpu().numpy(), rtol=1e-5, atol=1e-6, err_msg=f"plan {plan} {k}")
        assert res.machine(1)["model-input"].shape == (333, 12) and res.machine(1)["model-output"].shape == (333, 4)
        assert srv.bytes_per_call()["h2d"] == sum(case["row_counts"]) * (12 + 4) * 4
        with pytest.raises(ValueError):
            srv.anomaly(Xh)                                       # y cannot default to X when the widths differ
        srv.close()


@pytest.mark.gpu
def test_kfcv_detector_over_transformed_target_regressor():
    """The reference's third serializability config (test_anomaly_detectors.py:508-538) run, not just parsed:
    DiffBasedKFCVAnomalyDetector over TransformedTargetRegressor(MinMaxScaler, Pipeline[MinMaxScaler, KerasAutoEncoder
    with validation_split + EarlyStopping]).  This composition has no fused route (the target transformer sits outside
    the Pipeline), so it exercises the generic sklearn path through the GPU estimator: K-fold cross_validate, fit,
    anomaly() with smoothing + percentile thresholds; the estimator inside must equal a manual composition."""
    import yaml
    from sklearn.model_selection import KFold
    from gordo_b200 import serializer
    cfg = yaml.safe_load("""
    gordo.machine.model.anomaly.diff.DiffBasedKFCVAnomalyDetector:
        base_estimator:
            sklearn.compose.TransformedTargetRegressor:
                transformer:
                    sklearn.preprocessing.MinMaxScaler
                regressor:
                    sklearn.pipeline.Pipeline:
                        steps:
                        - sklearn.preprocessing.MinMaxScaler
                        - gordo.machine.model.models.KerasAutoEncoder:
                            kind: feedforward_hourglass
                            batch_size: 128
                            compression_factor: 0.5
                            encoding_layers: 1
                            func: tanh
                            out_func: linear
                            optimizer: Adam
                            loss: mse
                            epochs: 12
                            validation_split: 0.1
                            callbacks:
                                - tensorflow.keras.callbacks.EarlyStopping:
                                    monitor: val_loss
                                    patience: 3
                                    restore_best_weights: true
        scaler: sklearn.preprocessing.MinMaxScaler
        window: 24
        shuffle: true
        threshold_percentile: 0.975
    """)
    rng = np.random.default_rng(5)
    t = np.arange(1500)[:, None]
    X = pd.DataFrame((np.sin(t / 50.0 + np.arange(6)) * np.arange(1, 7) + 0.05 * rng.standard_normal((1500, 6))).astype(np.float32),
                     index=pd.date_range("2020-01-01", periods=1500, freq="10min", tz="UTC"), columns=[f"tag-{i}" for i in range(6)])
    torch.manual_seed(0); np.random.seed(0)
    model = serializer.from_definition(cfg, redirect_gordo=True)
    cv = model.cross_validate(X=X, y=X, cv=KFold(n_splits=3, shuffle=True, random_state=0))
    assert len(cv["estimator"]) == 3
    assert np.isfinite(model.aggregate_threshold_) and model.aggregate_threshold_ > 0
    assert np.asarray(model.feature_thresholds_).shape == (6,) and np.isfinite(np.asarray(model.feature_thresholds_)).all()
    model.fit(X, X)
    est = model.base_estimator.regressor_.steps[1][1]
    hist = est.get_metadata()["history"]
    assert "val_loss" in hist and 1 <= len(hist["loss"]) <= 12 and hist["loss"][-1] < hist["loss"][0]
    frame = model.anomaly(X, X)
    assert {"model-input", "model-output", "tag-anomaly-scaled", "tag-anomaly-unscaled", "total-anomaly-scaled",
            "total-anomaly-unscaled", "smooth-tag-anomaly-scaled", "smooth-total-anomaly-scaled",
            "anomaly-confidence", "total-anomaly-confidence"} <= set(frame.columns.get_level_values(0))
    # the TransformedTargetRegressor inverts the target scaling: model-output lives in the units of y and is the
    # manual composition of the fitted parts
    inner = model.base_estimator
    manual = inner.transformer_.inverse_transform(inner.regressor_.predict(X))
    np.testing.assert_allclose(frame["model-output"].to_numpy(), manual, rtol=1e-5, atol=1e-5)
    err = np.abs(frame["model-output"].to_numpy() - X.to_numpy())
    np.testing.assert_allclose(frame["tag-anomaly-unscaled"].to_numpy(), err, rtol=1e-5, atol=1e-6)
    conf = frame["total-anomaly-confidence"].to_numpy().ravel()
    want = frame["total-anomaly-scaled"].to_numpy().ravel() / model.aggregate_threshold_      # diff.py:436-441: not the smoothed one
    np.testing.assert_allclose(conf, want, rtol=1e-5)
    assert np.isnan(frame["smooth-total-anomaly-scaled"].to_numpy()[:23]).all() and \
        np.isfinite(frame["smooth-total-anomaly-scaled"].to_numpy()[23:]).all()               # rolling(24).median()
