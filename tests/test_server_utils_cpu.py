"""
§8 f-4 wire formats (CPU): gordo_b200.server.utils against what the reference's own gordo/server/utils.py produced
(tests/golden/server_codec_golden.json, recorded by tests/golden/make_server_codec_golden.py), and the
fleet fast paths (column groups -> parquet bytes / nested dict without the DataFrame pivot) against the frame path.
"""
import base64
import io
import json
import os

import numpy as np
import pandas as pd
import pytest

from gordo_b200.machine.model import utils as mu
from gordo_b200.server import utils as su

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _groups(n=40, T=3, seed=0):
    rng = np.random.default_rng(seed)
    tags = ["tag 1", "tag-2", "t3"][:T]
    return [("model-input", rng.random((n, T)), tags), ("model-output", rng.random((n, T)).astype(np.float32), tags),
            ("tag-anomaly-scaled", rng.random((n, T)), tags), ("total-anomaly-scaled", rng.random(n), None),
            ("tag-anomaly-unscaled", rng.random((n, T)), tags), ("total-anomaly-unscaled", rng.random(n), None),
            ("anomaly-confidence", rng.random((n, T)), tags), ("total-anomaly-confidence", rng.random(n), None)]


@pytest.mark.parametrize("with_time", [True, False])
def test_column_fast_paths_equal_the_frame_path(with_time):
    groups = _groups()
    index = pd.date_range("2020-03-01", periods=40, freq="10min", tz="UTC") if with_time else None
    freq = pd.Timedelta("10min") if with_time else None
    df = mu.assemble_frame(groups, index, freq)
    a = su.dataframe_from_parquet_bytes(su.dataframe_into_parquet_bytes(df))
    b = su.dataframe_from_parquet_bytes(su.columns_into_parquet_bytes(groups, index, freq))
    pd.testing.assert_frame_equal(a, b)
    pd.testing.assert_frame_equal(a, df, check_freq=False)
    assert list(b.columns) == list(df.columns) and isinstance(b.columns, pd.MultiIndex)
    d1, d2 = su.dataframe_to_dict(df), su.columns_to_dict(groups, index, freq)
    assert json.dumps(d1, sort_keys=True, default=str) == json.dumps(d2, sort_keys=True, default=str)
    back = su.dataframe_from_dict(json.loads(json.dumps(d2, default=str)))
    np.testing.assert_allclose(back["tag-anomaly-scaled"].to_numpy(), df["tag-anomaly-scaled"].to_numpy())
    assert len(back) == 40 and back.index.is_monotonic_increasing
    # a longer input than output (LSTM offset): the frame keeps the last len(output) index entries
    if with_time:
        long_index = pd.date_range("2020-03-01", periods=50, freq="10min", tz="UTC")
        c = su.dataframe_from_parquet_bytes(su.columns_into_parquet_bytes(groups, long_index, freq))
        assert c.index[0] == long_index[10] and len(c) == 40


def test_empty_and_plain_frames():
    groups = [(n, np.asarray(v)[:0], s) for n, v, s in _groups()]
    assert len(su.dataframe_from_parquet_bytes(su.columns_into_parquet_bytes(groups))) == 0
    plain = pd.DataFrame({"a": [1.0, 2.0], "b": [3.0, 4.0]})
    assert su.dataframe_to_dict(plain) == plain.to_dict()
    pd.testing.assert_frame_equal(su.dataframe_from_dict(plain.to_dict()), plain)


CODEC_CASES = ("time_index", "no_index")


def codec_frame(case):
    """The anomaly frame of ``_groups()``, with a 10-minute time index or none."""
    if case == "time_index":
        index, freq = pd.date_range("2020-03-01", periods=40, freq="10min", tz="UTC"), pd.Timedelta("10min")
    else:
        index, freq = None, None
    return mu.assemble_frame(_groups(), index, freq)


def frame_record(df):
    """A frame as plain JSON data: columns, index, dtypes and every value by column (JSON floats round-trip exactly)."""
    col = lambda c: list(c) if isinstance(c, tuple) else c
    cell = lambda v: v if v is None or isinstance(v, (bool, int, float)) else str(v)
    return {"columns": [col(c) for c in df.columns], "column_type": type(df.columns).__name__,
            "column_names": list(df.columns.names), "index": [str(v) for v in df.index],
            "index_type": type(df.index).__name__, "index_dtype": str(df.index.dtype), "index_name": df.index.name,
            "index_freq": getattr(df.index, "freqstr", None), "dtypes": [str(t) for t in df.dtypes],
            "values": [[cell(v) for v in df.iloc[:, j].tolist()] for j in range(df.shape[1])]}


def _read_parquet_as_gordo_does(raw):
    import pyarrow.parquet as pq
    return pq.read_table(io.BytesIO(raw)).to_pandas()


def test_codecs_match_the_reference_functions():
    """Against the original gordo's own codecs, recorded by tests/golden/make_server_codec_golden.py."""
    with open(os.path.join(ROOT, "tests", "golden", "server_codec_golden.json")) as f:
        golden = json.load(f)
    assert sorted(golden) == sorted(CODEC_CASES)
    for case in CODEC_CASES:
        _check_codecs(case, golden[case])


def _check_codecs(case, want):
    import pyarrow.parquet as pq
    df = codec_frame(case)
    index, freq = (df.index, pd.Timedelta("10min")) if case == "time_index" else (None, None)
    groups = _groups()
    # gordo's JSON body of the frame vs ours on the frame and on the raw column groups
    d = su.dataframe_to_dict(df)
    assert d == su.columns_to_dict(groups, index, freq), case
    assert json.loads(json.dumps(d, default=str)) == want["to_dict"], case
    # gordo's parquet bytes vs ours: the same Arrow table (schema, pandas metadata, data) ...
    ref_raw = base64.b64decode(want["parquet_base64"])
    ref_table = pq.read_table(io.BytesIO(ref_raw))
    for raw in (su.dataframe_into_parquet_bytes(df), su.columns_into_parquet_bytes(groups, index, freq)):
        table = pq.read_table(io.BytesIO(raw))
        assert table.equals(ref_table) and table.schema.metadata == ref_table.schema.metadata, case
        # ... which gordo's reader turns into the frame it read from its own bytes
        assert frame_record(_read_parquet_as_gordo_does(raw)) == want["from_parquet"], case
    # our reader on gordo's bytes, and our dict reader on gordo's JSON body, give the frames gordo's readers gave
    assert frame_record(su.dataframe_from_parquet_bytes(ref_raw)) == want["from_parquet"], case
    assert frame_record(su.dataframe_from_dict(want["to_dict"])) == want["from_dict"], case
