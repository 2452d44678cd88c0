"""
Record the original gordo's response codecs (gordo/server/utils.py:47-160) on the frames of
tests/test_server_utils_cpu.py -> server_codec_golden.json.

    python tests/golden/make_server_codec_golden.py <gordo source checkout>

gordo/server/utils.py is executed unmodified from the checkout with flask / werkzeug / gordo-core stubbed (none of
them takes part in the codecs).  Per case (time index or none): what ``dataframe_to_dict`` returns (after a JSON
round trip), the bytes ``dataframe_into_parquet_bytes`` writes, the frame ``dataframe_from_parquet_bytes`` reads back
from them, and the frame ``dataframe_from_dict`` rebuilds from the JSON body.
"""
import base64
import importlib.util
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def _stub(name, **kw):
    m = types.ModuleType(name)
    m.__dict__.update(kw)
    sys.modules[name] = m
    return m


def load_reference_utils(reference):
    path = os.path.join(reference, "gordo", "server", "utils.py")
    if not os.path.isfile(path):
        raise SystemExit(f"{reference} holds no gordo/server/utils.py")
    _stub("flask", request=None, g=None, jsonify=None, make_response=None, Response=object)
    _stub("werkzeug")
    _stub("werkzeug.exceptions", NotFound=Exception, UnprocessableEntity=Exception, InternalServerError=Exception)
    g = _stub("gordo")
    g.__path__ = []
    g.serializer = None
    _stub("gordo.serializer")
    srv = _stub("gordo.server")
    srv.__path__ = [os.path.dirname(path)]
    _stub("gordo.server.properties", get_tags=None, get_target_tags=None)
    spec = importlib.util.spec_from_file_location("gordo.server.utils", path)
    ref = importlib.util.module_from_spec(spec)
    sys.modules["gordo.server.utils"] = ref
    spec.loader.exec_module(ref)
    return ref


def main(reference):
    from tests import test_server_utils_cpu as t
    ref = load_reference_utils(os.path.abspath(reference))
    out = {}
    for name in t.CODEC_CASES:
        df = t.codec_frame(name)
        body = json.loads(json.dumps(ref.dataframe_to_dict(df), default=str))
        raw = ref.dataframe_into_parquet_bytes(df)
        out[name] = {"to_dict": body, "parquet_base64": base64.b64encode(raw).decode("ascii"),
                     "from_parquet": t.frame_record(ref.dataframe_from_parquet_bytes(raw)),
                     "from_dict": t.frame_record(ref.dataframe_from_dict(body))}
    path = os.path.join(HERE, "server_codec_golden.json")
    with open(path, "w") as f:
        json.dump(out, f)              # key order is part of the JSON body: not sorted
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
