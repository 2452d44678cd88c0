"""
Record how the original gordo's serializer and ModelBuilder treat the gordo_b200 classes -> seam_golden.json.

    python tests/golden/make_seam_golden.py <gordo source checkout>

The reference modules are executed unmodified from the checkout through tests/reference_loader.py (TensorFlow /
Keras / gordo-core / xarray stubbed; none of them takes part in what is recorded).  Recorded:
  serializer: for each model definition, the object graph gordo's ``from_definition`` builds (class paths and
              constructor parameters), what gordo's ``into_definition`` writes for it, and what reading that back gives;
  builder:    the model definition ``ModelBuilder._build`` resolves after FleetModelBuilder redirected it, the estimator
              it built from it, the keyword arguments of its ``model.cross_validate(...)`` call, the CV split metadata,
              and the parameter names of ``ModelBuilder.__init__`` / ``ModelBuilder.build``.
tests/test_seam_reference_cpu.py checks gordo_b200 against this file.
"""
import inspect
import json
import os
import sys
import traceback

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def _builder_case(ref, rl, seam, evaluation):
    import numpy as np
    import gordo_b200.builder as b
    from gordo_b200.machine.model.anomaly import diff
    X = seam.builder_frame()
    rl.StubDataset.registry["d0"] = (X, X)
    machine = rl.StubMachine("m0", seam.BUILDER_MODEL, {"key": "d0"}, evaluation=evaluation)
    builder = b.FleetModelBuilder(machine)
    assert isinstance(builder, ref["build_model"].ModelBuilder)
    seen = {}
    original = diff.DiffBasedAnomalyDetector.cross_validate

    def recording(self, **kwargs):
        seen["model"] = seam.describe(self)
        seen["kwargs"] = sorted(kwargs)
        seen["return_estimator"] = kwargs.get("return_estimator")
        seen["cv"] = seam.describe(kwargs.get("cv"))
        seen["scoring"] = sorted(kwargs.get("scoring") or {})
        seen["X_is_the_dataset"] = bool(np.array_equal(np.asarray(kwargs["X"]), X.to_numpy()))
        raise RuntimeError("recorded")
    diff.DiffBasedAnomalyDetector.cross_validate = recording
    try:
        builder.build()
        raise SystemExit("the recording cross_validate was never called")
    except Exception as e:
        tb = traceback.format_exc()
        assert "recorded" in str(e) + tb and "_build" in tb, tb
    finally:
        diff.DiffBasedAnomalyDetector.cross_validate = original
    seen["resolved_model"] = builder.machine.model
    return seen


def main(reference):
    from tests import reference_loader as rl
    from tests import test_seam_reference_cpu as seam
    rl.REF = os.path.abspath(reference)
    if not rl.available():
        raise SystemExit(f"{reference} holds no gordo package")
    ref = rl.load()
    ser = ref["serializer"]
    out = {"serializer": {}, "builder": {}}
    for name, definition in seam.DEFINITIONS.items():
        model = ser.from_definition(definition)
        written = ser.into_definition(model)
        out["serializer"][name] = {"built": seam.describe(model), "into_definition": written,
                                   "read_back": seam.describe(ser.from_definition(written))}
    MB = ref["build_model"].ModelBuilder
    out["builder"]["signatures"] = {"__init__": list(inspect.signature(MB.__init__).parameters),
                                    "build": list(inspect.signature(MB.build).parameters)}
    out["builder"]["cases"] = {name: _builder_case(ref, rl, seam, dict(evaluation))
                               for name, evaluation in seam.BUILDER_EVALUATIONS.items()}
    from sklearn.model_selection import TimeSeriesSplit
    splits = MB.build_split_dict(seam.builder_frame(), TimeSeriesSplit(n_splits=3))
    out["builder"]["split_metadata"] = {k: str(v) for k, v in splits.items()}
    path = os.path.join(HERE, "seam_golden.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
