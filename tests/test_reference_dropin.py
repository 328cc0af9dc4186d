"""The drop-in boundary: `integration.register_with_reference` inside a clearml-serving dispatcher (CPU).

`integration.register_with_reference(name)` adds the engine to clearml-serving's registry
(clearml_serving/serving/preprocess_service.py:230-243); its ModelRequestProcessor.process_request
(model_request_processor.py:253-304) then builds the engine lazily from its ModelEndpoint (:287-291) and runs its 3-stage
pipeline (:1309-1369) over it.  clearml-serving is not a dependency of this project, so the test installs this package's
ports of that registry and dispatcher under clearml-serving's module names, and requires the replies to equal, value and
JSON form, those the reference's OWN dispatcher returned for the same requests (tests/golden/reference_dropin.json,
written by oracle/gen_golden.py through `serve` below).  Only the native layer is faked (host-side model / stream
executing the packed blob with the kernel's rules), so everything above the C ABI -- the mixin inside the registry's
class hierarchy, marshalling, batcher, futures -- is the real code."""
import asyncio
import json
import os
import sys
import types

import numpy as np
import pytest

from oracle import oracle as orc
from tests import blob_interp
from tests.fakes import FakeStream

ENGINE_NAMES = ["b200", "xgboost"]      # "xgboost": shadow the built-in engine name


class _BlobModel(object):
    """native.Model stand-in: executes the packed forest blob on the host (tests/blob_interp.py)"""

    def __init__(self, kind, blob, device=0):
        d = blob_interp.decode(blob)
        self.kind, self.blob, self.device = kind, blob, device
        self.n_inputs, self.n_outputs = 1, 1
        self.in_dtypes = [np.dtype(np.float32)]
        self.out_dtypes = [np.dtype(np.float64 if d["acc_mode"] == 1 else np.float32)]
        self.in_row_elems, self.out_row_elems = [d["n_features"]], [1]
        self.fn = lambda x: blob_interp.predict(blob, x)

        class _I(object):
            kind = 1
        self.info = _I()
        self.freed = False

    def free(self):
        self.freed = True


def install_fake_native(mp):
    """mp: a pytest MonkeyPatch.  Returns the list of models the engine creates."""
    from clearml_serving_b200 import native, scheduler
    made = []

    def model(kind, blob, device=0):
        m = _BlobModel(kind, blob, device)
        made.append(m)
        return m
    mp.setattr(native, "Model", model)
    mp.setattr(scheduler.native, "Stream",
               lambda m, max_rows, max_row_elems=0, n_slots=4: FakeStream(m, max_rows, n_slots=n_slots))
    return made


def reference_dispatcher(ref):
    """the reference's own registry and dispatcher (oracle/ref_harness.py)"""
    import clearml   # the stub package (oracle/refstubs): Model(model_id).get_local_copy() -> a local path
    from oracle import ref_harness as rh
    return types.SimpleNamespace(
        base=ref.ps.BasePreprocessRequest, endpoint=ref.endpoints.ModelEndpoint, model_paths=clearml.Model._paths,
        processor=lambda eps: rh.make_processor(ref, eps), not_found=ref.mrp.EndpointNotFoundException)


def port_dispatcher(mp):
    """this package's registry and dispatcher, importable under clearml-serving's module names for this test only"""
    from clearml_serving_b200 import model_request_processor as mrp
    from clearml_serving_b200 import preprocess_service as ps
    from clearml_serving_b200.endpoints import ModelEndpoint
    base = ps.BasePreprocessRequest
    mp.setattr(base, "_engines", dict(base._engines))
    mp.setattr(base, "_engine_modules", set(base._engine_modules))
    paths = {}
    mp.setattr(base, "_model_resolver", paths.get)
    for name in ("clearml_serving", "clearml_serving.serving"):
        mp.setitem(sys.modules, name, types.ModuleType(name))
    mp.setitem(sys.modules, "clearml_serving.serving.preprocess_service", ps)

    def processor(eps):
        p = mrp.ModelRequestProcessor()
        for ep in eps.values():
            p.add_endpoint(ep)
        return p
    return types.SimpleNamespace(base=base, endpoint=ModelEndpoint, model_paths=paths, processor=processor,
                                 not_found=mrp.EndpointNotFoundException)


def serve(d, engine_name, tmp_dir, made):
    """Registers the b200 engine as `engine_name` in dispatcher `d`, serves one raw request and 40 concurrent ones
    through it, checks them against the oracle, and returns the replies as JSON-able data."""
    import clearml_serving_b200.integration as b2s
    cls = b2s.register_with_reference(engine_name)
    assert d.base.get_engine_cls(engine_name) is cls
    assert issubclass(cls, d.base) and cls.is_process_async

    forest = orc.synth_xgb_forest(n_trees=31, depth=5, n_features=8, seed=12, ragged=True)
    path = os.path.join(tmp_dir, "model.json")
    with open(path, "w") as f:
        json.dump(orc.xgb_json_from_forest(forest, base_score=0.5), f)
    d.model_paths["model-123"] = path

    # user code exactly as clearml-serving loads it: a Preprocess class from a task artifact (here injected after the
    # constructor ran, as oracle/ref_harness.make_engine does for the reference's own engines)
    class Pre(object):
        def preprocess(self, body, state, collect_custom_statistics_fn=None):
            return np.array([[body["x{}".format(i)] for i in range(8)]], dtype=np.float32)

        def postprocess(self, data, state, collect_custom_statistics_fn=None):
            return dict(y=data.tolist())
    ep = d.endpoint(engine_type=engine_name, serving_url="trees", model_id="model-123",
                    auxiliary_cfg={"max_batch_size": 16, "dynamic_batching.max_queue_delay_microseconds": 2000})
    proc = d.processor({"trees": ep})                        # NO engine injected: process_request must build it
    rng = np.random.default_rng(0)
    X = rng.standard_normal((40, 8)).astype(np.float32)
    want = orc.forest_predict_xgb(forest, X, 0.5)

    async def run():
        first = await proc.process_request(base_url="trees", version=None,
                                           request_body=X[0:1].tolist(), serve_type="process")   # no user code yet: raw rows in
        eng = proc._engine_processor_lookup["trees"]
        assert type(eng) is cls and len(made) == 1
        eng._preprocess = Pre()
        replies = await asyncio.gather(*[
            proc.process_request(base_url="trees", version=None, serve_type="process",
                                 request_body={"x{}".format(j): float(X[i, j]) for j in range(8)}) for i in range(40)])
        return first, replies, eng
    first, replies, eng = asyncio.run(run())
    assert np.float32(np.asarray(first).ravel()[0]) == want[0]
    got = np.array([r["y"][0] for r in replies], dtype=np.float32)
    assert np.array_equal(got, want)                                        # bit-exact through the dispatcher's pipeline
    st = eng.engine_stats()
    assert st["requests"] == 41 and st["batches"] < 41                      # the 40 concurrent requests were batched
    # unknown endpoint: the dispatcher's own exception type (-> 404 in its REST layer)
    with pytest.raises(d.not_found):
        asyncio.run(proc.process_request(base_url="nope", version=None, request_body={}, serve_type="process"))
    # engines are dropped on reconfiguration (model_request_processor.py:1026-1028): unload releases the native objects
    proc._engine_processor_lookup.clear()
    eng.unload()
    assert made[0].freed
    d.model_paths.pop("model-123", None)
    return dict(first=dict(type=type(first).__name__, dtype=str(np.asarray(first).dtype), value=np.asarray(first).tolist()),
                replies=replies, not_found=d.not_found.__name__)


@pytest.mark.parametrize("engine_name", ENGINE_NAMES)
def test_registered_b200_engine_replies_like_the_reference_dispatcher(tmp_path, monkeypatch, golden_dir, engine_name):
    made = install_fake_native(monkeypatch)
    got = serve(port_dispatcher(monkeypatch), engine_name, str(tmp_path), made)
    with open(os.path.join(golden_dir, "reference_dropin.json")) as f:
        want = json.load(f)[engine_name]
    assert got == want
