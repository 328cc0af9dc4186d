"""Generate tests/golden/* by running the REFERENCE's own code (from /root/reference, under the
stubs in oracle/ref_harness.py) on seeded synthetic inputs.

Run in the build container only (needs /root/reference):   python oracle/gen_golden.py
The outputs are committed; the GPU box and the test-suite only read the fixtures.

Fixtures
  lr_iris.npz          BASELINE.json configs[0]: LogisticRegression on iris through the reference's
                       ModelRequestProcessor.process_request -> SKLearnPreprocessRequest.process
                       (model_request_processor.py:253-304,1309-1369; preprocess_service.py:459-464)
  sk_gbr.npz sk_rf.npz tree ensembles through the same reference engine class (fp64 outputs)
  sk_gbr_cfg2.npz      the same engine class at the BASELINE.json configs[1] SHAPE: GradientBoostingRegressor with
                       1000 stages x depth 6 on 32 features (the headline workload's tree count / depth / width,
                       produced by the reference itself), incl. rows on thresholds +-1 ulp
  triton_marshal.json  the reference's TritonPreprocessRequest.process (preprocess_service.py:313-446)
                       run unmodified against an in-process fake tritonserver: wire-level dtypes /
                       shapes and decoded outputs for the marshalling edge cases
  rest_contract.json   the reference FastAPI app (main.py) under starlette TestClient:
                       request -> (status, body) pairs incl. 404/422 detail strings
  reference_dropin.json the b200 engine registered into the reference's registry by integration.register_with_reference
                       and served by the reference's ModelRequestProcessor.process_request: the replies, per engine name
"""
import asyncio
import gzip
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh  # noqa: E402
from oracle import oracle as orc  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


class IrisPreprocess(object):
    """examples/sklearn/preprocess.py:12-19 widened from x0,x1 to x0..x3 (BASELINE configs[0])."""

    def preprocess(self, body, state, collect_custom_statistics_fn=None):
        return [[body.get("x0", None), body.get("x1", None), body.get("x2", None), body.get("x3", None)], ]

    def postprocess(self, data, state, collect_custom_statistics_fn=None):
        return dict(y=data.tolist() if isinstance(data, np.ndarray) else data)


class RaisingPreprocess(object):
    def preprocess(self, body, state, collect_custom_statistics_fn=None):
        if "boom" in body:
            raise ValueError("bad request field")
        if "boom_rt" in body:
            raise RuntimeError("runtime failure")
        return [[body.get("x0", None), body.get("x1", None), body.get("x2", None), body.get("x3", None)], ]

    def postprocess(self, data, state, collect_custom_statistics_fn=None):
        return dict(y=data.tolist())


def gen_lr(ref):
    from sklearn.datasets import load_iris
    from sklearn.linear_model import LogisticRegression
    Xtr, ytr = load_iris(return_X_y=True)
    model = LogisticRegression(max_iter=1000).fit(Xtr, ytr)
    rng = np.random.default_rng(0)
    X = rng.uniform(0, 8, (256, 4))
    ep = ref.endpoints.ModelEndpoint(engine_type="sklearn", serving_url="iris")
    eng = rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep, model=model, preprocess=IrisPreprocess())
    proc = rh.make_processor(ref, {"iris": ep}, {"iris": eng})

    async def run():
        out = []
        for row in X:
            body = {"x%d" % i: float(v) for i, v in enumerate(row)}
            r = await proc.process_request(base_url="iris", version=None, request_body=body, serve_type="process")
            out.append(r["y"][0])
        return out

    y = np.asarray(asyncio.run(run()), dtype=np.int64)
    scores = model.decision_function(X)
    # binary variant (n_out == 1 path: score > 0)
    yb = (ytr == 2).astype(np.int64)
    model_b = LogisticRegression(max_iter=1000).fit(Xtr, yb)
    eng_b = rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep, model=model_b)
    y_b = np.asarray(eng_b.process(X, {}, None), dtype=np.int64)
    np.savez(os.path.join(GOLD, "lr_iris.npz"),
             coef=model.coef_, intercept=model.intercept_, classes=model.classes_,
             X=X, y=y, scores=scores,
             coef_b=model_b.coef_, intercept_b=model_b.intercept_, classes_b=model_b.classes_,
             y_b=y_b, scores_b=model_b.decision_function(X))
    print("lr_iris: labels", np.bincount(y), "binary", np.bincount(y_b))
    return model


def _tree_inputs(forest, n_features, rng, n=384):
    X = rng.standard_normal((n, n_features)).astype(np.float32) * 1.5
    # rows sitting exactly ON thresholds (and one ulp either side) to pin the <= boundary
    internal = np.nonzero(forest["left"] >= 0)[0]
    pick = rng.choice(internal, size=min(96, len(internal)), replace=False)
    for j, g in enumerate(pick):
        f = int(forest["feat"][g])
        t32 = np.float32(forest["thr"][g])
        row = 3 * j
        if row + 2 >= n:
            break
        X[row, f] = t32
        X[row + 1, f] = np.nextafter(t32, np.float32(np.inf))
        X[row + 2, f] = np.nextafter(t32, np.float32(-np.inf))
    return X


def gen_trees(ref):
    from sklearn.ensemble import GradientBoostingRegressor, RandomForestRegressor
    rng = np.random.default_rng(7)
    F = 16
    Xtr = rng.standard_normal((600, F))
    ytr = Xtr[:, 0] * 2 + np.sin(Xtr[:, 1] * 3) + Xtr[:, 2] * Xtr[:, 3] + 0.1 * rng.standard_normal(600)
    ep = ref.endpoints.ModelEndpoint(engine_type="sklearn", serving_url="trees")

    gbr = GradientBoostingRegressor(n_estimators=40, max_depth=5, learning_rate=0.1, random_state=0).fit(Xtr, ytr)
    forest = orc.forest_from_sklearn([e[0] for e in gbr.estimators_], F)
    X = _tree_inputs(forest, F, rng)
    eng = rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep, model=gbr)
    y = np.asarray(eng.process(X, {}, None), dtype=np.float64)
    init = float(gbr.init_.constant_.ravel()[0])
    np.savez(os.path.join(GOLD, "sk_gbr.npz"), X=X, y=y, init=init, scale=float(gbr.learning_rate),
             divisor=1.0, **forest)
    chk = orc.forest_predict_f64(forest, X, init, float(gbr.learning_rate), 1.0)
    print("sk_gbr: oracle bit-identical to reference:", bool(np.array_equal(chk, y)),
          "max|d|", float(np.abs(chk - y).max()))

    rf = RandomForestRegressor(n_estimators=25, max_depth=7, random_state=0, n_jobs=1).fit(Xtr, ytr)
    forest = orc.forest_from_sklearn(rf.estimators_, F)
    X = _tree_inputs(forest, F, rng)
    eng = rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep, model=rf)
    y = np.asarray(eng.process(X, {}, None), dtype=np.float64)
    np.savez(os.path.join(GOLD, "sk_rf.npz"), X=X, y=y, init=0.0, scale=1.0,
             divisor=float(len(rf.estimators_)), **forest)
    chk = orc.forest_predict_f64(forest, X, 0.0, 1.0, float(len(rf.estimators_)))
    print("sk_rf: oracle bit-identical to reference:", bool(np.array_equal(chk, y)),
          "max|d|", float(np.abs(chk - y).max()))


def gen_trees_cfg2(ref):
    """BASELINE.json configs[1] shape through the REAL reference engine class
    (SKLearnPreprocessRequest.process, preprocess_service.py:459-464): 1000 trees x depth 6 x 32 features."""
    from sklearn.ensemble import GradientBoostingRegressor
    rng = np.random.default_rng(11)
    F = 32
    Xtr = rng.standard_normal((3000, F))
    ytr = (Xtr[:, 0] * 2 + np.sin(Xtr[:, 1] * 3) + Xtr[:, 2] * Xtr[:, 3] + np.abs(Xtr[:, 4:12]).sum(1) * 0.3
           + 0.5 * rng.standard_normal(3000))
    gbr = GradientBoostingRegressor(n_estimators=1000, max_depth=6, learning_rate=0.05, subsample=0.5,
                                    random_state=0).fit(Xtr, ytr)
    forest = orc.forest_from_sklearn([e[0] for e in gbr.estimators_], F)
    X = _tree_inputs(forest, F, rng, n=320)
    ep = ref.endpoints.ModelEndpoint(engine_type="sklearn", serving_url="trees_cfg2")
    eng = rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep, model=gbr)
    y = np.asarray(eng.process(X, {}, None), dtype=np.float64)
    # one request at a time as the serving path sees them (batch = 1): must be the same bits
    y1 = np.concatenate([np.asarray(eng.process(X[i:i + 1], {}, None), dtype=np.float64) for i in range(64)])
    assert np.array_equal(y1, y[:64])
    init = float(gbr.init_.constant_.ravel()[0])
    compact = dict(forest)
    compact["feat"] = forest["feat"].astype(np.int16)
    # internal-node values are never read (only leaves carry an output): stored as 0, which keeps the file under 1 MB
    compact["value"] = np.where(forest["left"] < 0, forest["value"], 0.0)
    np.savez_compressed(os.path.join(GOLD, "sk_gbr_cfg2.npz"), X=X, y=y, init=init, scale=float(gbr.learning_rate),
                        divisor=1.0, **compact)
    chk = orc.forest_predict_f64(forest, X, init, float(gbr.learning_rate), 1.0)
    print("sk_gbr_cfg2: trees", len(forest["tree_offset"]) - 1, "nodes", len(forest["left"]),
          "oracle bit-identical to reference:", bool(np.array_equal(chk, y)), "max|d|", float(np.abs(chk - y).max()))


def gen_triton_marshal(ref):
    """Each case: endpoint io spec + python `data` -> what went on the wire + what came back."""
    cases = []

    def run_case(name, io, data, model_fn):
        ep = ref.endpoints.ModelEndpoint(engine_type="triton", serving_url=name, **io)
        eng = rh.make_engine(ref, ref.ps.TritonPreprocessRequest, ep)
        rh.FakeTritonServer.models[name] = model_fn
        rec = dict(name=name, io=io, data=data)
        try:
            out = asyncio.run(eng.process(data, {}, None))
            req = rh.FakeTritonServer.last_request
            rec["wire_inputs"] = [dict(name=t.name, datatype=t.datatype, shape=list(t.shape)) for t in req.inputs]
            rec["model_name"] = req.model_name
            outs = out if isinstance(out, list) else [out]
            rec["returns_list"] = isinstance(out, list)
            rec["outputs"] = [dict(dtype=str(o.dtype), shape=list(o.shape), values=o.ravel().tolist()) for o in outs]
        except Exception as ex:  # noqa
            rec["raises"] = type(ex).__name__
            rec["message"] = str(ex)
        cases.append(rec)

    run_case("single_fp32",
             dict(input_size=[[1, 4]], input_type=["float32"], input_name=["INPUT__0"],
                  output_size=[[-1, 2]], output_type=["float32"], output_name=["OUTPUT__0"]),
             [[1, 2.5, 3, 4]], lambda ins: [ins[0][:, :2] * 2])
    run_case("f64_data_cast_to_f32",
             dict(input_size=[[3]], input_type=["float32"], input_name=["x"],
                  output_size=[[3]], output_type=["float32"], output_name=["y"]),
             [0.1, 0.2, 0.3], lambda ins: [ins[0] + 1])
    run_case("hf_three_int32",
             dict(input_size=[[-1], [-1], [-1]], input_type=["int32", "int32", "int32"],
                  input_name=["input_ids", "token_type_ids", "attention_mask"],
                  output_size=[[2]], output_type=["float32"], output_name=["output"]),
             [[[101, 2023, 2003, 102]], [[0, 0, 0, 0]], [[1, 1, 1, 1]]],
             lambda ins: [np.stack([ins[0].sum(1), ins[2].sum(1)], 1).astype(np.float32)])
    run_case("uint8_image",
             dict(input_size=[[1, 2, 2]], input_type=["uint8"], input_name=["img"],
                  output_size=[[-1, 4]], output_type=["float32"], output_name=["p"]),
             [[[1, 2], [3, 255]]], lambda ins: [ins[0].reshape(1, 4).astype(np.float32) / 255])
    run_case("two_outputs_type_clamp",
             dict(input_size=[[2]], input_type=["float32"], input_name=["x"],
                  output_size=[[2], [2]], output_type=["float32"], output_name=["a", "b"]),
             [1.0, 2.0], lambda ins: [ins[0] * 2, ins[0] * 3])
    run_case("int64_tokens",
             dict(input_size=[[-1]], input_type=["int64"], input_name=["ids"],
                  output_size=[[1]], output_type=["int64"], output_name=["n"]),
             [[5, 6, 7]], lambda ins: [np.array([ins[0].sum()], dtype=np.int64)])
    # model name on the wire is "{serving_url}_{version}" (preprocess_service.py:375-377)
    rh.FakeTritonServer.models["versioned_name_3"] = lambda ins: [ins[0] - 1]
    run_case("versioned_name",
             dict(version="3", input_size=[[2]], input_type=["float64"], input_name=["x"],
                  output_size=[[2]], output_type=["float64"], output_name=["y"]),
             [1.5, 2.5], lambda ins: [ins[0] - 1])
    run_case("fp16_unsupported",
             dict(input_size=[[2]], input_type=["float16"], input_name=["x"],
                  output_size=[[2]], output_type=["float32"], output_name=["y"]),
             [1.0, 2.0], lambda ins: [ins[0]])
    with open(os.path.join(GOLD, "triton_marshal.json"), "w") as f:
        json.dump(cases, f, indent=1)
    for c in cases:
        print("triton_marshal:", c["name"], c.get("raises") or [o["dtype"] + str(o["shape"]) for o in c["outputs"]])


def gen_rest(ref, lr_model):
    from starlette.testclient import TestClient
    ep = ref.endpoints.ModelEndpoint(engine_type="sklearn", serving_url="iris")
    ep_v = ref.endpoints.ModelEndpoint(engine_type="sklearn", serving_url="iris/2", version="2")
    ep_bad = ref.endpoints.ModelEndpoint(engine_type="sklearn", serving_url="bad")
    engines = {
        "iris": rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep, model=lr_model, preprocess=IrisPreprocess()),
        "iris/2": rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep_v, model=lr_model, preprocess=IrisPreprocess()),
        "bad": rh.make_engine(ref, ref.ps.SKLearnPreprocessRequest, ep_bad, model=lr_model, preprocess=RaisingPreprocess()),
    }
    ref.main.processor = rh.make_processor(ref, {"iris": ep, "iris/2": ep_v, "bad": ep_bad}, engines)
    client = TestClient(ref.main.app, raise_server_exceptions=False)
    body = {"x0": 5.1, "x1": 3.5, "x2": 1.4, "x3": 0.2}
    body2 = {"x0": 6.7, "x1": 3.0, "x2": 5.2, "x3": 2.3}
    reqs = [
        dict(name="ok", path="/serve/iris", json=body),
        dict(name="ok_trailing_slash", path="/serve/iris/", json=body2),
        dict(name="ok_version", path="/serve/iris/2", json=body2),
        dict(name="unknown_endpoint", path="/serve/nope", json=body),
        dict(name="unknown_version", path="/serve/iris/9", json=body),
        dict(name="preprocess_value_error", path="/serve/bad", json={"boom": 1}),
        dict(name="preprocess_runtime_error", path="/serve/bad", json={"boom_rt": 1}),
        dict(name="gzip_body", path="/serve/iris", gzip_json=body),
        dict(name="get_not_allowed", path="/serve/iris", method="GET"),
    ]
    out = []
    for r in reqs:
        if r.get("method") == "GET":
            resp = client.get(r["path"])
        elif "gzip_json" in r:
            resp = client.post(r["path"], content=gzip.compress(json.dumps(r["gzip_json"]).encode()),
                               headers={"Content-Encoding": "gzip", "Content-Type": "application/json"})
        else:
            resp = client.post(r["path"], json=r["json"])
        try:
            payload = resp.json()
        except Exception:  # noqa
            payload = resp.text
        rec = dict(r)
        rec.update(status=resp.status_code, response=payload)
        out.append(rec)
        print("rest:", r["name"], resp.status_code, str(payload)[:110])
    with open(os.path.join(GOLD, "rest_contract.json"), "w") as f:
        json.dump(out, f, indent=1)


def gen_dropin(ref):
    """tests/test_reference_dropin.py's scenario through the reference's own dispatcher, per engine name"""
    import tempfile
    import pytest
    from tests import test_reference_dropin as t
    out = {}
    for name in t.ENGINE_NAMES:
        with pytest.MonkeyPatch.context() as mp, tempfile.TemporaryDirectory() as tmp:
            made = t.install_fake_native(mp)
            out[name] = t.serve(t.reference_dispatcher(ref), name, tmp, made)
    with open(os.path.join(GOLD, "reference_dropin.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("reference_dropin:", {k: len(v["replies"]) for k, v in out.items()})


def main():
    os.makedirs(GOLD, exist_ok=True)
    ref = rh.load_reference()
    lr = gen_lr(ref)
    gen_trees(ref)
    gen_trees_cfg2(ref)
    gen_triton_marshal(ref)
    gen_rest(ref, lr)
    gen_dropin(ref)


if __name__ == "__main__":
    main()
