"""Generates tests/golden/hotpath_golden_{f32,f64}.npz by EXECUTING THE REFERENCE'S OWN SOURCE FILES
(read from a checkout of the original deep_recommenders project, never copied) under the numpy-backed
`tensorflow` stand-in in oracle/tf_shim.  Needs no GPU.  The .npz files are committed and the tests
read only them; rerun this by hand when the golden cases change.

    python tests/golden/make_golden.py <checkout of the original deep_recommenders project>

What executes from the reference:
  keras/models/ranking/fm.py        FM.call (:23-37), FactorizationMachine.call (:54-63)
  keras/models/ranking/deepfm.py    DeepFM.call (:36-47)
  keras/models/ranking/dcn.py       Cross.build / call (:35-88) full, low-rank, diag_scale, no-bias
  keras/models/retrieval/sbcnm.py   HardNegativeMining, RemoveAccidentalNegative,
                                    SamplingProbabilityCorrection, Retrieval.call default path
  estimator/models/feature_interaction/fm.py   fm (:10-26), FM.call (:41-56)
  estimator/models/feature_interaction/dnn.py  dnn (:9-31)
  estimator/models/ranking/deepfm.py           DeepFM.call (:30-43)
and, into tests/golden/retrieval_golden.npz (SURVEY 8f #3):
  keras/models/retrieval/factorized_top_k.py   _take_long_axis (:26-41), _exclude (:44-67), Streaming.call (:180-262),
                                               BruteForce.index / call (:277-334), TopK.query_with_exclusions (:113-131),
                                               FactorizedTopK.update_state / result (:487-522)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "deep_recommenders")):
    sys.exit("usage: python tests/golden/make_golden.py <checkout of the original deep_recommenders project>")
REFERENCE = os.path.abspath(sys.argv[1])
sys.path.insert(0, os.path.join(ROOT, "oracle", "tf_shim"))
sys.path.insert(0, REFERENCE)
sys.dont_write_bytecode = True

import tensorflow as tf  # noqa: E402  (the shim)

assert "tf_shim" in tf.__file__, "real TensorFlow found: use it directly instead of the shim"


def generate(dtype):
    tf.set_default_dtype(dtype)
    tf.random.set_seed(1234)
    tf._LINEAR.clear()
    del tf._DENSE_LAYERS[:]
    rng = np.random.RandomState(7)
    out = {}

    def rnd(*shape, scale=1.0):
        return (rng.standard_normal(shape) * scale).astype(dtype)

    # ---- keras FM layer ------------------------------------------------------------------------
    from deep_recommenders.keras.models.ranking import FM, DeepFM, FactorizationMachine
    for tag, (B, N, S, D) in {"fm_a": (10, 10, 5, 5), "fm_b": (64, 40, 26, 16)}.items():
        sparse = rng.randint(0, 2, size=(B, N)).astype(dtype)
        emb = rnd(B, S, D)
        layer = FM()
        y0 = layer(sparse, emb)                      # zero-init linear (test_fm.py:17-26 situation)
        layer._linear.kernel = rnd(N, 1, scale=0.3)
        layer._linear.bias = rnd(1, scale=0.3)
        y1 = layer(sparse, emb)
        ylin = layer(sparse)
        out.update({f"{tag}_sparse": sparse, f"{tag}_emb": emb, f"{tag}_kernel": layer._linear.kernel,
                    f"{tag}_bias": layer._linear.bias, f"{tag}_y_zero": np.asarray(y0), f"{tag}_y": np.asarray(y1),
                    f"{tag}_y_linear_only": np.asarray(ylin)})

    # ---- estimator fm() ----------------------------------------------------------------------------
    from deep_recommenders.estimator.models.feature_interaction import fm as est_fm, FM as EstFM, dnn as est_dnn
    for tag, shp in {"estfm_a": (10, 2, 3), "estfm_b": (32, 6, 16)}.items():
        x = rnd(*shp)
        out[f"{tag}_x"] = x
        out[f"{tag}_y"] = np.asarray(est_fm(tf.convert_to_tensor(x)))
    try:
        est_fm(tf.convert_to_tensor(rnd(4, 6)))
        raise AssertionError("rank check did not fire")
    except ValueError as e:
        out["estfm_rank_error"] = np.asarray(str(e))

    # ---- Cross ---------------------------------------------------------------------------------------
    from deep_recommenders.keras.models.ranking.dcn import Cross
    c = Cross(projection_dim=None, kernel_init="ones")
    out["cross_kat_y"] = np.asarray(c(np.asarray([[0.1, 0.2, 0.3]], dtype), np.asarray([[0.4, 0.5, 0.6]], dtype)))
    cases = {"cross_full": dict(), "cross_diag": dict(diag_scale=0.5), "cross_nobias": dict(use_bias=False),
             "cross_lowrank": dict(projection_dim=4), "cross_lowrank_diag": dict(projection_dim=3, diag_scale=0.25)}
    for tag, kw in cases.items():
        B, d = 16, 13
        x0, x = rnd(B, d), rnd(B, d)
        layer = Cross(**kw)
        layer(x0, x)                                  # build
        if kw.get("projection_dim") is None:
            layer._dense.kernel = rnd(d, d, scale=0.3)
            if layer._dense.bias is not None:
                layer._dense.bias = rnd(d, scale=0.3)
            out[f"{tag}_w"] = layer._dense.kernel
            if layer._dense.bias is not None:
                out[f"{tag}_b"] = layer._dense.bias
        else:
            r = kw["projection_dim"]
            layer._dense_u.kernel = rnd(d, r, scale=0.3)
            layer._dense_v.kernel = rnd(r, d, scale=0.3)
            layer._dense_v.bias = rnd(d, scale=0.3)
            out[f"{tag}_u"], out[f"{tag}_v"], out[f"{tag}_b"] = layer._dense_u.kernel, layer._dense_v.kernel, layer._dense_v.bias
        out[f"{tag}_x0"], out[f"{tag}_x"] = x0, x
        out[f"{tag}_y"] = np.asarray(layer(x0, x))
        out[f"{tag}_y_xnone"] = np.asarray(layer(x0))
        out[f"{tag}_config_keys"] = np.asarray(sorted(layer.get_config().keys()))
    for bad in (dict(projection_dim=7), dict(projection_dim=-1)):
        try:
            Cross(**bad)(rnd(2, 13))
            raise AssertionError("projection_dim check did not fire")
        except ValueError as e:
            out["cross_projection_error"] = np.asarray(str(e))
    try:
        Cross()(rnd(2, 13), rnd(2, 12))
        raise AssertionError("dim check did not fire")
    except ValueError as e:
        out["cross_dim_error"] = np.asarray(str(e))

    # ---- sbcnm ---------------------------------------------------------------------------------------
    from deep_recommenders.keras.models.retrieval import sbcnm
    r42 = np.random.RandomState(42)
    logits = r42.uniform(size=(2, 20)).astype(np.float32)
    labels = r42.permutation(np.eye(2, 20).T).T.astype(np.float32)
    out["hnm_logits"], out["hnm_labels"] = logits, labels
    for k in (3, 5, 10, 15, 30):
        ol, oy = sbcnm.HardNegativeMining(k)(logits, labels)
        out[f"hnm_k{k}_logits"], out[f"hnm_k{k}_labels"] = np.asarray(ol), np.asarray(oy)
    r42 = np.random.RandomState(42)
    logits = r42.uniform(size=(2, 4)).astype(np.float32)
    labels = r42.permutation(np.eye(2, 4).T).T.astype(np.float32)
    ident = r42.randint(0, 3, size=4)
    out["ran_logits"], out["ran_labels"], out["ran_ids"] = logits, labels, ident
    out["ran_out"] = np.asarray(sbcnm.RemoveAccidentalNegative()(logits, labels, ident))
    lg = rnd(12, 12)
    ids = rng.randint(0, 4, size=12)
    p = rng.uniform(0.05, 1.0, size=12).astype(dtype)
    out["ran2_logits"], out["ran2_ids"], out["spc_p"] = lg, ids, p
    out["ran2_out"] = np.asarray(sbcnm.RemoveAccidentalNegative()(lg, np.eye(12, dtype=dtype), ids))
    out["spc_out"] = np.asarray(sbcnm.SamplingProbabilityCorrection()(lg, p))
    for tag, (nq, D, tau, use_w) in {"ret_a": (8, 16, None, False), "ret_b": (33, 64, 0.5, True),
                                     "ret_c": (70, 32, 2.0, True)}.items():
        q, cc = rnd(nq, D, scale=0.5), rnd(nq, D, scale=0.5)
        w = rng.uniform(0.5, 2.0, size=nq).astype(dtype) if use_w else None
        loss = sbcnm.Retrieval(temperature=tau)(q, cc, sample_weight=w)
        out[f"{tag}_q"], out[f"{tag}_c"], out[f"{tag}_loss"] = q, cc, np.asarray(loss)
        out[f"{tag}_tau"] = np.asarray(-1.0 if tau is None else tau)
        if w is not None:
            out[f"{tag}_w"] = w

    # ---- estimator dnn() ---------------------------------------------------------------------------
    x = rnd(20, 12)
    n0 = len(tf._DENSE_LAYERS)
    y = est_dnn(tf.convert_to_tensor(x), [8, 4, 1])
    ls = tf._DENSE_LAYERS[n0:]
    out["dnn_x"], out["dnn_y"] = x, np.asarray(y)
    for i, l in enumerate(ls):
        out[f"dnn_w{i}"], out[f"dnn_b{i}"] = l.kernel, l.bias
    out["dnn_acts"] = np.asarray([str(getattr(l.activation, "__name__", l.activation)) for l in ls])

    # ---- keras models on feature columns -------------------------------------------------------
    def build_columns():
        cols = [tf.feature_column.categorical_column_with_identity("user_id", 50),
                tf.feature_column.categorical_column_with_identity("movie_id", 40),
                tf.feature_column.categorical_column_with_vocabulary_list("gender", ["F", "M"]),
                tf.feature_column.categorical_column_with_identity("age", 7)]
        return ([tf.feature_column.indicator_column(c) for c in cols],
                [tf.feature_column.embedding_column(c, dimension=16) for c in cols])

    B = 48
    feats = {   # insertion order deliberately NOT sorted: the keras models iterate inputs.items()
        "user_id": rng.randint(-1, 51, size=(B, 1)),      # includes -1 and 50 (out of range)
        "age": rng.randint(0, 7, size=(B, 1)),
        "movie_id": rng.randint(0, 40, size=(B, 1)),
        "gender": np.asarray([["F"], ["M"], ["X"]] * (B // 3), dtype=object),   # "X" is OOV
    }
    out["cols_order_inputs"] = np.asarray(list(feats.keys()))
    for k, v in feats.items():
        out[f"feat_{k}"] = v.astype(str) if v.dtype == object else v

    ind, emb = build_columns()
    model = FactorizationMachine(ind, emb)
    model(feats)
    nsp = sum(c.categorical_column.num_buckets for c in ind)
    model._kernel._linear.kernel = rnd(nsp, 1, scale=0.3)
    model._kernel._linear.bias = rnd(1, scale=0.3)
    out["kfm_prob"] = np.asarray(model(feats))
    out["kfm_lin_kernel"], out["kfm_lin_bias"] = model._kernel._linear.kernel, model._kernel._linear.bias
    out["kfm_sparse_order"] = np.asarray([c.name for c in model._sparse_features_layer.columns])
    for c in emb:
        out[f"kfm_table_{c.categorical_column.key}"] = c.table

    ind, emb = build_columns()
    model = DeepFM(ind, emb, dnn_units_size=[32, 8])
    model(feats)
    model._fm._linear.kernel = rnd(nsp, 1, scale=0.3)
    model._fm._linear.bias = rnd(1, scale=0.3)
    out["kdfm_prob"] = np.asarray(model(feats))
    out["kdfm_lin_kernel"], out["kdfm_lin_bias"] = model._fm._linear.kernel, model._fm._linear.bias
    for c in emb:
        out[f"kdfm_table_{c.categorical_column.key}"] = c.table
    for i, l in enumerate(model._dnn.layers):
        out[f"kdfm_w{i}"], out[f"kdfm_b{i}"] = l.kernel, l.bias

    # ---- estimator FM / DeepFM -------------------------------------------------------------------
    ind, emb = build_columns()
    efm = EstFM(ind, emb)
    efm(feats)
    ws, b = tf.linear_model_weights(ind)
    for k in ws:
        ws[k][:] = rnd(*ws[k].shape, scale=0.3)
    b[:] = rnd(1, scale=0.3)
    out["efm_logit"] = np.asarray(efm(feats))
    out["efm_emb_order"] = np.asarray([c.name for c in emb])
    for c in emb:
        out[f"efm_table_{c.categorical_column.key}"] = c.table
    for k in ws:
        out[f"efm_lin_{k}"] = ws[k]
    out["efm_lin_bias"] = b.copy()

    from deep_recommenders.estimator.models.ranking.deepfm import DeepFM as EstDeepFM
    n0 = len(tf._DENSE_LAYERS)
    edfm = EstDeepFM(ind, emb, [16, 4], dnn_activation=tf.nn.relu)
    out["edfm_prob"] = np.asarray(edfm(feats))
    for i, l in enumerate(tf._DENSE_LAYERS[n0:]):
        out[f"edfm_w{i}"], out[f"edfm_b{i}"] = l.kernel, l.bias
    return out


def generate_retrieval():
    """Executes the reference's factorized_top_k.py (float32, its own dtype) on seeded inputs."""
    tf.set_default_dtype(np.float32)
    import importlib
    ftk = importlib.import_module("deep_recommenders.keras.models.retrieval.factorized_top_k")
    out = {}
    rng = np.random.RandomState(11)
    # _take_long_axis / _exclude: the reference's own KATs (tests/keras/test_factorized_top_k.py:17-34) and random cases
    arr = np.asarray([[0.1, 0.2, 0.3], [0.4, 0.5, 0.6]], np.float32)
    out["tla_kat"] = np.asarray(ftk._take_long_axis(tf.constant(arr), tf.constant([[0, 1], [2, 1]])))
    x, y = ftk._exclude(tf.constant(arr), tf.constant([[0, 1, 2], [3, 4, 5]]), tf.constant([[1, 2], [3, 5]]), 1)
    out["exclude_kat_scores"], out["exclude_kat_ids"] = np.asarray(x), np.asarray(y)
    scores = rng.standard_normal((9, 40)).astype(np.float32)
    ident = np.stack([rng.permutation(200)[:40] for _ in range(9)]).astype(np.int64)
    excl = np.stack([np.concatenate([ident[r, rng.permutation(40)[:3]], [100000 + r]]) for r in range(9)]).astype(np.int64)
    idx = rng.randint(0, 40, size=(9, 7)).astype(np.int32)
    out.update(tla_arr=scores, tla_idx=idx, tla_out=np.asarray(ftk._take_long_axis(tf.constant(scores), tf.constant(idx))))
    for k in (5, 40, 60):
        xs, xi = ftk._exclude(tf.constant(scores), tf.constant(ident), tf.constant(excl), k)
        out[f"exclude_k{k}_scores"], out[f"exclude_k{k}_ids"] = np.asarray(xs), np.asarray(xi)
    out.update(exclude_scores=scores, exclude_ident=ident, exclude_excl=excl)

    # indexes: 100 candidates x 4 (the reference test's sizes, :90-96), batches of 32, with and without identifiers
    rs = np.random.RandomState(42)
    cand = rs.normal(size=(100, 4)).astype(np.float32)
    queries = rs.normal(size=(10, 4)).astype(np.float32)
    true_c = rs.normal(size=(10, 4)).astype(np.float32)
    names = (np.arange(100) * 3 + 7).astype(np.int64)
    out.update(idx_candidates=cand, idx_queries=queries, idx_true=true_c, idx_names=names)
    cds = tf.data.Dataset.from_tensor_slices(cand).batch(32)
    nds = tf.data.Dataset.from_tensor_slices(names).batch(32)
    for tag, ids in (("noid", None), ("id", nds)):
        st = ftk.Streaming(k=10).index(cds, ids)
        s, i = st(tf.constant(queries))
        out[f"streaming_{tag}_scores"], out[f"streaming_{tag}_ids"] = np.asarray(s), np.asarray(i)
        bf = ftk.BruteForce(k=10).index(cds, ids)
        s, i = bf(tf.constant(queries))
        out[f"brute_{tag}_scores"], out[f"brute_{tag}_ids"] = np.asarray(s), np.asarray(i)
        s, i = bf(tf.constant(queries), k=3)
        out[f"brute_{tag}_k3_ids"] = np.asarray(i)
    bf = ftk.BruteForce(k=5).index(tf.constant(cand), tf.constant(names))
    s5, i5 = bf(tf.constant(queries))
    ban = np.asarray(i5)[:, [0, 2]].astype(np.int64)
    xs, xi = bf.query_with_exclusions(tf.constant(queries), tf.constant(ban), k=5)
    out.update(qwe_ban=ban, qwe_scores=np.asarray(xs), qwe_ids=np.asarray(xi))
    small = ftk.Streaming(k=50).index(tf.data.Dataset.from_tensor_slices(cand[:40]).batch(32))     # k > batch: clipped
    s, i = small(tf.constant(queries))
    out["streaming_small_scores"], out["streaming_small_ids"] = np.asarray(s), np.asarray(i)
    try:
        ftk.Streaming(k=50, handle_incomplete_batches=False).index(tf.data.Dataset.from_tensor_slices(cand[:40]).batch(32))(tf.constant(queries))
        out["streaming_small_error"] = np.asarray("")
    except ValueError as e:
        out["streaming_small_error"] = np.asarray(str(e))
    # FactorizedTopK metric (:464-522) with the reference test's ks
    ks = [1, 5, 10, 50]
    for tag, layer in (("streaming", ftk.Streaming), ("brute", ftk.BruteForce), ("dataset", None)):
        c = cds if layer is None else layer().index(cds)
        metric = ftk.FactorizedTopK(candidates=c, metrics=[tf.keras.metrics.TopKCategoricalAccuracy(k=x, name=f"top_{x}")
                                                         for x in ks], k=max(ks))
        metric.update_state(query_embeddings=tf.constant(queries), true_candidate_embeddings=tf.constant(true_c))
        out[f"metric_{tag}"] = np.asarray([float(np.asarray(v)) for v in metric.result()], np.float64)
    out["metric_ks"] = np.asarray(ks)
    return out


def main():
    data = generate_retrieval()
    path = os.path.join(HERE, "retrieval_golden.npz")
    np.savez_compressed(path, **data)
    print(path, len(data), "arrays", os.path.getsize(path), "bytes")
    for name, dt in (("f32", np.float32), ("f64", np.float64)):
        data = generate(dt)
        path = os.path.join(HERE, f"hotpath_golden_{name}.npz")
        np.savez_compressed(path, **data)
        print(path, len(data), "arrays", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
