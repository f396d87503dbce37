"""Row g1 of the round-1 verdict: the assembled DCN and TwoTower models (the model classes north_star names on top of
Cross / DNN / the in-batch softmax) checked against float64 compositions of the oracle's layer restatements:
forward, loss and EVERY gradient of one step.

Stacking follows the reference's own model-level test (tests/keras/test_dcn.py:27-32):
    x1 = Cross()(x0, x0); x2 = Cross()(x0, x1); ... ; logits = Dense(1)(...)
and the two-tower step follows Retrieval.call (keras/models/retrieval/sbcnm.py:120-151) with the helper layers'
intended semantics (temperature, accidental-hit removal, sampling-probability correction).
"""
import numpy as np
import pytest
import torch

from oracle import reference_np as R

pytestmark = pytest.mark.gpu

F64 = np.float64


def npy(t):
    return t.detach().cpu().numpy()


def _dnn_backward(hs, ws, g_out, act_all=True):
    """float64 backward through [Dense(relu)...] given hs = [input, h1, ..., h_last]; activation on every layer when
    act_all (DNN(out_units=0)) else linear last layer.  ReLU masks come from hs (the oracle's own forward)."""
    gws, gbs, sws, sbs = [], [], [], []
    g = g_out
    for i in range(len(ws) - 1, -1, -1):
        relu = act_all or i < len(ws) - 1
        gx, gw, gb = R.dense_grad(hs[i], ws[i], hs[i + 1], g, "relu" if relu else None, F64)
        gz = np.abs(g * (hs[i + 1] > 0)) if relu else np.abs(g)
        gws.append(gw)
        gbs.append(gb)
        sws.append(np.abs(hs[i]).T @ gz)          # sum of |terms| of every dot product (cancellation-aware scale:
        sbs.append(gz.sum(0))                     # e.g. the last-layer bias gradient of a tower is exactly 0 in theory)
        g = gx
    _dnn_backward.scales = (sws[::-1], sbs[::-1])
    return g, gws[::-1], gbs[::-1]


@pytest.mark.parametrize("B,S,D,units,ncross,alpha", [
    (200, 6, 8, [32, 16], 2, 0.0),
    (513, 26, 32, [64, 32, 16], 3, 0.1),     # C3-shaped (26 slots, D = 32 -> d = 832, 3 cross layers), small tower
])
def test_dcn_step_matches_oracle(B, S, D, units, ncross, alpha):
    from deep_recommenders.keras.layers import DCN
    rows = [97 + 3 * i for i in range(S)]
    model = DCN(rows, D, num_cross=ncross, dnn_units=units, diag_scale=alpha, seed=5, device="cuda")
    rng = np.random.default_rng(B + S)
    ids = np.stack([rng.integers(-1, r, B) for r in rows], axis=1).astype(np.int64)     # -1 = OOV -> zero row
    y = rng.integers(0, 2, (B, 1)).astype(np.float32)
    idt, yt = torch.from_numpy(ids).cuda(), torch.from_numpy(y).cuda()
    z = model.logits(idt)                                     # builds the lazily created layers
    gen = torch.Generator(device="cuda").manual_seed(B + S)   # not the global generator: its state depends on earlier tests
    with torch.no_grad():                                     # zero-init biases would hide bias-path errors
        for c in model.cross:
            c.bias.normal_(0, 0.1, generator=gen)
        for l in model.dnn.layers:
            l.bias.normal_(0, 0.1, generator=gen)
    model.zero_grad()
    z = model.logits(idt)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(z, yt, reduction="sum")
    loss.backward()

    # ---- float64 oracle composition -----------------------------------------------------
    coll = model.embeddings
    tables = [npy(coll.table(s)) for s in range(S)]
    stack = R.stack_embeddings(tables, ids)                   # [B, S, D], gathered rows (bit-exact copies)
    x0 = stack.reshape(B, S * D).astype(F64)
    cw = [npy(c.kernel).astype(F64) for c in model.cross]
    cb = [npy(c.bias).astype(F64) for c in model.cross]
    xs = [x0]
    for w, b in zip(cw, cb):
        nxt, _ = R.cross(x0, xs[-1], w, b, None, None, alpha, F64)
        xs.append(nxt)
    dw = [npy(l.kernel).astype(F64) for l in model.dnn.layers]
    db = [npy(l.bias).astype(F64) for l in model.dnn.layers]
    # ReLU masks: a unit whose pre-activation lies within rounding of 0 (the float32 forward against this float64 one)
    # may fall on either side, and one such unit moves a whole batch row's term in the weight-gradient column it feeds.
    # Those units take the side the GPU forward took; every other unit's side must agree with the float64 forward.
    with torch.no_grad():
        h_gpu = model.embeddings(idt, want_logit=False)[0].view(B, -1)
    hs = [x0]
    for w, b, layer in zip(dw, db, model.dnn.layers):
        zpre = R.dense(hs[-1], w, b, None, F64)
        with torch.no_grad():
            h_gpu = layer(h_gpu)
        on = npy(h_gpu) > 0
        near0 = np.abs(zpre) <= 2e-5 * (np.abs(hs[-1]) @ np.abs(w) + np.abs(b))
        assert np.array_equal(on[~near0], zpre[~near0] > 0), "ReLU pattern differs from the float64 forward"
        h = np.maximum(zpre, 0)
        h[near0 & on] = np.maximum(zpre[near0 & on], np.finfo(F64).tiny)
        h[near0 & ~on] = 0.0
        hs.append(h)
    hw, hb = npy(model.head.kernel).astype(F64), npy(model.head.bias).astype(F64)
    feat = np.concatenate([xs[-1], hs[-1]], axis=1)
    z_ref = feat @ hw + hb
    p = 1.0 / (1.0 + np.exp(-z_ref))
    loss_ref = float(np.sum(np.maximum(z_ref, 0) - z_ref * y + np.log1p(np.exp(-np.abs(z_ref)))))
    # forward
    zs = np.abs(feat) @ np.abs(hw) + np.abs(hb)
    assert (np.abs(npy(z) - z_ref) <= 2e-5 * zs + 1e-6).all()
    assert abs(float(loss) - loss_ref) <= 1e-5 * abs(loss_ref) + 1e-4
    # backward
    gz = p - y
    g_feat = gz @ hw.T
    want = {"head.kernel": feat.T @ gz, "head.bias": gz.sum(0)}
    d = S * D
    g_x, g_deep = g_feat[:, :d], g_feat[:, d:]
    g_x0_dnn, gws, gbs = _dnn_backward(hs, dw, g_deep, act_all=True)
    scale = {}
    for i, (gw, gb) in enumerate(zip(gws, gbs)):
        want[f"dnn.{i}.kernel"], want[f"dnn.{i}.bias"] = gw, gb
        scale[f"dnn.{i}.kernel"], scale[f"dnn.{i}.bias"] = _dnn_backward.scales[0][i], _dnn_backward.scales[1][i]
    g_x0 = g_x0_dnn.copy()
    g = g_x
    for i in range(ncross - 1, -1, -1):
        gr = R.cross_grad(x0, xs[i], g, cw[i], None, None, cb[i], alpha, F64)
        want[f"cross.{i}.kernel"], want[f"cross.{i}.bias"] = gr["gw"], gr["gb"]
        g_x0 += gr["gx0"]
        g = gr["gx"]
    g_x0 += g                                                 # xs[0] is x0 itself
    got = {"head.kernel": model.head.kernel.grad, "head.bias": model.head.bias.grad}
    for i, l in enumerate(model.dnn.layers):
        got[f"dnn.{i}.kernel"], got[f"dnn.{i}.bias"] = l.kernel.grad, l.bias.grad
    for i, c in enumerate(model.cross):
        got[f"cross.{i}.kernel"], got[f"cross.{i}.bias"] = c.kernel.grad, c.bias.grad
    for k, ref in want.items():
        a = npy(got[k]).reshape(ref.shape)
        # the composition's intermediate activations differ from the fp32 ones by ~1e-6 relative each, and a few
        # ReLU units sit within rounding of 0: tolerance 1e-4 of the gradient's own scale + exact-zero slack
        sc = scale.get(k, np.abs(ref).max())
        assert (np.abs(a - ref) <= 1e-4 * sc + 1e-6).all(), (k, np.abs(a - ref).max(), np.abs(ref).max())
    # table gradients: scatter-add of g_x0 rows (TF: IndexedSlices densified)
    g_tab = [np.zeros_like(t, dtype=F64) for t in tables]
    g3 = g_x0.reshape(B, S, D)
    for s in range(S):
        ok = ids[:, s] >= 0
        np.add.at(g_tab[s], ids[ok, s], g3[ok, s])
    gw_arena = npy(coll.emb_view(coll.weight.grad)) if coll.weight.grad is not None else None
    assert gw_arena is not None, "DCN embedding arena received no gradient"
    off = 0
    for s in range(S):
        a = gw_arena[off:off + rows[s]]
        assert np.abs(a - g_tab[s]).max() <= 1e-4 * np.abs(g_tab[s]).max() + 1e-6, ("table", s)
        off += rows[s]


@pytest.mark.parametrize("B,D,units,tau,accidental,with_p", [
    (128, 32, (), 0.5, True, False),
    (300, 64, (48, 24), 0.2, True, True),
    (257, 64, (), None, False, False),
])
def test_two_tower_step_matches_oracle(B, D, units, tau, accidental, with_p):
    from deep_recommenders.keras.layers import TwoTower
    nu, ni = 500, 400
    tt = TwoTower(nu, ni, dim=D, tower_units=units, temperature=tau, seed=3, device="cuda")
    rng = np.random.default_rng(B + D)
    u = rng.integers(0, nu, B).astype(np.int64)
    it = rng.integers(0, ni // 4, B).astype(np.int64)        # many duplicate items: accidental hits do occur
    sw = rng.uniform(0.5, 1.5, B).astype(np.float32)
    pj = rng.uniform(0.01, 0.5, B).astype(np.float32) if with_p else None
    ut, itt = torch.from_numpy(u).cuda(), torch.from_numpy(it).cuda()
    kw = dict(sample_weight=torch.from_numpy(sw).cuda(),
              candidate_sampling_probability=None if pj is None else torch.from_numpy(pj).cuda(),
              remove_accidental_hits=accidental)
    loss = tt(ut, itt, **kw)
    tt.zero_grad()
    loss = tt(ut, itt, **kw)
    loss.backward()

    def tower(table, ids, dnn):
        e = R.embedding_lookup(npy(table), ids).astype(F64)
        if dnn is None:
            return e, [e], []
        ws = [npy(l.kernel).astype(F64) for l in dnn.layers]
        bs = [npy(l.bias).astype(F64) for l in dnn.layers]
        hs = [e]
        for i, (w, b) in enumerate(zip(ws, bs)):
            hs.append(R.dense(hs[-1], w, b, "relu" if i < len(ws) - 1 else None, F64))
        return hs[-1], hs, ws

    q, qh, qw = tower(tt.user_table, u, tt.user_dnn)
    c, ch, cwt = tower(tt.item_table, it, tt.item_dnn)
    cid = it if accidental else None
    loss_ref, _, _ = R.retrieval_loss(q, c, sw, pj, cid, tau, None, F64)
    assert abs(float(loss) - float(loss_ref)) <= 2e-5 * abs(float(loss_ref)) + 1e-4
    gq, gc = R.retrieval_grad(q, c, sw, pj, cid, tau, F64)

    def check_tower(table_param, ids, dnn, hs, ws, g_out, name):
        if dnn is not None:
            g_e, gws, gbs = _dnn_backward(hs, ws, g_out, act_all=False)
            sws, sbs = _dnn_backward.scales
            for i, l in enumerate(dnn.layers):
                for a, ref, sc, k in ((l.kernel.grad, gws[i], sws[i], "kernel"), (l.bias.grad, gbs[i], sbs[i], "bias")):
                    assert (np.abs(npy(a) - ref) <= 1e-4 * sc + 1e-6).all(), (name, i, k)
        else:
            g_e = g_out
        want = np.zeros(tuple(table_param.shape), F64)
        np.add.at(want, ids, g_e)
        got = npy(table_param.grad)
        assert np.abs(got - want).max() <= 1e-4 * np.abs(want).max() + 1e-6, name

    check_tower(tt.user_table, u, tt.user_dnn, qh, qw, gq, "user")
    check_tower(tt.item_table, it, tt.item_dnn, ch, cwt, gc, "item")
