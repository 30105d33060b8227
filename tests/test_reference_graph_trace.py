"""Architecture parity against the reference's OWN graph-construction code.

tests/golden/reference_graph_trace.json is the canonical layer list obtained by executing /root/reference/adversarial.py
(+ layers.py, ops.py) unmodified under a recording shim of tensorflow (tests/golden/make_reference_graph_trace.py).  Here the
PRODUCT's graph code (pnp_b200.adversarial / networks / layers / ops) runs on CPU with recording stand-ins for its six kernel
entry points (functional.conv_layer, res_block, max_pool2, phase_shift, disc_input, fc) on meta tensors, and the two lists must
agree event by event: filter variable name + shape, stride, dilation, padding rule, dropout keep_prob source, batch-norm scope /
training switch / trainable flag, skip kind, activation, pooling, PS parameters, discriminator input channel layout, matmuls,
plus the full variable table (376 names, shapes, trainable flags) and the weight lists behind the L2 terms.
Nothing here needs a GPU or reads /root/reference."""
import json
import os

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, "golden", "reference_graph_trace.json")) as _f:
    REF = json.load(_f)

CFG = {"mr_front_trainable": False, "ct_front_trainable": True, "joint_trainable": False, "cls_trainable": True, "m_cls_trainable": True}
COST = {"regularizer": 1e-4, "gan_regularizer": 1e-4, "miu_dis": 1e-3, "miu_gen": 2e-3, "lambda_mask_loss": 0.1}
KEEP_PH = 0.4375          # stands for the keep_prob placeholder (a value no Python default of the reference uses)
B = REF["batch"]


class _Tracer(object):
    """recording stand-ins for the kernels behind pnp_b200.functional"""

    def __init__(self, F, rt):
        self.F, self.rt = F, rt
        self.events = []
        self.names = {id(v): k for k, v in rt.graph.vars.items()}
        self.src = {}                      # id(tensor) -> provenance label

    def name(self, t):
        return self.names[id(t)]

    def _conv(self, x, W, cfg, skip):
        F = self.F
        _, g = F._geometry(tuple(x.shape), tuple(W.shape), cfg)
        bn = cfg.bn
        ev = {"op": "conv", "w": self.name(W), "wshape": list(W.shape), "w_trainable": bool(W.requires_grad), "stride": cfg.stride, "dil": cfg.dil,
              "padding": cfg.padding, "in": list(x.shape[1:]), "out": [g.Ho, g.Wo, g.Cout], "keep": float(cfg.keep_prob),
              "bn": None if bn is None else self.name(bn.gamma).rsplit("/", 1)[0],
              "bn_train": None if bn is None else bool(cfg.bn_training), "bn_trainable": None if bn is None else bool(bn.gamma.requires_grad),
              "act": {F.ACT_NONE: "none", F.ACT_RELU: "relu", F.ACT_LRELU: "lrelu0.2"}[cfg.act], "skip": skip,
              "input_layout": getattr(x, "_layout", None)}
        self.events.append(ev)
        y = torch.empty(x.shape[0], g.Ho, g.Wo, g.Cout, device="meta")
        self.src[id(y)] = "out_of:" + ev["w"]
        self._keep = getattr(self, "_keep", []) + [y]          # keep ids alive / unique
        return y

    def conv_layer(self, x, W, cfg, skip=None):
        assert skip is None
        return self._conv(x, W, cfg, "none")

    def res_block(self, x, W1, W2, cfg1, cfg2):
        assert cfg1.skip_off == 0
        h = self._conv(x, W1, cfg1, "none")
        return self._conv(h, W2, cfg2, ("pad%d" % cfg2.skip_off) if cfg2.skip_off else "identity")

    def tail_ps_conv(self, X, w, r, n_channel, batch_size):
        # the product's seventh kernel entry point: ops.PS -> conv2d(padding='SYMMETRIC', keep_prob 1) in one launch
        # (functional._TailFn, numerically pinned by tests/test_ops_gpu.py::test_tail_ps_mirror_conv_equals_three_kernels);
        # structurally it IS the reference's two calls (source_segmenter.py:200-207), so it is recorded as such
        flat = self.phase_shift(X, r, n_channel, batch_size)
        return self.conv_layer(flat, w, self.F.LayerCfg(padding="SYMMETRIC", keep_prob=1.0))

    def max_pool2(self, x):
        self.events.append({"op": "maxpool", "k": 2, "stride": 2, "in": list(x.shape[1:]), "out": [x.shape[1] // 2, x.shape[2] // 2, x.shape[3]]})
        y = torch.empty(x.shape[0], x.shape[1] // 2, x.shape[2] // 2, x.shape[3], device="meta")
        self._keep = getattr(self, "_keep", []) + [y]
        return y

    def _ps_event(self, X, r, n_channel):
        assert X.shape[3] == r * r * n_channel
        self.events.append({"op": "PS", "r": r, "n_channel": n_channel, "in": list(X.shape[1:]), "out": [X.shape[1] * r, X.shape[2] * r, n_channel],
                            "of": self.src.get(id(X))})

    def phase_shift(self, X, r, n_channel, batch_size):
        assert batch_size == B
        self._ps_event(X, r, n_channel)
        y = torch.empty(X.shape[0], X.shape[1] * r, X.shape[2] * r, n_channel, device="meta")
        self.src[id(y)] = "PS(%s)" % self.src.get(id(X))
        self._keep = getattr(self, "_keep", []) + [y]
        return y

    def disc_input(self, c4, c6, b7, c9, logits, batch_size, r=8):
        assert batch_size == B and r == 8
        layout = []
        for t, ntile in zip((c4, c6, b7, c9), (3, 1, 1, 1)):       # the fused gather of functional._DiscInputFn
            g = t.shape[3] // (r * r)
            self._ps_event(t, r, g)
            layout += [["PS(%s)" % self.src.get(id(t)), g]] * ntile
        layout += [[self.src.get(id(logits)), logits.shape[3]], ["argmax(%s)" % self.src.get(id(logits)), 1]]
        y = torch.empty(logits.shape[0], logits.shape[1], logits.shape[2], sum(c for _, c in layout), device="meta")
        y._layout = layout
        self._keep = getattr(self, "_keep", []) + [y]
        return y

    def fc(self, x, w):
        self.events.append({"op": "fc", "w": self.name(w), "wshape": list(w.shape), "w_trainable": bool(w.requires_grad), "in": list(x.shape[1:])})
        return torch.empty(x.shape[0], w.shape[1], device="meta")


class _Graph(object):
    """the variable registry as it was when the fixture built its network (a later Full_DRN resets the global one)"""

    def __init__(self, vars_, order):
        self.vars, self.order = vars_, order
        self.graph = self


def _snapshot(rt):
    return _Graph(dict(rt.graph.vars), list(rt.graph.order))


@pytest.fixture(scope="module")
def product():
    from pnp_b200 import adversarial as A, functional as F, runtime as rt
    net = A.Full_DRN(3, 5, B, cost_kwargs=dict(COST), network_config=dict(CFG))
    tr = _Tracer(F, rt)
    saved = {k: getattr(F, k) for k in ("conv_layer", "res_block", "max_pool2", "phase_shift", "disc_input", "fc", "tail_ps_conv")}
    for k in saved:
        setattr(F, k, getattr(tr, k))
    try:
        out = {}

        def run(label, fn):
            tr.events = []
            r = fn()
            out[label] = tr.events
            return r
        x = torch.empty(B, 256, 256, 3, device="meta")
        # distinct BN switch values per sub-graph prove which switch feeds which layers
        mr = run("mr", lambda: net.segment(x, "mr", KEEP_PH, front_bn=True, joint_bn=False))
        ct = run("ct", lambda: net.segment(x, "ct", KEEP_PH, front_bn=False, joint_bn=True))
        run("cls", lambda: net.create_classifier(ct["c4_2"], ct["c6_2"], ct["b7"], ct["c9_2"], ct["logits"]))
        run("mask", lambda: net.create_mask_critic(ct["logits"]))
    finally:
        for k, v in saved.items():
            setattr(F, k, v)
    return net, _snapshot(rt), out


def _ref_events(section):
    return [e for e in REF["events"] if e["section"] == section]


def _norm_ref(ev, bn_switch):
    """reference event -> the product's vocabulary"""
    e = dict(ev)
    if e["op"] == "conv":
        e["keep"] = KEEP_PH if e["keep"] == "ph:keep_prob" else e["keep"]
        if isinstance(e["bn_train"], str):
            e["bn_train"] = bn_switch[e["bn_train"]]
    return e


CONV_KEYS = ("w", "wshape", "w_trainable", "stride", "dil", "padding", "in", "out", "keep", "bn", "bn_train", "bn_trainable", "act", "skip")


def _compare(ref_list, got_list, bn_switch, what):
    assert len(ref_list) == len(got_list), "%s: %d reference layers vs %d here" % (what, len(ref_list), len(got_list))
    for i, (r, g) in enumerate(zip(ref_list, got_list)):
        r = _norm_ref(r, bn_switch)
        assert r["op"] == g["op"], (what, i, r["op"], g["op"])
        if r["op"] == "conv":
            for k in CONV_KEYS:
                assert r[k] == g[k], "%s layer %d (%s): %s reference %r vs %r" % (what, i, r["w"], k, r[k], g[k])
            assert r["bn_decay"] in (None, 0.9)
            if r.get("input_layout"):
                assert g["input_layout"] == r["input_layout"], (what, i, r["input_layout"], g["input_layout"])
        elif r["op"] == "maxpool":
            assert (r["k"], r["stride"], r["in"], r["out"]) == (g["k"], g["stride"], g["in"], g["out"]), (what, i, r, g)
            assert r["padding"] == "SAME"          # even extents: SAME == VALID for the 2x2/2 pool
        elif r["op"] == "PS":
            for k in ("r", "n_channel", "in", "out", "of"):
                assert r[k] == g[k], (what, i, k, r[k], g[k])
            assert r["batch_size_arg"] == "self.batch_size"
        elif r["op"] == "fc":
            for k in ("w", "wshape", "w_trainable", "in"):
                assert r[k] == g[k], (what, i, k, r[k], g[k])


def test_reference_init_fails_where_the_survey_says():
    assert "predicter" in REF["init_error_after_classifier"]           # adversarial.py:102


def test_mr_and_ct_front_halves_match_the_reference_zip_network(product):
    _, _, got = product
    zipn = _ref_events("create_zip_network#1")
    assert len(zipn) == 48
    mr_ref, ct_ref = zipn[:24], zipn[24:]
    assert mr_ref[0]["input_src"] == "ph:mr_ph" and ct_ref[0]["input_src"].startswith("ph:")
    _compare(mr_ref, got["mr"][:24], {"ph:main_batchnorm_training_switch": True}, "MR front (groups 1-6)")
    _compare(ct_ref, got["ct"][:24], {"ph:adapt_batchnorm_training_switch": False}, "CT front (adapt 1-6)")


def test_second_half_matches_both_reference_calls(product):
    _, _, got = product
    h1, h2 = _ref_events("create_second_half#1"), _ref_events("create_second_half#2")
    strip = lambda evs: [{k: v for k, v in e.items() if k not in ("section", "of")} for e in evs]
    assert strip(h1) == strip(h2)                                        # AUTO_REUSE: the very same layers on the other stream
    _compare(h1, got["ct"][24:], {"ph:joint_batchnorm_training_switch": True}, "second half (CT stream)")
    _compare(h2, got["mr"][24:], {"ph:joint_batchnorm_training_switch": False}, "second half (MR stream)")


def test_feature_discriminator_matches_the_reference(product):
    _, _, got = product
    c1, c2 = _ref_events("create_classifier#1"), _ref_events("create_classifier#2")
    assert [e["w"] for e in c1 if e["op"] != "PS"] == [e["w"] for e in c2 if e["op"] != "PS"]
    _compare(c1, got["cls"], {}, "feature discriminator")
    first = [e for e in got["cls"] if e["op"] == "conv"][0]
    assert sum(c for _, c in first["input_layout"]) == 32 == first["in"][2]


def test_mask_critic_matches_the_reference(product):
    _, _, got = product
    m1, m2 = _ref_events("create_mask_critic#1"), _ref_events("create_mask_critic#2")
    assert [e.get("w") for e in m1] == [e.get("w") for e in m2]
    _compare(m1, got["mask"], {}, "mask critic")


def test_variable_table_and_weight_lists_match_the_reference(product):
    net, rt, _ = product
    ref_vars = REF["variables"]
    # same 376 variables.  Global creation order differs harmlessly (the product builds the shared second half before the CT
    # front and a stage's filters before its batch-norm variables); nothing on the path depends on it: savers and the optimizer
    # variable lists go by name / scope substring (adversarial.py:478-501)
    ref_names = [v["name"] for v in ref_vars]
    assert sorted(ref_names) == sorted(rt.graph.order) and len(set(ref_names)) == len(ref_names) == 376
    top = lambda n: n.split("/")[0]
    is_w = lambda n: n.rsplit("/", 1)[1] not in ("beta", "gamma", "moving_mean", "moving_variance")
    for scope in sorted(set(top(n) for n in ref_names)):       # filter weights keep their creation order inside a scope
        assert [n for n in ref_names if top(n) == scope and is_w(n)] == [n for n in rt.graph.order if top(n) == scope and is_w(n)], scope
    for v in ref_vars:
        t = rt.graph.vars[v["name"]]
        assert list(t.shape) == v["shape"], v["name"]
        assert bool(t.requires_grad) == v["trainable"], v["name"]
    names = {id(v): k for k, v in rt.graph.vars.items()}
    for key in ("mr_front_weights", "ct_front_weights", "cls_weights", "m_cls_weights", "joint_weights"):
        assert [names[id(w)] for w in getattr(net, key)] == REF["weight_lists"][key], key
    # the reference's initialisers: weight_variable (stddev 0.01, tf.Variable) for MR groups 1-4, sharable (0.1) elsewhere
    kinds = {v["name"]: (v["kind"], v["stddev"]) for v in ref_vars if v["kind"] != "batch_norm"}
    assert all(kinds[n] == ("tf.Variable", 0.01) for n in kinds if n.split("/")[0] in ("group_1", "group_2", "group_3", "group_4"))
    assert all(kinds[n] == ("tf.get_variable", 0.1) for n in kinds if n.split("/")[0] not in ("group_1", "group_2", "group_3", "group_4"))


# ------------------------------------------------------------------------------------------------
# source segmenter (source_segmenter.py:48-273; the file's head up to `class Trainer` executed verbatim)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def product_segmenter():
    from pnp_b200 import source_segmenter as S, functional as F, runtime as rt
    args = REF["source_segmenter"]["ctor_args"]
    net = S.Full_DRN(3, 5, B, cost_kwargs={"cross_flag": True, "miu_cross": 1.0, "dice_flag": True, "miu_dice": 1.0, "regularizer": 1e-4}, **args)
    tr = _Tracer(F, rt)
    saved = {k: getattr(F, k) for k in ("conv_layer", "res_block", "max_pool2", "phase_shift", "disc_input", "fc", "tail_ps_conv")}
    for k in saved:
        setattr(F, k, getattr(tr, k))
    try:
        net.forward(torch.empty(B, 256, 256, 3, device="meta"), keep_prob=KEEP_PH, main_bn=True, adapt_bn=False)
    finally:
        for k, v in saved.items():
            setattr(F, k, v)
    return net, _snapshot(rt), tr.events


def test_source_segmenter_file_state_is_what_the_survey_says():
    s = REF["source_segmenter"]
    assert s["syntax_error"]["line"] == 611 and s["executed_lines"] == 302


def test_source_segmenter_network_matches_the_reference(product_segmenter):
    _, _, got = product_segmenter
    ref = REF["source_segmenter"]["events"]
    assert len(ref) == 37
    _compare(ref, got, {"ph:adapt_batchnorm_training_switch": False, "ph:main_batchnorm_training_switch": True}, "source segmenter")
    # groups 1-4 follow adapt_trainable / adapt_bn, groups 5+ main_trainable / main_bn
    for e in ref:
        if e["op"] == "conv":
            early = e["w"].split("/")[0] in ("group_1", "group_2", "group_3", "group_4")
            assert e["w_trainable"] == early, e["w"]
            if e["bn"]:
                assert e["bn_train"] == ("ph:adapt_batchnorm_training_switch" if early else "ph:main_batchnorm_training_switch"), e["w"]


def test_source_segmenter_variables_and_l2_list_match_the_reference(product_segmenter):
    net, rt, _ = product_segmenter
    ref = REF["source_segmenter"]
    names = [v["name"] for v in ref["variables"]]
    assert sorted(names) == sorted(rt.graph.order) and len(names) == 153
    for v in ref["variables"]:
        t = rt.graph.vars[v["name"]]
        assert list(t.shape) == v["shape"] and bool(t.requires_grad) == v["trainable"], v["name"]
        if v["kind"] == "tf.Variable":
            assert v["stddev"] == 0.01                           # weight_variable, layers.py:46-48
    # anonymous batch-norm scopes number in creation order: BatchNorm, BatchNorm_1, ... BatchNorm_29 at the top level
    bn_scopes = [n.rsplit("/", 1)[0] for n in names if n.endswith("/beta")]
    assert bn_scopes == ["BatchNorm"] + ["BatchNorm_%d" % i for i in range(1, 30)]
    # the L2 list with the reference's quirk (source_segmenter.py:132-135): wr4_4 twice, wr4_3 never
    ids = {id(v): k for k, v in rt.graph.vars.items()}
    assert [ids[id(w)] for w in net.conv_weights] == ref["conv_weights"]
    assert ref["conv_weights"].count("group_4/Variable_3") == 2 and "group_4/Variable_2" not in ref["conv_weights"]


# ------------------------------------------------------------------------------------------------
# training wiring: variable groups, optimizers, clip, cost arithmetic (adversarial.py:445-501, 633-656)
# ------------------------------------------------------------------------------------------------
def test_variable_groups_match_the_reference(product):
    net, rt, _ = product
    names = {id(v): k for k, v in rt.graph.vars.items()}
    for key in ("adapt_vars", "cls_vars", "seg_vars", "mri_seg_vars"):
        assert sorted(names[id(v)] for v in getattr(net, key)) == sorted(REF["var_groups"][key]), key
    assert len(REF["var_groups"]["cls_vars"]) == 122 and len(REF["var_groups"]["adapt_vars"]) == 101


def test_optimizer_wiring_matches_the_reference():
    from pnp_b200 import adversarial as A, runtime as rt
    net = A.Full_DRN(3, 5, B, cost_kwargs=dict(COST), network_config=dict(CFG))          # (makes its graph the current one)
    opt = REF["optimizer"]
    d_ref, g_ref = opt["optimizers"]
    sub = opt["train_config_used"]
    tr = A.Trainer(net, batch_size=B, opt_kwargs={"learning_rate": opt["learning_rate_node"]}, train_config=dict(sub, lr_update=False))
    names = {id(v): k for k, v in rt.graph.vars.items()}
    trainable = {v["name"] for v in REF["variables"] if v["trainable"]}
    # minimize(var_list=cls_vars / adapt_vars): the variables that can receive a gradient
    assert d_ref["kind"] == g_ref["kind"] == "RMSPropOptimizer" and d_ref["kwargs"] == g_ref["kwargs"] == {}
    assert sorted(names[id(v)] for v in tr.d_vars) == sorted(n for n in d_ref["var_list"] if n in trainable)
    assert sorted(names[id(v)] for v in tr.g_vars) == sorted(n for n in g_ref["var_list"] if n in trainable)
    assert tr.dis_optimizer.get_lr() == pytest.approx(d_ref["learning_rate"]) and tr.gen_optimizer.get_lr() == pytest.approx(g_ref["learning_rate"])
    assert (tr.dis_optimizer.decay, tr.dis_optimizer.momentum, tr.dis_optimizer.eps) == (0.9, 0.0, 1e-10)      # TF-1.4 defaults
    # objectives: dis_loss + dis_reg / dis_sub_iter   and   ct_gen_loss + gen_reg / gen_sub_iter
    assert d_ref["objective"] == {"dis_loss": 1.0, "dis_reg": pytest.approx(1.0 / sub["dis_sub_iter"])}
    assert g_ref["objective"] == {"ct_gen_loss": 1.0, "gen_reg": pytest.approx(1.0 / sub["gen_sub_iter"])}
    # ... which the product folds into per-variable weight decay: d(objective)/dw = coefficient * multiplicity * w
    mult = lambda key, n: REF["weight_lists"][key].count(n)
    wd_d = dict(zip((names[id(v)] for v in tr.d_vars), tr.dis_optimizer.seg_wd.tolist()))
    for n, got in wd_d.items():
        lam = net.lambda_mask_loss if n.startswith("mask_cls_scope") else 1.0
        m = mult("cls_weights", n) + mult("m_cls_weights", n)
        want = net.gan_reg_coeff * net.miu_dis * m * lam / sub["dis_sub_iter"]
        assert got == pytest.approx(want, rel=1e-6, abs=1e-12), n
    wd_g = dict(zip((names[id(v)] for v in tr.g_vars), tr.gen_optimizer.seg_wd.tolist()))
    for n, got in wd_g.items():
        want = net.gan_reg_coeff * net.miu_gen * mult("ct_front_weights", n) / sub["gen_sub_iter"]
        assert got == pytest.approx(want, rel=1e-6, abs=1e-12), n
    # clip_op: +-0.03 on every cls variable whose name contains "Variable" (26 filters / FC matrices, no batch-norm parameter)
    clip_ref = {c["var"]: (c["lo"], c["hi"]) for c in opt["clip"]}
    assert len(clip_ref) == 26 and set(clip_ref.values()) == {(-0.03, 0.03)} and all(c["of_same_var"] for c in opt["clip"])
    clip_got = dict(zip((names[id(v)] for v in tr.d_vars), tr.dis_optimizer.seg_clip.tolist()))
    assert {n for n, c in clip_got.items() if c > 0} == set(clip_ref) and all(c == pytest.approx(0.03) for c in clip_got.values() if c > 0)
    assert all(c == 0 for c in tr.gen_optimizer.seg_clip.tolist())


def test_oracle_cost_arithmetic_equals_the_reference_code():
    """adversarial.py:445-476 executed numerically by the reference vs OracleAdversarial.dis_losses / gen_losses"""
    import numpy as np
    from oracle import pnp_graphs as PG
    c = REF["cost_numeric"]
    for case in c["cases"]:
        ck = case["cost_kwargs"]
        lam = ck.get("lambda_mask_loss", 1.0)
        adv = PG.OracleAdversarial({}, B, dtype=torch.float64, miu_dis=ck["miu_dis"], miu_gen=ck["miu_gen"], lambda_mask_loss=lam,
                                   gan_regularizer=ck["gan_regularizer"], regularizer=ck["regularizer"])
        for n, v in c["l2"].items():
            if n in adv.ps.w:
                adv.ps.w[n] = torch.tensor([np.sqrt(2.0 * v)], dtype=torch.float64)        # l2_loss(w) == v
        co = {k: torch.tensor(v, dtype=torch.float64).reshape(-1, 1) for k, v in c["critic_outputs"].items()}
        dis_loss, dis_reg = adv.dis_losses(co["ct_cls"], co["mr_cls"], co["ct_mask"], co["mr_mask"])
        gen_loss, gen_reg = adv.gen_losses(co["ct_cls"], co["ct_mask"])
        for got, key in ((dis_loss, "dis_loss"), (dis_reg, "dis_reg"), (gen_loss, "gen_loss"), (gen_reg, "gen_reg")):
            assert float(got) == pytest.approx(case[key], rel=1e-12, abs=1e-18), (key, lam)
        del adv


def test_oracle_supervised_losses_equal_the_reference_code():
    """source_segmenter.py:241-273 executed numerically by the reference vs the oracle's numpy and torch forms"""
    import numpy as np
    from oracle import tf14_numpy as N, tf14_torch as T
    s = REF["source_segmenter"]["losses_numeric"]
    logits = np.array(s["logits"], dtype=np.float64)
    y = np.eye(5)[np.array(s["labels"])]
    assert N.softmax_weighted_loss(logits, y) == pytest.approx(s["weighted_loss"], rel=1e-12)
    assert N.dice_loss(logits, y) == pytest.approx(s["dice_loss"], rel=1e-12)
    lt, yt = torch.from_numpy(logits), torch.from_numpy(y)
    assert float(T.softmax_weighted_loss(lt, yt)) == pytest.approx(s["weighted_loss"], rel=1e-12)
    assert float(T.dice_loss(lt, yt)) == pytest.approx(s["dice_loss"], rel=1e-12)
    assert (np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)).min() < 0.005          # the clip is exercised


# ------------------------------------------------------------------------------------------------
# the training schedule and the per-step feeds (adversarial.py:767-946, executed verbatim against a recording Session)
# ------------------------------------------------------------------------------------------------
def test_training_schedule_and_step_feeds_match_the_reference(tmp_path):
    from pnp_b200 import adversarial as A, optim, runtime as rt, _C
    sched = REF["schedule"]
    ref_ops = []
    for e in sched["events"]:
        if e["op"] == "dis_optimizer":
            ref_ops.append("D")
        elif e["op"] == "clip_op":
            assert ref_ops and ref_ops[-1] == "D" and e["n"] == 26            # every discriminator update is followed by the clip
            ref_ops[-1] = "D+clip"
        elif e["op"] == "gen_optimizer":
            ref_ops.append("G")
    # step 0 trains nothing; dis_sub_iter grows by dis_sub_iter_inc every iter_upd_interval steps
    assert ref_ops == ["D+clip", "D+clip", "G"] * 2 + ["D+clip", "D+clip", "D+clip", "G"] * 2
    d_feeds = [e["feeds"] for e in sched["events"] if e["op"] == "dis_optimizer"]
    g_feeds = [e["feeds"] for e in sched["events"] if e["op"] == "gen_optimizer"]
    assert all(f == {"mr": "batch", "ct": "batch", "mr_front_bn": False, "joint_bn": False, "ct_front_bn": False, "cls_bn": True,
                     "keep_prob": 0.75} for f in d_feeds)
    assert all(f == {"ct": "batch", "mr_front_bn": False, "joint_bn": False, "ct_front_bn": True, "cls_bn": False, "keep_prob": 0.75}
               for f in g_feeds)
    assert [e for e in sched["events"] if e["op"] == "assign_lr"] == [{"op": "assign_lr", "value": 3e-4}]      # lr_update

    # ---- the product's loop with recording steps
    net = A.Full_DRN(3, 5, B, cost_kwargs=dict(COST), network_config=dict(CFG))
    tr = A.Trainer(net, num_cls=5, batch_size=B, opt_kwargs={"learning_rate": 3e-4}, train_config=dict(sched["train_config"]))
    got = []
    tr.d_step = lambda mr, ct, keep_prob=0.75, apply=True: got.append(("D+clip", keep_prob, tuple(mr.shape), tuple(ct.shape)))
    tr.g_step = lambda ct, keep_prob=0.75, apply=True: got.append(("G", keep_prob, tuple(ct.shape)))
    wd_before = tr.dis_optimizer.seg_wd.clone()
    mon = []
    tr.output_minibatch_stats = lambda step, ct, cty, mr, mry, log_dir=None, detail=False: mon.append((step, os.path.basename(log_dir), detail))
    tr.train(output_path=str(tmp_path), restore=True, restored_path=str(tmp_path), **sched["train_args"])
    # the monitoring passes (adversarial.py:894-922): every display_step a training batch, then a validation batch with the table
    # into FileWriter(output_path + "/train_log" + tag) / "/val_log" + tag (adversarial.py:807-808)
    tag = sched["train_config"].get("tag", "")
    assert mon and all(a[1:] == ("train_log" + tag, False) and b[1:] == ("val_log" + tag, True) and a[0] == b[0]
                       for a, b in zip(mon[0::2], mon[1::2]))
    assert [g[0] for g in got] == ref_ops
    assert all(g[1] == 0.75 for g in got) and all(g[2] == (B, 256, 256, 3) for g in got)
    assert tr.dis_sub_iter == 4 and tr.gen_sub_iter == 1
    assert torch.equal(tr.dis_optimizer.seg_wd, wd_before)          # the objective keeps its construction-time 1/dis_sub_iter

    # ---- which BN switches the product's two steps use: run them up to the segmenter calls
    calls = []

    class _Stop(Exception):
        pass

    def probe(n_expected):
        def segment(x, stream, keep_prob, front_bn, joint_bn=False):
            calls.append({"stream": stream, "keep_prob": keep_prob, "front_bn": front_bn, "joint_bn": joint_bn})
            if len(calls) == n_expected:
                raise _Stop()
            return {}
        return segment
    tr2 = A.Trainer(A.Full_DRN(3, 5, B, cost_kwargs=dict(COST), network_config=dict(CFG)), num_cls=5, batch_size=B,
                    opt_kwargs={"learning_rate": 3e-4}, train_config=dict(sched["train_config"]))
    # scratch.begin_step() drops its record of the used accumulators; with its zero-fill a no-op here, that record is restored
    # afterwards, or the next real step on a device would accumulate onto stale sums
    saved = (optim.call, _C.call, rt.stream, rt.scratch.off, rt.scratch.high)
    optim.call = _C.call = lambda *a, **k: None                      # no kernels: only the Python control flow is exercised
    rt.stream = lambda: None
    x = torch.empty(B, 256, 256, 3, device="meta")
    try:
        tr2.net.segment = probe(2)
        with pytest.raises(_Stop):
            tr2.d_step(x, x, 0.75)
        d_calls, calls = calls, []
        tr2.net.segment = probe(1)
        with pytest.raises(_Stop):
            tr2.g_step(x, 0.75)
        g_calls = calls
    finally:
        optim.call, _C.call, rt.stream, rt.scratch.off, rt.scratch.high = saved
    assert d_calls == [{"stream": "mr", "keep_prob": 0.75, "front_bn": d_feeds[0]["mr_front_bn"], "joint_bn": d_feeds[0]["joint_bn"]},
                       {"stream": "ct", "keep_prob": 0.75, "front_bn": d_feeds[0]["ct_front_bn"], "joint_bn": d_feeds[0]["joint_bn"]}]
    assert g_calls == [{"stream": "ct", "keep_prob": 0.75, "front_bn": g_feeds[0]["ct_front_bn"], "joint_bn": g_feeds[0]["joint_bn"]}]


# ------------------------------------------------------------------------------------------------
# checkpoint transplant chain (adversarial.py:503-531, 706-765 executed on the reference's lists/ and the traced tables)
# ------------------------------------------------------------------------------------------------
def test_transplant_chain_matches_the_reference(tmp_path):
    import numpy as np
    from pnp_b200 import adversarial as A, runtime as rt
    tp = REF["transplant"]
    strip = lambda n: n.split(":")[0]
    net = A.Full_DRN(3, 5, B, cost_kwargs=dict(COST), network_config=dict(CFG))
    V = rt.graph.vars

    # ---- _adapt_copy_weights: CT DAM <- MR front, 101 (destination, source) pairs from lists/half_zip_*_vars
    assert len(tp["adapt_copy"]) == 101 and "adapt_copy_internal_error" in tp          # the `internal` mode cannot work: 153 vs 101
    with torch.no_grad():
        for i, name in enumerate(rt.graph.order):
            V[name].fill_(float(i + 1))
    before = {n: float(V[n].detach().flatten()[0]) for n in rt.graph.order}
    net.adapt_copy_weights()
    changed = {n for n in rt.graph.order if float(V[n].detach().flatten()[0]) != before[n]}
    assert changed == {d for d, _ in tp["adapt_copy"]}
    for dst, src in tp["adapt_copy"]:
        assert torch.all(V[dst] == before[src]), (dst, src)

    # ---- _load_batch_norm_weights: baseline 'BatchNorm_k/*' -> 'group_g/pred_*' (lists/old_bn_list -> lists/pred_bn_list)
    assert len(tp["bn_copy"]) == 120 == tp["bn_copy_dict_len"]
    base = {}
    for k, (old, new) in enumerate(tp["bn_copy"]):
        base[strip(old)] = np.full(tuple(V[new].shape), 1000.0 + k, np.float32)
    np.savez(str(tmp_path / "baseline.npz"), **base)
    before = {n: float(V[n].detach().flatten()[0]) for n in rt.graph.order}
    net.load_batch_norm_weights(str(tmp_path / "baseline.npz"))
    changed = {n for n in rt.graph.order if float(V[n].detach().flatten()[0]) != before[n]}
    assert changed == {new for _, new in tp["bn_copy"]}
    for k, (old, new) in enumerate(tp["bn_copy"]):
        assert torch.all(V[new] == 1000.0 + k), (old, new)

    # ---- restore(no_gan=True) from a baseline-segmenter checkpoint: the 33 'group*' / 'output' filters, no batch norm, no slots
    rs = tp["restore_no_gan"]
    shapes = {v["name"]: v["shape"] for v in REF["source_segmenter"]["variables"]}
    ck = {}
    for k, n in enumerate(rs["checkpoint_names"]):
        base_name = n[:-5] if n.endswith("/Adam") else n
        ck[n] = np.full(tuple(shapes.get(base_name, [1])), 5000.0 + k, np.float32)
    np.savez(str(tmp_path / "seg.npz"), **ck)
    before = {n: float(V[n].detach().flatten()[0]) for n in rt.graph.order}
    net.restore(str(tmp_path / "seg.npz"), no_gan=True)
    changed = {n for n in rt.graph.order if float(V[n].detach().flatten()[0]) != before[n]}
    assert changed == set(rs["restored"]) and len(changed) == 33


# ------------------------------------------------------------------------------------------------
# source segmenter training (source_segmenter.py:312-570, class Trainer up to test_eval executed verbatim)
# ------------------------------------------------------------------------------------------------
def test_segmenter_training_schedule_feeds_and_adam_match_the_reference(tmp_path):
    from pnp_b200 import source_segmenter as S, optim, runtime as rt, _C
    ref = REF["source_segmenter"]
    sched = ref["schedule"]
    assert ref["executed_lines_trainer"] == 571                       # everything before `def test_eval` (syntax error at :611)
    # ---- Adam on cost + regularizer_loss over every trainable variable
    (adam,) = sched["optimizer"]
    assert adam == {"kind": "AdamOptimizer", "learning_rate": 1e-3, "kwargs": {}, "objective_src": "add(cost,regularizer_loss)", "var_list": None}
    net = S.Full_DRN(3, 5, B, cost_kwargs={"cross_flag": True, "miu_cross": 1.0, "dice_flag": True, "miu_dice": 1.0, "regularizer": 1e-4})
    tr = S.Trainer(net, train_list=[], val_list=[], num_cls=5, batch_size=B, opt_kwargs={"learning_rate": 1e-3}, checkpoint_space=1500,
                   optimizer="adam", lr_update_flag=False)
    names = {id(v): k for k, v in rt.graph.vars.items()}
    trainable = [v["name"] for v in ref["variables"] if v["kind"] != "batch_norm" or v["name"].endswith(("beta", "gamma"))]
    assert sorted(names[id(v)] for v in tr.trainables) == sorted(trainable)          # defaults: main/adapt trainable True
    assert tr.optimizer.get_lr() == pytest.approx(1e-3) and (tr.optimizer.b1, tr.optimizer.b2, tr.optimizer.eps) == (0.9, 0.999, 1e-8)
    # d(reg_coeff * sum l2_loss(conv_weights))/dw = reg_coeff * multiplicity * w   (wr4_4 twice, wr4_3 never)
    wd = dict(zip((names[id(v)] for v in tr.trainables), net.weight_decay_table(tr.trainables)))
    for n, c in wd.items():
        assert c == pytest.approx(1e-4 * ref["conv_weights"].count(n)), n
    assert wd["group_4/Variable_3"] == pytest.approx(2e-4) and wd["group_4/Variable_2"] == 0.0

    # ---- per-step feeds
    evs = sched["events"]
    train_feeds = [e["feeds"] for e in evs if e["op"] == "optimizer"]
    stats_feeds = [e["feeds"] for e in evs if e["op"] == "minibatch_stats"]
    val_feeds = [e["feeds"] for e in evs if e["op"] == "val_stats"]
    assert all(f == {"x": "batch", "y": "batch", "main_bn": True, "adapt_bn": True, "keep_prob": 0.75} for f in train_feeds)
    assert all(f == {"x": "batch", "y": "batch", "keep_prob": 1.0} for f in stats_feeds)       # BN switches at their default: True
    assert all(f == {"x": "batch", "y": "batch", "main_bn": False, "adapt_bn": False, "keep_prob": 1.0} for f in val_feeds)

    # ---- schedule: one Adam step per iteration, the stats pass (and validation) every display_step = 5 iterations, after it
    ref_ops = [e["op"] for e in evs]
    assert ref_ops == ["optimizer", "minibatch_stats", "val_stats"] + ["optimizer"] * 5 + ["minibatch_stats", "val_stats", "optimizer"]
    assert all(e["detail"] is True for e in evs if e["op"] == "val_stats")
    got = []
    tr.train_step = lambda x, y, keep_prob=0.75: got.append(("optimizer", keep_prob)) or (0.0, 0.0)
    tr.output_minibatch_stats = lambda x, y, step=None, log_dir=None: got.append(("minibatch_stats", os.path.basename(log_dir), step)) or 0.0
    tr.val_stats = lambda x, y, step=None, log_dir=None, detail=False: got.append(("val_stats", os.path.basename(log_dir), step, detail)) or {}
    tr.feed = lambda images, raw: (images, raw)
    tr.train(output_path=str(tmp_path), training_iters=7, epochs=1, restore=True, restored_path=str(tmp_path))
    assert [g[0] for g in got] == ref_ops and all(g[1] == 0.75 for g in got if g[0] == "optimizer")
    # the two writers of source_segmenter.py:464-465, the step each summary is filed under, the always-on per-organ table
    assert [g[1:] for g in got if g[0] == "minibatch_stats"] == [("train_log", 0), ("train_log", 5)]
    assert [g[1:] for g in got if g[0] == "val_stats"] == [("val_log", 0, True), ("val_log", 5, True)]

    # ---- the BN switches the product's three passes use
    calls = []

    class _Stop(Exception):
        pass

    def forward(x, keep_prob=1.0, main_bn=True, adapt_bn=True, return_taps=False):
        calls.append({"keep_prob": keep_prob, "main_bn": main_bn, "adapt_bn": adapt_bn})
        raise _Stop()
    tr2 = S.Trainer(S.Full_DRN(3, 5, B, cost_kwargs={"cross_flag": True, "miu_cross": 1.0, "dice_flag": True, "miu_dice": 1.0}),
                    train_list=[], val_list=[], num_cls=5, batch_size=B, opt_kwargs={"learning_rate": 1e-3}, optimizer="adam")
    tr2.net.forward = forward
    saved = (optim.call, _C.call, rt.stream, rt.scratch.off, rt.scratch.high)      # scratch: as in the adversarial probe above
    optim.call = _C.call = lambda *a, **k: None
    rt.stream = lambda: None
    x = torch.empty(B, 256, 256, 3, device="meta")
    try:
        for fn in (lambda: tr2.train_step(x, x, 0.75), lambda: tr2.output_minibatch_stats(x, x), lambda: tr2.val_stats(x, x)):
            with pytest.raises(_Stop):
                fn()
    finally:
        optim.call, _C.call, rt.stream, rt.scratch.off, rt.scratch.high = saved
    assert calls == [{"keep_prob": 0.75, "main_bn": True, "adapt_bn": True},
                     {"keep_prob": 1.0, "main_bn": True, "adapt_bn": True},
                     {"keep_prob": 1.0, "main_bn": False, "adapt_bn": False}]


# ------------------------------------------------------------------------------------------------
# input pipeline (adversarial.py:607-631 evaluated numerically on one parsed example)
# ------------------------------------------------------------------------------------------------
def test_tfrecord_decoding_matches_the_reference_pipeline(tmp_path):
    import numpy as np
    from pnp_b200 import tfrecord as R
    ip = REF["input_pipeline"]
    assert ip["feature_keys"] == sorted(["dsize_dim0", "dsize_dim1", "dsize_dim2", "lsize_dim0", "lsize_dim1", "lsize_dim2", "data_vol", "label_vol"])
    assert ip["pair_shape"] == [B, 256, 256, 4] and ip["shuffle_batch"]["batch_size"] == B
    # the same synthetic example (formula of make_reference_graph_trace.pipeline_example)
    i, j, c = np.meshgrid(np.arange(256), np.arange(256), np.arange(3), indexing="ij")
    data = (1000.0 * c + (i * 256 + j) % 997).astype(np.float32)
    label = ((i * 3 + j * 5 + c * 2) % 5).astype(np.float32)
    path = str(tmp_path / "one.tfrecords")
    R.write_record(path, [R.encode_example(data, label)])
    src = R.TFRecordSource([path], 1, seed=0)
    x, y = src.next()
    pair = np.concatenate([x.numpy()[0], y.numpy()[0][..., None].astype(np.float32)], axis=2)      # [256,256,4] like pair_feed
    rows, cols = ip["sample_rows"], ip["sample_cols"]
    np.testing.assert_array_equal(pair[np.ix_(rows, cols)], np.array(ip["samples"], dtype=np.float32))
    for ch in range(4):
        assert float(pair[:, :, ch].astype(np.float64).sum()) == ip["channel_sums"][ch], ch
    np.testing.assert_array_equal(y.numpy()[0], label[:, :, 1].astype(np.int64))                   # tf.slice(label_vol, [0,0,1], [256,256,1])


# ------------------------------------------------------------------------------------------------
# the ORACLE's graphs against the same reference trace (closes reference -> oracle on the CPU; the GPU tests close oracle -> kernels)
# ------------------------------------------------------------------------------------------------
class _OracleTracer(object):
    """recording stand-ins for the primitives of oracle/tf14_torch.py; the composite layers above them run unmodified"""

    def __init__(self, T, wname, bnname):
        self.T, self.wname, self.bnname = T, wname, bnname
        self.events, self.open, self.cur, self.pad = [], None, None, None
        self.keep = []

    def _new(self, shape):
        y = torch.empty(*shape, device="meta")
        self.keep.append(y)
        return y

    def close(self):
        if self.open is not None:
            self.events.append(self.open)
            self.open = None

    def conv2d_raw(self, x, w, stride=1, dilation=1, padding="SAME"):
        self.close()
        kh, kw, ci, co = w.shape
        assert ci == x.shape[3]
        if padding == "SYMMETRIC":
            ho = (x.shape[1] + 2 * (kh // 2) - ((kh - 1) * dilation + 1)) // stride + 1
            wo = (x.shape[2] + 2 * (kw // 2) - ((kw - 1) * dilation + 1)) // stride + 1
        else:
            assert padding == "SAME"
            ho, wo = -(-x.shape[1] // stride), -(-x.shape[2] // stride)
        y = self._new((x.shape[0], ho, wo, co))
        self.open = {"op": "conv", "w": self.wname[id(w)], "wshape": list(w.shape), "stride": stride, "dil": dilation, "padding": padding,
                     "in": list(x.shape[1:]), "out": [ho, wo, co], "keep": None, "bn": None, "bn_train": None, "skip": "none", "act": "none"}
        self.cur, self.pad = id(y), None
        return y

    def dropout(self, x, keep_prob, mask=None):
        assert self.open is not None and id(x) == self.cur and self.open["bn"] is None
        self.open["keep"] = float(keep_prob)
        y = self._new(x.shape)
        self.cur = id(y)
        return y

    def batch_norm(self, x, bn, is_training):
        assert self.open is not None and id(x) == self.cur
        self.open["bn"], self.open["bn_train"] = self.bnname[id(bn)], bool(is_training)
        y = self._new(x.shape)
        self.cur = id(y)
        return y

    def channel_pad_skip(self, x):
        self.pad = x.shape[-1] // 2
        return self._new(tuple(x.shape[:3]) + (2 * x.shape[3],))

    def act(self, x, leak):
        assert self.open is not None
        if id(x) != self.cur:                      # x is `xs + h`: the residual add of layers.py:164-166 / 186-189
            self.open["skip"] = ("pad%d" % self.pad) if self.pad else "identity"
        self.open["act"] = "lrelu0.2" if leak else "relu"
        self.close()
        y = self._new(x.shape)
        self.pad = None
        return y

    def max_pool2d(self, x, n=2):
        self.close()
        self.events.append({"op": "maxpool", "k": n, "stride": n, "in": list(x.shape[1:]), "out": [x.shape[1] // n, x.shape[2] // n, x.shape[3]]})
        return self._new((x.shape[0], x.shape[1] // n, x.shape[2] // n, x.shape[3]))

    def PS(self, X, r, n_channel, batch_size):
        self.close()
        assert batch_size == B and X.shape[3] == r * r * n_channel
        self.events.append({"op": "PS", "r": r, "n_channel": n_channel, "in": list(X.shape[1:]), "out": [X.shape[1] * r, X.shape[2] * r, n_channel]})
        return self._new((X.shape[0], X.shape[1] * r, X.shape[2] * r, n_channel))


def test_oracle_graphs_match_the_reference_trace():
    from oracle import pnp_graphs as PG, tf14_torch as T
    adv = PG.OracleAdversarial({}, B, critic_keep_prob=0.75)
    wname, bnname = {}, {id(bn): k for k, bn in adv.ps.bn.items()}
    for k in list(adv.ps.w):
        t = torch.empty(adv.ps.w[k].shape, device="meta")
        adv.ps.w[k] = t
        wname[id(t)] = k
    tr = _OracleTracer(T, wname, bnname)
    names = ("conv2d_raw", "dropout", "batch_norm", "channel_pad_skip", "act", "max_pool2d", "PS")
    saved = {k: getattr(T, k) for k in names}
    for k in names:
        setattr(T, k, getattr(tr, k))
    try:
        got = {}

        def run(label, fn):
            tr.events = []
            r = fn()
            tr.close()
            got[label] = tr.events
            return r
        x = torch.empty(B, 256, 256, 3, device="meta")
        run("mr", lambda: adv.segment(x, "mr", KEEP_PH, front_bn=True, joint_bn=False))
        ct = run("ct", lambda: adv.segment(x, "ct", KEEP_PH, front_bn=False, joint_bn=True))
        run("cls", lambda: adv.classifier(ct["c4_2"], ct["c6_2"], ct["b7"], ct["c9_2"], ct["logits"]))
        run("mask", lambda: adv.mask_critic(ct["logits"]))
    finally:
        for k, v in saved.items():
            setattr(T, k, v)

    keys = ("w", "wshape", "stride", "dil", "padding", "in", "out", "keep", "bn", "bn_train", "act", "skip")

    def compare(ref_list, got_list, bn_switch, what):
        ref_list = [e for e in ref_list if e["op"] != "fc"]              # the oracle's matmul is a plain torch `@`
        assert len(ref_list) == len(got_list), (what, len(ref_list), len(got_list))
        for i, (r, g) in enumerate(zip(ref_list, got_list)):
            r = _norm_ref(r, bn_switch)
            assert r["op"] == g["op"], (what, i)
            for k in (keys if r["op"] == "conv" else ("r", "n_channel", "in", "out") if r["op"] == "PS" else ("k", "stride", "in", "out")):
                assert r[k] == g[k], "%s layer %d (%s): %s reference %r vs oracle %r" % (what, i, r.get("w"), k, r[k], g[k])
    zipn = _ref_events("create_zip_network#1")
    compare(zipn[:24], got["mr"][:24], {"ph:main_batchnorm_training_switch": True}, "oracle MR front")
    compare(zipn[24:], got["ct"][:24], {"ph:adapt_batchnorm_training_switch": False}, "oracle CT front")
    compare(_ref_events("create_second_half#1"), got["ct"][24:], {"ph:joint_batchnorm_training_switch": True}, "oracle second half (CT)")
    compare(_ref_events("create_second_half#2"), got["mr"][24:], {"ph:joint_batchnorm_training_switch": False}, "oracle second half (MR)")
    compare(_ref_events("create_classifier#1"), got["cls"], {}, "oracle feature discriminator")
    compare(_ref_events("create_mask_critic#1"), got["mask"], {}, "oracle mask critic")
    # variable tables of the oracle's layout() against the reference's
    ws, bns = PG.OracleAdversarial.layout(5)
    ref_w = {v["name"]: v["shape"] for v in REF["variables"] if v["kind"] != "batch_norm"}
    assert {n: list(s) for n, s in ws} == ref_w
    ref_bn = {v["name"].rsplit("/", 1)[0]: v["shape"][0] for v in REF["variables"] if v["kind"] == "batch_norm"}
    assert dict(bns) == ref_bn


def test_oracle_segmenter_matches_the_reference_trace():
    from oracle import pnp_graphs as PG, tf14_torch as T
    seg = PG.OracleSegmenter({}, B)
    wname, bnname = {}, {id(bn): k for k, bn in seg.ps.bn.items()}
    for k in list(seg.ps.w):
        t = torch.empty(seg.ps.w[k].shape, device="meta")
        seg.ps.w[k] = t
        wname[id(t)] = k
    tr = _OracleTracer(T, wname, bnname)
    names = ("conv2d_raw", "dropout", "batch_norm", "channel_pad_skip", "act", "max_pool2d", "PS")
    saved = {k: getattr(T, k) for k in names}
    for k in names:
        setattr(T, k, getattr(tr, k))
    try:
        seg.forward(torch.empty(B, 256, 256, 3, device="meta"), keep_prob=KEEP_PH, bn_train=True)
        tr.close()
    finally:
        for k, v in saved.items():
            setattr(T, k, v)
    ref = REF["source_segmenter"]["events"]
    assert len(ref) == len(tr.events) == 37
    sw = {"ph:adapt_batchnorm_training_switch": True, "ph:main_batchnorm_training_switch": True}      # the oracle has one switch
    for i, (r, g) in enumerate(zip(ref, tr.events)):
        r = _norm_ref(r, sw)
        assert r["op"] == g["op"], i
        for k in (("w", "wshape", "stride", "dil", "padding", "in", "out", "keep", "bn", "bn_train", "act", "skip") if r["op"] == "conv"
                  else ("r", "n_channel", "in", "out") if r["op"] == "PS" else ("k", "stride", "in", "out")):
            assert r[k] == g[k], "segmenter layer %d (%s): %s reference %r vs oracle %r" % (i, r.get("w"), k, r[k], g[k])
    # variable layout and the L2 list (with the wr4_4 / wr4_3 quirk)
    ws, bns = PG.OracleSegmenter.layout(5)
    rv = REF["source_segmenter"]["variables"]
    assert {n: list(s) for n, s in ws} == {v["name"]: v["shape"] for v in rv if v["kind"] != "batch_norm"}
    assert dict(bns) == {v["name"].rsplit("/", 1)[0]: v["shape"][0] for v in rv if v["kind"] == "batch_norm"}
    assert sorted(seg.l2_names) == sorted(REF["source_segmenter"]["conv_weights"])


def test_gan_checkpoint_restore_branches_match_the_reference(tmp_path):
    """adversarial.py:533-574: clear_rms, the full restore, and the relaxed branch a partial checkpoint falls into"""
    import numpy as np
    from pnp_b200 import adversarial as A, runtime as rt
    cases = REF["transplant"]["restore_gan"]
    for label, kw in (("full_default", {}), ("full_clear_rms", {"clear_rms": True}), ("partial_default", {})):
        case = cases[label]
        net = A.Full_DRN(3, 5, B, cost_kwargs=dict(COST), network_config=dict(CFG, restore_skip_kwd=case["skip_kwd"]))
        V = rt.graph.vars
        stored = [n for n in case["checkpoint_names"] if "RMSProp" not in n]      # this checkpoint format carries no optimizer slots
        np.savez(str(tmp_path / (label + ".npz")), **{n: np.full(tuple(V[n].shape), 7.5, np.float32) for n in stored})
        with torch.no_grad():
            for n in rt.graph.order:
                V[n].fill_(-1.0)
        net.restore(str(tmp_path / (label + ".npz")), **kw)
        changed = sorted(n for n in rt.graph.order if float(V[n].detach().flatten()[0]) == 7.5)
        want = sorted(n for n in case["restored"] if "RMSProp" not in n)
        assert changed == want, (label, len(changed), len(want))
    assert len(cases["partial_default"]["restored"]) == 254 and not any("cls" in n for n in cases["partial_default"]["restored"])
