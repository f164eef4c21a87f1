"""Pins oracle/picnn_np.py and oracle/gd_grad_np.py against tests/golden/picnn_tfshim.npz: the outputs of the
REFERENCE'S OWN graph code (multi-label-cls/icnn_ebundle.py Model.__init__/f, multi-label-cls/icnn-back.py
Model.__init__/f, RL/src/icnn.py Agent.negQ / Agent.bundle_entropy) executed unmodified on the TensorFlow /
tflearn stand-in oracle/tf_shim.py by oracle/gen_golden_tfshim.py.  CPU only; the golden file and the seeded
inputs travel, /root/reference is not read here."""
import os

import numpy as np
import pytest

from oracle import bundle_np, gd_grad_np, picnn_np
from oracle.gen_golden_tfshim import case_inputs


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "picnn_tfshim.npz"))


def close(a, b, what, rtol=1e-10):
    scale = max(float(np.abs(b).max()), 1e-30)
    err = float(np.abs(np.asarray(a, dtype=np.float64) - b).max())
    assert err <= rtol * scale + 1e-18, (what, err, scale)


@pytest.mark.parametrize("tag", ["ml_fg_c3", "ml_fg_bn"])
def test_energy_and_gradient_match_the_reference_graph(tag, gold):
    """E_ = Model.f(x, y) and dE_dy_ = tf.gradients(E_, y_) (multi-label-cls/icnn_ebundle.py:131,146,316-388);
    'ml_fg_bn' carries real batch-norm statistics on the u-path and non-zero biases on every biased layer."""
    c = case_inputs(tag)
    f, g = picnn_np.make_fg(c["p"], c["x"])(c["y"])
    close(f, gold[tag + "_f"], "f")
    close(g, gold[tag + "_g"], "g")
    # dE_entr_dy_ (:132-135): the entropy-regularised objective's gradient the bundle method's optimum zeroes
    close(g + np.log(c["y"]) - np.log1p(-c["y"]), gold[tag + "_g_entr"], "g_entr")


def test_batchnorm_fold_equals_the_reference_graph(gold):
    """The device path honours batch-norm by folding it into the consumer weights (workloads.fold_batchnorm):
    the folded, bn-free parameters must give the reference graph's values too."""
    from icnn_b200 import workloads
    c = case_inputs("ml_fg_bn")
    q = workloads.fold_batchnorm(c["p"])
    assert all(b is None for b in q.bn)
    f, g = picnn_np.make_fg(q, c["x"])(c["y"])
    close(f, gold["ml_fg_bn_f"], "f", rtol=1e-9)
    close(g, gold["ml_fg_bn_g"], "g", rtol=1e-9)


def test_rl_negq_and_affine_wrapper_match_the_reference_graph(gold):
    """Agent.negQ (leaky-ReLU, gate biases 1: RL/src/icnn.py:325-404) under the wrapper of Agent.bundle_entropy
    (:150-153: a = 2x - 1, grad *= 2)."""
    c = case_inputs("rl_fg_c4")
    f, g = picnn_np.make_fg(c["p"], c["x"], affine=True)(c["y"])
    close(f, gold["rl_fg_c4_f"], "negQ")
    close(g, gold["rl_fg_c4_g"], "grad")


def test_rl_entropy_regularised_objective_matches_the_reference_graph(gold):
    """func = _fg_entr of the RL agent's Adam argmin: negQ - entropy(act) and its action gradient
    (RL/src/icnn.py:60-63, entropy :455-458 -- tf.clip_by_value passes no gradient outside [1e-4, 1 - 1e-4]),
    including actions at the ends Agent.adam clips to (:211)."""
    from oracle import adam_np
    c = case_inputs("rl_fg_entr_c4")
    f, g = adam_np.make_fg_entr(c["p"], c["x"])(c["x"], c["y"])
    close(f, gold["rl_fg_entr_c4_f"], "negQ_entr")
    close(g, gold["rl_fg_entr_c4_g"], "act_grad_entr")


def test_rl_action_selection_end_to_end(gold, golden_dir):
    """Agent.bundle_entropy(func, obs) executed in full by the generator -- the reference's negQ graph inside the
    reference's RL solveBatch -- against the oracle pair (picnn_np + bundle_np), and against the solver golden
    'c4_rl' (same seeded rows, produced with picnn_np as fg): the two golden chains agree."""
    c = case_inputs("rl_act_c4")
    with np.errstate(all="ignore"):
        y = bundle_np.solve_batch(picnn_np.make_fg(c["p"], c["x"], affine=True), c["y"].copy(), nIter=5,
                                  variant="rl")[0]
    act = gold["rl_act_c4_act"]
    c4 = np.load(os.path.join(golden_dir, "c4_rl.npz"))
    assert str(c4["config"]) == "C4" and int(c4["nIter"]) == 5
    # f and grad of the two chains differ by float64 summation order (1e-16); the RL copy's Newton systems are
    # numerically singular on some samples (DESIGN.md section 4) and amplify that: measured median 1.8e-15,
    # 5 of 48 rows between 1e-9 and 5e-8
    for mine in (2.0 * y - 1.0, 2.0 * c4["x"][:act.shape[0]] - 1.0):
        err = np.abs(mine - act).max(axis=1)
        assert np.median(err) < 1e-12 and err.max() < 1e-6 and (err > 1e-9).mean() <= 0.15, np.sort(err)[-6:]


def test_callback_trace_of_the_reference_benchmark(gold):
    """multi-label-cls/ebundle-vs-gd.py:84-107 run by the generator with the reference's own pieces (Model graph as fg,
    lib/bundle_entropy.solveBatch, entr(), callback (t, es, x) -> mean(es - entr(x))): the oracle pair reproduces the
    plotted trace and y* -- the callback contract (a12: called with the batch's f and the live iterate before the
    per-sample loop, lib/bundle_entropy.py:208-209)."""
    c = case_inputs("trace_c3")
    seen, trace = [], []

    def cb(t, es, x):
        seen.append(t)
        trace.append(float(np.mean(es - picnn_np.entr(x))))
    with np.errstate(all="ignore"):
        y = bundle_np.solve_batch(picnn_np.make_fg(c["p"], c["x"]), c["y"].copy(), nIter=c["nIter"], callback=cb)[0]
    assert seen == list(gold["trace_c3_iters"])
    np.testing.assert_allclose(trace, gold["trace_c3_f_minus_H"], rtol=0, atol=1e-9)
    assert np.abs(y - gold["trace_c3_yN"]).max() < 1e-9
    assert trace[-1] < trace[0]                              # the bundle method descends the entropy-regularised objective


GRAD_KEYS = {"u%d__W": ("x", "dWu"), "u%d__b": ("x", "dbu"), "z%d_zu_u__W": ("x", "dWzu"), "z%d_zu_u__b": ("x", "dbzu"),
             "z%d_yu_u__W": ("x", "dWyu"), "z%d_yu_u__b": ("x", "dbyu"), "z%d_zu_proj__W": ("g", "dWz"),
             "z%d_yu__W": ("g", "dWy")}


@pytest.mark.parametrize("tag", ["gd_c3", "gdgrad_small"])
def test_unrolled_gd_and_training_gradient_match_the_reference_graph(tag, gold):
    """yn_, energies_, mse_ and opt.compute_gradients(mse_, theta_) of the back-optimisation script
    (multi-label-cls/icnn-back.py:116-139): the momentum-GD recurrence and TensorFlow's double backprop through
    tf.gradients(Ei_, yi_), here through the reference's own unrolled graph."""
    c = case_inputs(tag)
    p, x, y0, tY = c["p"], c["x"], c["y"], c["trueY"]
    yN, fN = picnn_np.momentum_gd(picnn_np.make_fg(p, x), y0, c["nIter"], c["lr"], c["momentum"])
    close(yN, gold[tag + "_yN"], "yN")
    close(fN, gold[tag + "_energies"], "energies")
    assert abs(float(((yN - tY) ** 2).mean()) - float(gold[tag + "_mse"])) < 1e-13
    y2, gr = gd_grad_np.gd_backward(p, picnn_np.gates(p, x), y0, c["nIter"], c["lr"], c["momentum"],
                                    lambda y: 2.0 * (y - tY) / y.size)
    close(y2, gold[tag + "_yN"], "yN (gd_backward)")
    xg = gd_grad_np.xpath_backward(p, x, gr["dcy"], gr["dcz"])
    theta = [str(t) for t in gold[tag + "_theta"]]
    # tf.trainable_variables() in creation order: u-path first, then per z-layer zu_u, zu_proj, yu_u, yu, u
    assert theta[:3] == ["u0__W", "u0__b", "u0__bn__beta"] or theta[:2] == ["u0__W", "u0__b"]
    assert len(theta) == 2 * p.L + 2 * (p.L - 1) + 5 * (p.L + 1) + 3 * p.L
    checked = 0
    for l in range(p.L + 1):
        for pat, (src, key) in GRAD_KEYS.items():
            name = "%s_grad_%s" % (tag, pat % l)
            if name not in gold.files:
                continue
            mine = (xg if src == "x" else gr)[key]
            assert l < len(mine) and mine[l] is not None, name
            close(mine[l], gold[name], name, rtol=1e-9)
            checked += 1
        # the additive gate d_l = fc(prevU) does not enter dE/dy: TensorFlow returns zeros / None for its parameters
        for nm in ("%s_grad_z%d_u__W" % (tag, l), "%s_grad_z%d_u__b" % (tag, l)):
            if nm in gold.files:
                assert not np.any(gold[nm])
    assert checked >= (8 * p.L + 3 if tag == "gdgrad_small" else 8)


@pytest.mark.parametrize("tag", ["conv_small", "conv_olivetti"])
def test_conv_picnn_helper_matches_the_reference_graph(tag, gold):
    """tests/conv_picnn.py -- the user-side ``fg`` the GPU callback-mode test drives K2 with at the Olivetti dims
    (SURVEY.md 8d config 2) -- against E_ / dE_dy_ of the reference's own convolutional Model.__init__ / Model.f
    (completion/icnn_ebundle.py:105-161,337-452) executed on oracle/tf_shim.py: same wiring (u-path convs 32x8/4,
    64x4/2, 64x3/1 + FC 512, 1; y_red path; gates), 'SAME' padding, NHWC flatten order of the dense layers."""
    from oracle.gen_golden_tfshim import conv_case
    net, x, y = conv_case(tag)
    f, g = net.make_fg(x)(y)
    close(f, gold[tag + "_f"], "E_")
    close(g, gold[tag + "_g"], "dE_dy_")


def test_committed_goldens_regenerate_from_the_reference(gold):
    """The committed vectors ARE what the reference's code produces on the stand-in, bit for bit: every array has
    the SHA-256 that oracle/gen_reference_digests.py recorded from oracle/gen_golden_tfshim.generate()."""
    from oracle import gen_reference_digests
    want = gen_reference_digests.load()["picnn_tfshim.npz"]
    assert sorted(want) == sorted(gold.files)
    for k in gold.files:
        assert gen_reference_digests.array_digest(gold[k]) == want[k], k
