"""The numpy restatement (oracle/bundle_np.py) against vectors produced by the UNMODIFIED
reference modules (oracle/gen_golden.py -> tests/golden/*.npz).  CPU only."""
import glob
import os

import numpy as np
import pytest

from oracle import bundle_np, gen_reference_digests, picnn_np, synth
from oracle.gen_golden import inputs_digest

CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(
    os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
    if os.path.basename(p)[:-4] not in ("adam", "argmin_grad", "gd_grad", "picnn_tfshim"))   # those have their own tests


def _run(gold):
    cfgname = str(gold["config"])
    cfg = synth.CONFIGS[cfgname]
    p, x, y0 = synth.make_inputs(cfgname, B=int(gold["B"]))
    assert inputs_digest(p, x, y0) == str(gold["digest"]), "synthetic input generator drifted"
    fg = picnn_np.make_fg(p, x, affine=cfg["affine"])
    with np.errstate(all="ignore"):
        return bundle_np.solve_batch(fg, y0.copy(), nIter=int(gold["nIter"]),
                                     variant=str(gold["variant"]),
                                     solver=str(gold["solver"]) or "pc")


@pytest.mark.parametrize("case", CASES)
def test_restatement_matches_reference(case, golden_dir):
    gold = np.load(os.path.join(golden_dir, case + ".npz"))
    if case in ("c2_pc", "c5_pc"):
        pytest.importorskip("numpy")  # slow-ish (~10 s) but kept: the big-n pins
    x, A, b, lam, xs, nIters = _run(gold)
    counts = np.array([len(a) for a in A])
    np.testing.assert_array_equal(counts, gold["counts"])
    np.testing.assert_array_equal(np.array(nIters), gold["nIters"])
    # same algorithm, same arithmetic up to BLAS summation order (dense diag vs vector scale)
    np.testing.assert_allclose(x, gold["x"], rtol=0, atol=1e-9)
    for u in range(len(A)):
        k = counts[u]
        if k:
            np.testing.assert_allclose(lam[u], gold["lam"][u, :k], rtol=0, atol=1e-8)
            np.testing.assert_allclose(np.array(b[u]), gold["b"][u, :k], rtol=0, atol=1e-9)
            if "A" in gold.files:
                np.testing.assert_allclose(np.array(A[u]), gold["A"][u, :k], rtol=0, atol=1e-9)
                np.testing.assert_allclose(np.array(xs[u]), gold["xs"][u, :k], rtol=0, atol=1e-9)


def test_invariants_on_golden(golden_dir):
    """Known-answer invariants derived from the reference code (SURVEY.md section 8c)."""
    for case in ("c1_dual", "c3_dual", "t_dual"):
        gold = np.load(os.path.join(golden_dir, case + ".npz"))
        cnt = gold["counts"]
        for u in range(len(cnt)):
            k = cnt[u]
            lam = gold["lam"][u, :k]
            assert np.all(lam > 0) and abs(lam.sum() - 1.0) < 1e-9
            if int(gold["nIters"][u]) == int(gold["nIter"]):   # not rank-stopped: x = sigma(-G^T lam)
                y = 1.0 / (1.0 + np.exp(gold["A"][u, :k].T.dot(lam)))
                np.testing.assert_allclose(y, gold["x"][u], atol=1e-12)
    gold = np.load(os.path.join(golden_dir, "c4_rl.npz"))
    assert gold["x"].min() >= 0.03 and gold["x"].max() <= 0.97


def test_pc_and_dual_agree_on_subproblem():
    """pdipm_pc and a converged dual Newton solve the same strictly convex subproblem."""
    rs = np.random.RandomState(0)
    for k, n in [(1, 8), (3, 8), (5, 40), (9, 159)]:
        G = rs.randn(k, n)
        h = rs.randn(k)
        with np.errstate(all="ignore"):
            y, z = bundle_np.pdipm_pc(G, h)
            lam = bundle_np.proj_newton_logistic(G, h, line_search=True)
        yd = 1.0 / (1.0 + np.exp(G.T.dot(lam)))
        np.testing.assert_allclose(y, yd, atol=2e-7)
        np.testing.assert_allclose(z, lam, atol=2e-6)
        # pdipm_boyd (20 damped iterations) does not reach the optimum on generic inputs; it is
        # pinned by the reference-generated c1_boyd golden case instead.


def test_argmin_grad_restatement_matches_reference_bodies(golden_dir):
    """oracle/argmin_grad_np.py vs crossEntrGrad / mseGrad exec'd from the reference sources
    (oracle/gen_golden_grad.py)."""
    from oracle import argmin_grad_np
    gold = np.load(os.path.join(golden_dir, "argmin_grad.npz"))
    for tag, cfgname, B, nIter in (("c1", "C1", 32, 5), ("c3", "C3", 12, 10)):
        p, x, y0 = synth.make_inputs(cfgname, B=B)
        with np.errstate(all="ignore"):
            o = bundle_np.solve_batch(picnn_np.make_fg(p, x), y0.copy(), nIter=nIter)
        np.testing.assert_array_equal(np.array([len(a) for a in o[1]]), gold[tag + "_counts"])
        for loss in ("xent", "mse"):
            for j in range(B):
                with np.errstate(all="ignore"):
                    cy, clam, ct = argmin_grad_np.argmin_grad(o[0][j], gold[tag + "_trueY"][j], np.array(o[1][j]), loss)
                ref = gold["%s_%s_cy" % (tag, loss)][j]
                np.testing.assert_allclose(cy, ref, atol=1e-7 * max(1.0, np.abs(ref).max()))
                np.testing.assert_allclose(clam, gold["%s_%s_clam" % (tag, loss)][j, :len(clam)],
                                           atol=1e-7 * max(1.0, np.abs(clam).max()))


def test_train_step_pairs_match_the_reference_method(golden_dir):
    """oracle/argmin_grad_np.train_step_pairs vs the (fd_ys, fd_vs, fd_cs) feeds built by the reference's own
    Model.train_step_fd (multi-label-cls/icnn_ebundle.py:296-314 with crossEntrGrad,
    completion/icnn_ebundle.py:315-335 with mseGrad), exec'd unmodified by oracle/gen_golden_grad.py."""
    from oracle import argmin_grad_np
    gold = np.load(os.path.join(golden_dir, "argmin_grad.npz"))
    for tag, cfgname, B, nIter in (("c1", "C1", 32, 5), ("c3", "C3", 12, 10)):
        p, x, y0 = synth.make_inputs(cfgname, B=B)
        with np.errstate(all="ignore"):
            yN, G, h, lam, ys, _ = bundle_np.solve_batch(picnn_np.make_fg(p, x), y0.copy(), nIter=nIter)
        for loss in ("xent", "mse"):
            with np.errstate(all="ignore"):
                fys, fvs, fcs = argmin_grad_np.train_step_pairs(yN, gold[tag + "_trueY"], G, ys, lam, loss)
            rys, rvs, rcs = (gold["%s_%s_fd_%s" % (tag, loss, k)] for k in ("ys", "vs", "cs"))
            assert fys.shape == rys.shape and fvs.shape == rvs.shape and fcs.shape == rcs.shape
            np.testing.assert_allclose(fys, rys, rtol=0, atol=1e-9)
            scale = max(1.0, np.abs(rvs).max(), np.abs(rcs).max())
            np.testing.assert_allclose(fvs, rvs, rtol=0, atol=1e-7 * scale)
            np.testing.assert_allclose(fcs, rcs, rtol=0, atol=1e-7 * scale)


def test_adam_restatement_matches_reference_body(golden_dir):
    """oracle/adam_np.py vs Agent.adam exec'd from RL/src/icnn.py (oracle/gen_golden_adam.py)."""
    from oracle import adam_np
    gold = np.load(os.path.join(golden_dir, "adam.npz"))
    p, x, _ = synth.make_inputs("C4", B=96)
    best, its = adam_np.adam(adam_np.make_fg_entr(p, x), x, p.n)
    assert its == int(gold["c4_iters"])
    np.testing.assert_allclose(best, gold["c4_act_best"], atol=1e-12)


@pytest.mark.parametrize("case", gen_reference_digests.SOLVER_CASES)
def test_committed_goldens_regenerate_from_the_reference(case, golden_dir):
    """The goldens are the reference's output, bit for bit: every array of the committed file has the SHA-256 that
    oracle/gen_reference_digests.py recorded from the unmodified reference module run on the same seeded case."""
    want = gen_reference_digests.load()[case + ".npz"]
    gold = np.load(os.path.join(golden_dir, case + ".npz"))
    assert sorted(want) == sorted(gold.files)
    for k in gold.files:
        assert gen_reference_digests.array_digest(gold[k]) == want[k], k
