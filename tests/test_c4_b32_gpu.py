"""The BENCHED workload (BASELINE config 4, B = 32 dialogs) against the committed oracle fixture
tests/golden/c4_b32__mn-att-ques-im-hist__disc.npz (fp64 oracle, batched structure, same init / batch seeds as
bench.py) — every math mode, option stream overlapped (the benched schedule), at the benched size:

  * training step: loss, every parameter segment's gradient (l2 norm + a strided sample of the flat gradient)
  * eval step: scores, the full (320,100) rank matrix -> `rank_agreement` (fraction of identical entries), top-1
    agreement, and the R@1/5/10 / mean-rank / MRR deltas through processRanks (utils.lua:131-160)

north_star asks for bit-exact ranks; fp32 mode delivers that up to ties of fp32 rounding, the tensor-core modes are
held to measured agreement floors (DESIGN.md §7) and the measured numbers are attached to each test's report as the
property `c4_b32_parity` (visible with `--junitxml`)."""
import json
import os

import numpy as np
import pytest

from helpers import full_params, seg_slices
from visdial_b200 import VD_MATH_F16, VD_MATH_FP32, VD_MATH_TF32, Batch, Engine, init_parameters
from visdial_b200.synthetic import make_batch
from visdial_b200.utils import processRanks

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "c4_b32__mn-att-ques-im-hist__disc.npz")

# stated tolerances per mode: (loss rel, gradient-sample abs error / segment abs-max, segment-norm rel, score abs,
#                              rank agreement floor, top-1 agreement floor, |delta MRR| ceiling)
TOL = {
    VD_MATH_FP32: dict(loss=2e-5, grad=2e-4, norm=2e-4, score=2e-4, agree=0.995, top1=0.996, mrr=2e-3),
    VD_MATH_TF32: dict(loss=3e-3, grad=2e-2, norm=1e-2, score=2e-2, agree=0.80, top1=0.97, mrr=1e-2),
    VD_MATH_F16: dict(loss=3e-3, grad=2e-2, norm=1e-2, score=2e-2, agree=0.80, top1=0.97, mrr=1e-2),
}
NAMES = {VD_MATH_FP32: "fp32", VD_MATH_TF32: "tf32", VD_MATH_F16: "f16"}


@pytest.fixture(scope="module")
def fixture():
    return np.load(FIX)


def _setup(fx, mode):
    p = full_params("mn-att-ques-im-hist", "disc")
    flat = init_parameters(p, seed=int(fx["init_seed"]))
    nb = make_batch(p, int(fx["B"]), seed=int(fx["batch_seed"]))
    eng = Engine(p)
    eng.set_math_mode(mode)
    eng.set_parameters(flat)
    return p, nb, eng


@pytest.mark.parametrize("mode", [VD_MATH_FP32, VD_MATH_TF32, VD_MATH_F16])
def test_train_step_matches_fixture(fixture, mode, record_property):
    fx, tol = fixture, TOL[mode]
    p, nb, eng = _setup(fx, mode)
    eng.set_training(1)
    eng.set_dropout_seed(int(fx["drop_seed"]), int(fx["drop_iter"]))
    eng.zero_grad()
    loss = eng.forward_backward(Batch(nb))
    g = eng.get_gradients().astype(np.float64)
    eng.close()
    ref_loss = float(fx["train_loss"])
    assert abs(loss - ref_loss) < tol["loss"] * abs(ref_loss), (loss, ref_loss)
    stride = int(fx["stride"])
    sample, ref = g[::stride], fx["grad_sample"]
    idx = np.arange(0, g.size, stride)
    sl = seg_slices(p)
    worst, worst_norm, rec = 0.0, 0.0, {}
    for name, amax, nrm in zip(fx["seg_names"], fx["seg_absmax"], fx["seg_norm"]):
        s = sl[str(name)]
        if amax < 1e-9:                      # mathematically zero gradient (softmax shift invariance)
            continue
        m = (idx >= s.start) & (idx < s.stop)
        e = float(np.abs(sample[m] - ref[m]).max() / amax) if m.any() else 0.0
        en = abs(float(np.sqrt((g[s] ** 2).sum())) - nrm) / nrm
        rec[str(name)] = [e, en]
        worst, worst_norm = max(worst, e), max(worst_norm, en)
    record_property("c4_b32_parity", json.dumps({"train_" + NAMES[mode]: {
        "loss": loss, "ref_loss": ref_loss, "worst_grad_err_over_segmax": worst, "worst_segnorm_rel": worst_norm,
        "per_segment": rec}}, sort_keys=True))
    assert worst < tol["grad"], (worst, rec)
    assert worst_norm < tol["norm"], (worst_norm, rec)


@pytest.mark.parametrize("mode", [VD_MATH_FP32, VD_MATH_TF32, VD_MATH_F16])
def test_eval_ranks_match_fixture(fixture, mode, record_property):
    fx, tol = fixture, TOL[mode]
    p, nb, eng = _setup(fx, mode)
    eng.set_training(0)
    b = Batch(nb)
    eng.encoder_forward(b)
    scores = eng.decoder_forward(b).numpy().astype(np.float64)
    ranks = eng.retrieve(Batch(nb), use_gt=False)
    gt_ranks = eng.retrieve(Batch(nb), use_gt=True)
    eng.close()
    ref_sc, ref_r = fx["eval_scores"], fx["eval_ranks"]
    dev = float(np.abs(scores - ref_sc).max())
    agree = float((ranks == ref_r).mean())
    top1 = float(((ranks == 1).argmax(1) == (ref_r == 1).argmax(1)).mean())
    # how far do the entries that differ move?  (a flip between two near-tied options moves both by one place)
    moved = np.abs(ranks.astype(np.int64) - ref_r)
    got_m = processRanks(gt_ranks.reshape(-1), verbose=False)
    ref_m = dict(zip(("r@1", "r@5", "r@10", "medianR", "meanR", "meanRR"), fx["metrics"]))
    delta = {k: float(got_m[k] - ref_m[k]) for k in ("r@1", "r@5", "r@10", "meanR", "meanRR")}
    assert np.array_equal(np.sort(ranks, 1), np.tile(np.arange(1, 101), (ranks.shape[0], 1)))     # a permutation per row
    record_property("c4_b32_parity", json.dumps({"eval_" + NAMES[mode]: {
        "max_score_dev": dev, "rank_agreement": agree, "top1_agreement": top1, "max_rank_move": int(moved.max()),
        "mean_rank_move": float(moved.mean()), "gt_rank_agreement": float((gt_ranks.reshape(-1) == fx["gt_ranks"]).mean()),
        "metric_delta": delta, "score_absmax": float(np.abs(ref_sc).max())}}, sort_keys=True))
    assert dev < tol["score"] * max(1.0, float(np.abs(ref_sc).max())), dev
    assert agree >= tol["agree"], agree
    assert top1 >= tol["top1"], top1
    assert abs(delta["meanRR"]) <= tol["mrr"], delta
