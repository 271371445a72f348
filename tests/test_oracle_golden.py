"""Pins oracle/block_oracle.py (the CPU restatement) against outputs of the UNMODIFIED reference:
committed golden vectors (tests/golden, made by oracle/make_golden.py)."""
import pytest
import torch

from oracle import block_oracle as bo
from tests.util import golden_loss_cases, nerr, run_oracle_block

CASES = ["dense_train", "dense_eval", "dense_train_u0", "dense_train_T5", "dense_train_F16", "dense_train_F4",
         "dense_unnormed", "permuted_train", "class_major_train", "shuffled_train", "sparse_train", "sparse_eval",
         "duplicates_train"]


@pytest.mark.parametrize("name", CASES)
def test_restatement_matches_reference_fp64(golden_block_cases, name):
    case = golden_block_cases[name]
    outs, gin, gparam, buffers = run_oracle_block(bo, case, torch.float64)
    for k in outs:
        assert nerr(outs[k], case["out_f64"][k]) < 1e-10, k
    for k in gin:
        assert nerr(gin[k], case["gin_f64"][k]) < 1e-8, k
    assert set(gparam) == set(case["gparam_f64"])
    scale = max(v.abs().max().item() for v in case["gparam_f64"].values())
    for k, g in gparam.items():
        ref = case["gparam_f64"][k]
        # analytically-zero gradients (biases feeding a train-mode BN) are noise in the reference too
        assert (g - ref).abs().max().item() <= 1e-8 * max(scale, ref.abs().max().item()), k
    if case["training"] and case.get("normed", True):
        for k, v in case["buffers_f64"].items():
            if k.endswith("num_batches_tracked"):
                assert int(buffers[k]) == int(v), k
            else:
                assert nerr(buffers[k], v) < 1e-10, k


def test_double_norm_is_pinned(golden_block_cases):
    """edge BatchNorm gets two running-stat updates per forward, node BatchNorms one (SURVEY 0.2)."""
    b = golden_block_cases["dense_train"]["buffers_f64"]
    assert int(b["edge_model.norm.num_batches_tracked"]) == 2
    assert int(b["s_model.norm.num_batches_tracked"]) == 1
    assert int(b["t_model.norm.num_batches_tracked"]) == 1


def test_gnn_shipped_weights_fp64(golden_gnn_case):
    case = golden_gnn_case
    sd = bo.cast_state(case["state"], torch.float64)      # the reference's shipped checkpoint, stored with its outputs
    for training in (True, False):
        x_s, x_t, x_e, u = bo.gnn_forward(sd, 3, case["edge_index"], case["x_s"], case["x_t"], case["x_e"], case["u"],
                                          training=training, buffers={})
        time = bo.edge_prediction(sd, x_e, scale=42 / 12)
        gold = case[("train_" if training else "eval_") + "f64"]
        assert nerr(x_e, gold["x_e"]) < 1e-9
        assert nerr(x_s, gold["x_s"]) < 1e-9
        assert nerr(x_t, gold["x_t"]) < 1e-9
        assert nerr(u, gold["u"]) < 1e-9
        assert nerr(time, gold["time"]) < 1e-9


def test_integer_time_definition():
    time = torch.tensor([3.0, 5.0, 9.0, 2.9])
    hours = torch.tensor([2.0, 6.0])
    tgt = torch.tensor([0, 0, 1, 1])
    visits, t_int = bo.integer_times(time, hours, tgt)
    assert visits.tolist() == [2.0, 2.0, 2.0, 0.0]      # 1.5 -> 2 and 2.5 -> 2: round-half-even
    assert t_int.tolist() == [4.0, 4.0, 12.0, 0.0]


# ---------------------------------------------------------------------------------------------
# training loss (SURVEY.md section 8f row N1): oracle/loss_oracle.py against the unmodified reference
# ---------------------------------------------------------------------------------------------
def test_loss_oracle_matches_reference():
    from oracle import loss_oracle as lo
    cases = golden_loss_cases()
    assert len(cases) == 8
    for c in cases:
        S, T = c["S"], c["T"]
        tol = 1e-10 if c["time"].dtype == torch.float64 else 2e-5
        time = c["time"].clone().requires_grad_(True)
        r = lo.loss_terms(time, c["noise"], c["class_info"], bo.complete_bipartite(S, T), S, T, nfields=c["nfields"],
                          total_time=c["total_time"], wutils=c["wutils"], wvar=c["wvar"])
        r["loss"].backward()

        def close(a, b, what):
            err = (a.detach().double() - b.double()).abs().max().item() / max(b.double().abs().max().item(), 1e-30)
            assert err < tol, (what, S, T, str(time.dtype), err)

        close(r["loss"], c["loss"], "loss")
        close(r["totutils"], c["totutils"], "totutils")
        close(r["n_prime"], c["n_prime"], "n_prime")
        close(r["fiber_time"], c["fiber_time"], "fiber_time")
        close(r["time"], c["time2"], "time")
        close(r["variance"], c["variance"], "variance")
        close(time.grad, c["g_time"], "grad time")


def test_oracle_training_step_reproduces_reference_trajectory():
    """The oracle port of the whole step (block_oracle.gnn_forward + loss_oracle + torch Adam) replays the trajectory of the
    UNMODIFIED reference src/train.py run as __main__ (tests/golden/train_steps.pt, oracle/make_golden_train.py)."""
    import os
    from oracle import loss_oracle as lo
    d = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "train_steps.pt"))
    c = d["config"]
    state = {k: v.clone() for k, v in d["init_state"].items()}
    params = {k: v.requires_grad_(True) for k, v in state.items() if v.is_floating_point() and "running" not in k}
    opt = torch.optim.Adam(list(params.values()), lr=c["lr"])
    bufs = {}
    S, T = c["NFIBERS"], c["NCLASSES"]
    losses, utils = [], []
    for k in range(d["compare_epochs"]):
        opt.zero_grad()
        full = dict(state)
        full.update(bufs)
        xs, xt, xe, u = bo.gnn_forward(full, c["B"], d["edge_index"], d["x_s"], d["class_info"], d["x_e"], d["x_u"],
                                       training=True, buffers=bufs)
        tm = bo.edge_prediction(full, xe, c["TOTAL_TIME"] / T).squeeze(-1)
        out = lo.loss_terms(tm, d["noise"][k], d["class_info"], d["edge_index"], S, T, c["NFIELDS"], c["TOTAL_TIME"], c["wutils"],
                            c["wvar"], c["pclass"], c["pfiber"], float(d["sharps"][k]))
        out["loss"].backward()
        opt.step()
        losses.append(float(out["loss"]))
        utils.append(float(out["totutils"]))
    _check_trajectory(d, losses, utils, {k: v.detach() for k, v in params.items()})


def _check_trajectory(d, losses, utils, params_now):
    """Compares the first d["compare_epochs"] epochs.  Two fp32 executions of this loop cannot agree to rounding: Adam's
    first steps are sign-like (lr * g / |g|), and the raw inputs of src/train.py:88-91 (fibre index 0..K-1, galaxy counts
    up to 96 300 straight into the encoders) leave block 0 with gradient entries that are fp32 noise (measured: the
    reference and the CPU port disagree on the SIGN of a third of mpb.0.global_model.0.weight.grad at the very first
    step), so such weights walk +-lr per epoch in either run; once the sharpness passes ~10 the loss (a min over classes of
    a near-floor function) jumps by 5 % between the two.  Bounds over the compared epochs: loss / utility curves within
    1 % / 2 % of their range, every weight within the 2 * lr * epochs two such walks can separate, and the weights as a
    whole (relative L2) within 2 % (the CPU port itself sits at 0.9 %)."""
    c, n = d["config"], d["compare_epochs"]
    ref_l, ref_u = d["losses"].tolist()[:n], d["utilities"].tolist()[:n]
    scale_l, scale_u = max(abs(x) for x in ref_l), max(ref_u)
    for k, (a, b) in enumerate(zip(losses[:n], ref_l)):
        assert abs(a - b) <= 1e-2 * scale_l, ("loss", k, a, b)
    for k, (a, b) in enumerate(zip(utils[:n], ref_u)):
        assert abs(a - b) <= 2e-2 * scale_u, ("utility", k, a, b)
    num = den = 0.0
    for k, v in params_now.items():
        r = d["params_after_compare"][k].double()
        diff = (v.double().cpu() - r).abs().max().item()
        assert diff <= 2 * c["lr"] * n, (k, diff)
        num += float(((v.double().cpu() - r) ** 2).sum())
        den += float((r ** 2).sum())
    rel = (num / den) ** 0.5
    worst_l = max(abs(a - b) for a, b in zip(losses[:n], ref_l)) / scale_l
    print("trajectory vs the unmodified reference over %d epochs: loss curve within %.2e of its range, weights relative L2 %.2e"
          % (n, worst_l, rel))
    assert rel <= 2e-2, rel
