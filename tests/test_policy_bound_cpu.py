"""CPU tests of the propagated policy-forward error bound (tests/policy_bound.py): it holds for emulations of every kernel's
operand arithmetic (soundness), it is tight enough that planted layout and precision defects of the tcgen05 pipeline exceed it
(discrimination), and its arithmetic equals a direct float64 computation on a toy net."""
import numpy as np
import pytest

import policy_bound as pb

DEFECTS = ("lo_dropped", "bias_row", "w2_halves", "head_split", "mean_f32")
# Defects that the network itself hides, so that no sound bound on the outputs can see them: with every weight x 1e-3 an error
# is attenuated 1e3-fold per layer while float16's subnormal floor (2^-25 absolute per lo part, which the kernel really has
# there) does not shrink with it.
HIDDEN = {("near_zero", "mean_f32"), ("near_zero", "lo_dropped")}


@pytest.fixture(scope="module", params=[20, 17])
def sets(request, golden_dir):
    return request.param, pb.weight_sets(golden_dir, request.param), pb.input_sets(request.param)


def test_bound_holds_for_every_emulated_forward(sets):
    D, ws, ins = sets
    for wn, sd in ws.items():
        for impl in ("fp32", "tensor", "tensor_fast"):
            worst = 0.0
            for iname, (x, st) in ins.items():
                m, v, bm, bv = pb.forward_with_bound(sd, x, impl, st)
                assert np.isfinite(bm).all() and np.isfinite(bv).all()
                em, ev = pb.emulate(sd, x, impl, st)
                r = pb.max_ratio(em, ev, m, v, bm, bv)
                assert max(r) <= 1.0, (D, wn, impl, iname, r)
                worst = max(worst, *r)
            print(f"soundness obs_dim={D} {wn:15s} {impl:12s} max(err/bound) = {worst:.3g}")


def test_planted_defects_exceed_the_tensor_bound(sets):
    D, ws, ins = sets
    for wn, sd in ws.items():
        for defect in DEFECTS:
            worst = 0.0
            for iname, (x, st) in ins.items():
                if defect == "mean_f32" and st is None:
                    continue
                m, v, bm, bv = pb.forward_with_bound(sd, x, "tensor", st)
                em, ev = pb.emulate(sd, x, "tensor", st, defect=defect)
                worst = max(worst, *pb.max_ratio(em, ev, m, v, bm, bv))
            print(f"discrimination obs_dim={D} {wn:15s} {defect:10s} max(err/bound) = {worst:.3g}")
            if (wn, defect) not in HIDDEN:
                assert worst > 1.0, (D, wn, defect, worst)


def test_defect_hidden_by_the_net_is_caught_where_it_is_planted(golden_dir):
    """The exemptions above are properties of the weights, not of the bound: the same defects are far outside the bound on the
    shipped weights, and with a float32 mean the normalised input itself is off by far more than e_0."""
    D = 20
    x, st = pb.input_sets(D)["vecnorm"]
    v, e0 = pb.normalised_input(x, "tensor", st)
    bad = pb._norm_f32(x, st, 1e-8, 10.0, mean_lo=False)
    good = pb._norm_f32(x, st, 1e-8, 10.0)
    assert (np.abs(good - v) <= e0).all()
    assert (np.abs(bad - v) / e0).max() > 1e3


def test_bound_arithmetic_on_a_toy_net():
    """Three 2-unit tanh layers and a 1-output head, bound recomputed by hand in float64."""
    rng = np.random.default_rng(0)
    Ws = [rng.standard_normal((2, 2)) for _ in range(3)]
    bs = [rng.standard_normal(2) for _ in range(3)]
    Wh, bh = rng.standard_normal((1, 2)), rng.standard_normal(1)
    x = rng.standard_normal((5, 2))
    c = pb.CONST["tensor"]
    ks = (7, 9, 11)
    out, bo = pb._net_bound(list(zip(Ws, bs)), (Wh, bh), x, np.zeros_like(x), c, ks)
    for r in range(5):
        h, e = x[r].copy(), np.zeros(2)
        for (W, b), K in zip(zip(Ws, bs), ks):
            z = np.array([sum(W[j, k] * h[k] for k in range(2)) + b[j] for j in range(2)])
            dz = np.zeros(2)
            for j in range(2):
                dz[j] = sum(abs(W[j, k]) * e[k] for k in range(2))
                dz[j] += (c["u_op"] + K * c["u_acc"]) * (sum(abs(W[j, k]) * (abs(h[k]) + e[k]) for k in range(2)) + abs(b[j]))
                dz[j] += c["f"] * (abs(W[j, 0]) + abs(W[j, 1]) + abs(h[0]) + e[0] + abs(h[1]) + e[1] + 1)
            L = np.array([1 / np.cosh(max(abs(z[j]) - dz[j], 0.0)) ** 2 for j in range(2)])
            h, e = np.tanh(z), np.minimum(2.0, L * dz) + c["eps_tanh"]
        want_out = Wh[0] @ h + bh[0]
        want_b = abs(Wh[0]) @ e + pb.HEAD_U * (abs(Wh[0]) @ (abs(h) + e) + abs(bh[0]))
        assert abs(out[r, 0] - want_out) < 1e-12 and abs(bo[r, 0] - want_b) <= 1e-12 * want_b
