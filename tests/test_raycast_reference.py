"""CPU tests of the float64 ray-cast reference (tests/raycast_reference.py) on analytic fields: a crossing known in
closed form, a bracket holding two roots (the first must win), a ray that starts inside, and misses."""
import math

import torch

from raycast_reference import cast64, first_inside, in_box64, refine

AABB = torch.tensor([[-3.0, -3.0, -3.0], [3.0, 3.0, 3.0]])
STEP = 0.1
S = 64


def _samples(o, d):
    """The marcher's fp32 depths k * STEP from t_min = 0, its fp32 points and box test."""
    t = (torch.arange(S, dtype=torch.float32) * torch.tensor(STEP, dtype=torch.float32)).expand(o.shape[0], S)
    p = o.float()[:, None, :] + d.float()[:, None, :] * t[..., None]
    inbox = ((p >= AABB[0]) & (p <= AABB[1])).all(dim=-1)
    return t, p, inbox


def _rays(o, d):
    return torch.tensor(o, dtype=torch.float32), torch.tensor(d, dtype=torch.float32)


def test_crossing_in_closed_form():
    """alpha = (1 + tanh(x)) / 2 along +x: the level set is the plane x = atanh(2 level - 1)."""
    level = 0.3
    x_star = math.atanh(2 * level - 1)
    o, d = _rays([[-2.0, 0.1, 0.2], [-2.5, -1.0, 0.5]], [[1.0, 0.0, 0.0], [0.8, 0.1, -0.1]])
    t, p, inbox = _samples(o, d)
    res = cast64(o, d, t, p, inbox, lambda p: 0.5 * (1.0 + torch.tanh(p[:, 0])), AABB, level, P=15)
    t_exact = (x_star - o[:, 0].double()) / d[:, 0].double()
    k_exact = torch.ceil(t_exact / STEP).long()
    assert torch.equal(res["k"], k_exact)
    assert bool((res["lo"] < t_exact).all() and (t_exact <= res["hi"]).all())
    assert bool(((res["hi"] - res["lo"]) <= 1.001 * STEP * 2.0 ** -20).all())     # fp32 sample spacing: STEP to 1e-6
    assert float((res["t_star"] - t_exact).abs().max()) <= 1e-12


def test_the_first_of_two_roots_in_a_bracket_wins():
    """Inside on [a, a + 0.014] and on [b, inf) with t_{k-1} < a < b < t_k: bisection of [t_{k-1}, t_k] would settle on
    b, the first-crossing subdivision finds a."""
    level = 0.5
    a, b = 1.213, 1.271                        # both in (1.2, 1.3): the bracket of sample 13 on a ray from x = 0

    def alpha(p):
        x = p[:, 0]
        return (((x >= a) & (x <= a + 0.014)) | (x >= b)).double() * 0.9

    for P in (15, 7):
        o, d = _rays([[0.0, 0.0, 0.0]], [[1.0, 0.0, 0.0]])
        t, p, inbox = _samples(o, d)
        res = cast64(o, d, t, p, inbox, alpha, AABB, level, P=P)
        assert int(res["k"][0]) == 13
        assert abs(float(res["t_star"][0]) - a) <= 1e-12, (P, float(res["t_star"][0]))
        assert float(res["lo"][0]) < a <= float(res["hi"][0])


def test_a_ray_starting_inside_reports_its_first_sample():
    o, d = _rays([[0.5, 0.0, 0.0], [-1.0, 2.0, 0.0]], [[1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    t, p, inbox = _samples(o, d)
    res = cast64(o, d, t, p, inbox, lambda p: torch.full((p.shape[0],), 0.7, dtype=torch.float64), AABB, 0.5, P=15)
    assert res["k"].tolist() == [0, 0]
    assert torch.equal(res["t_star"], t[:, 0].double()) and torch.equal(res["hi"], res["lo"])


def test_misses():
    """Below the level everywhere; and a field above the level everywhere but a ray that never enters the box."""
    o, d = _rays([[0.0, 0.0, 0.0], [0.0, 0.0, 4.0]], [[1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    t, p, inbox = _samples(o, d)
    res = cast64(o, d, t, p, inbox, lambda p: torch.full((p.shape[0],), 0.1, dtype=torch.float64), AABB, 0.5, P=15)
    assert res["k"].tolist() == [-1, -1] and bool(torch.isinf(res["t_star"]).all())
    res = cast64(o[1:], d[1:], t[1:], p[1:], inbox[1:], lambda x: torch.ones(x.shape[0], dtype=torch.float64), AABB,
                 0.5, P=7)
    assert res["k"].tolist() == [-1]
    assert not bool(inbox[1].any())


def test_box_face_crossing():
    """A field above the level everywhere: the crossing is where the ray enters the box."""
    o, d = _rays([[-3.35, 0.0, 0.0]], [[1.0, 0.0, 0.0]])
    t, p, inbox = _samples(o, d)
    res = cast64(o, d, t, p, inbox, lambda p: torch.ones(p.shape[0], dtype=torch.float64), AABB, 0.5, P=15)
    assert int(res["k"][0]) == 4
    assert abs(float(res["t_star"][0]) - 0.35) <= 1e-6
    assert bool(in_box64(AABB, o.double() + d.double() * res["t_star"][0]).all())


def test_fp32_refinement_terminates_at_adjacent_floats():
    """The same subdivision in float32 keeps lo outside and hi inside and stops where no float lies between them."""
    x0 = torch.tensor([0.7123456], dtype=torch.float32)
    lo, hi, rounds = refine(torch.tensor([0.7], dtype=torch.float32), torch.tensor([0.8], dtype=torch.float32),
                            lambda rows, t: t >= x0[rows, None], 15)
    assert float(lo[0]) < float(x0[0]) <= float(hi[0])
    assert float(torch.nextafter(lo, torch.tensor([1.0]))[0]) == float(hi[0])
    assert 1 <= int(rounds[0]) <= 8
    assert first_inside(torch.tensor([[False, True, True], [False, False, False]])).tolist() == [1, -1]
