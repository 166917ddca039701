"""GPU: `BatchedWorld` with joints (revolute Joint, FixedJoint, X / Y / Rot / TotalConstraint) and no-contact pairs.

* reproduces trajectories of unmodified reference `World`s (tests/golden/bworld_joints.npz, recorded by
  tests/golden/make_joint_world_golden.py), with and without post-stabilisation;
* lcpb200_joint_rows / lcpb200_joint_move / lcpb200_find_contacts_masked against the torch paths;
* static pins and TotalConstraint joints give the same trajectory; gradients against finite differences;
* the banded large-scene route with equality rows against the CPU oracle, and its row limit.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "bworld_joints.npz")


def _golden_world(z, post_stab, dtype=torch.float64):
    from lcp_physics_b200.scenes import joint_chain_specs
    from lcp_physics_b200.world import BatchedWorld
    t = lambda k: torch.from_numpy(z[k]).to(dtype)
    js, nc = joint_chain_specs(t("anchor"))
    return BatchedWorld(t("pos"), t("rad"), vel=t("vel"), mass=t("mass"), restitution=t("rest"), fric_coeff=t("fric"),
                        gravity=100.0, static=[0], dt=1.0 / 30, post_stab=post_stab, joints=js, no_contact=nc)


@pytest.mark.parametrize("post_stab", [False, True])
def test_joint_world_reproduces_reference_worlds(post_stab):
    z = np.load(GOLDEN)
    world = _golden_world(z, post_stab)
    assert world.ne == 3 + 2 * 5 + 2 + 3 and not world.large
    tag = "ps" if post_stab else "nops"
    P, V, NC, T = (torch.from_numpy(z[tag + s]) for s in ("_p", "_v", "_nc", "_t"))
    worst_p, worst_v = 0.0, 0.0
    for k in range(P.shape[0]):
        world.step()
        assert torch.equal(world.counts.cpu().long(), NC[k].long()), (k, world.counts.tolist(), NC[k].tolist())
        assert torch.allclose(world.t.cpu(), T[k], rtol=0, atol=1e-12), k          # same dt-halving history
        worst_p = max(worst_p, float((world.p.cpu() - P[k]).abs().max()))
        worst_v = max(worst_v, float((world.v.cpu().reshape(P.shape[1], -1, 3) - V[k]).abs().max()))
    assert worst_p < 1e-6 and worst_v < 1e-5, (worst_p, worst_v)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_joint_kernels_match_torch_paths(dtype):
    """lcpb200_joint_rows (A and ge = A v) and lcpb200_joint_move (rot1, pos1, with some scenes flagged done) against
    joint_rows_torch / move_joints_torch, over several steps of a batch."""
    from lcp_physics_b200.scenes import joint_chain_specs, make_joint_chain
    from lcp_physics_b200.world import BatchedWorld
    ic = make_joint_chain(64, seed=3, dtype=dtype)
    js, nc = joint_chain_specs(ic["anchor"])
    w = BatchedWorld(ic["pos"], ic["rad"], vel=ic["vel"], mass=ic["mass"], restitution=ic["rest"], fric_coeff=ic["fric"],
                     gravity=100.0, static=[0], joints=js, no_contact=nc, post_stab=True)
    tol = 1e-13 if dtype == torch.float64 else 1e-5
    g = torch.Generator(device=w.device).manual_seed(0)
    for step in range(6):
        v = w.v
        A, ge = w.joint_rows(v)
        At, get = w.joint_rows_torch(v)
        scale = float(At.abs().max())
        assert torch.allclose(A, At, rtol=tol, atol=tol * scale), step
        terms = torch.bmm(At.abs(), v.abs().unsqueeze(2)).squeeze(2)                   # size of the summed terms
        assert bool(((ge - get).abs() <= tol * (get.abs() + terms)).all()), step
        start = w.j_rot1.clone()
        rot0, pos0 = w.j_rot1.clone(), w.j_pos1.clone()
        dts = torch.full((w.B,), 1.0 / 30, dtype=dtype, device=w.device) / 2 ** torch.randint(0, 3, (w.B,), device=w.device, generator=g)
        done = torch.rand(w.B, device=w.device, generator=g) < 0.3
        w.move_joints(start, v, dts, done)
        rot_k, pos_k = w.j_rot1.clone(), w.j_pos1.clone()
        w.j_rot1, w.j_pos1 = rot0.clone(), pos0.clone()
        w.move_joints_torch(start, v, dts, done)
        r1max = float(w.j_r1.max())
        assert torch.allclose(rot_k, w.j_rot1, rtol=tol, atol=tol * 10), step
        assert torch.allclose(pos_k, w.j_pos1, rtol=tol, atol=tol * r1max), step
        assert torch.equal(rot_k[done], rot0[done]) and torch.equal(pos_k[done], pos0[done])
        w.j_rot1, w.j_pos1 = rot0, pos0
        w.step()


def _find_contacts_call(w, skip_words, masked=True):
    from lcp_physics_b200 import _lib
    lib = _lib.load()
    pos_c = w.p[:, :, 1:].contiguous()
    b1 = torch.empty(w.B, w.cap, dtype=torch.int32, device=w.device)
    b2, counts = torch.empty_like(b1), torch.empty(w.B, dtype=torch.int32, device=w.device)
    st = ctypes.c_void_p(torch.cuda.current_stream(w.device).cuda_stream)
    if masked:
        _lib.check(lib.lcpb200_find_contacts_masked(_lib.dtype_code(w.dtype), w.B, w.nb, w.cap, w.eps, _lib.ptr(pos_c),
                                                    _lib.ptr(w.rad), _lib.ptr(skip_words), _lib.ptr(b1), _lib.ptr(b2),
                                                    _lib.ptr(counts), st))
    else:
        _lib.check(lib.lcpb200_find_contacts(_lib.dtype_code(w.dtype), w.B, w.nb, w.cap, w.eps, _lib.ptr(pos_c),
                                             _lib.ptr(w.rad), _lib.ptr(b1), _lib.ptr(b2), _lib.ptr(counts), st))
    return counts, b1, b2


def _check_masked_against_torch(w):
    counts, b1, b2 = w.find_contacts_torch()
    assert torch.equal(counts, w.counts), (counts.tolist(), w.counts.tolist())
    valid = torch.arange(w.cap, device=w.device).unsqueeze(0) < counts.unsqueeze(1)
    assert torch.equal(b1[valid], w.c_b1[valid]) and torch.equal(b2[valid], w.c_b2[valid])
    # no listed pair is a masked one
    q = w.c_b1.long() * (2 * w.nb - w.c_b1.long() - 1) // 2 + w.c_b2.long() - w.c_b1.long() - 1
    assert not bool(w.skip_mask[q[valid]].any())


def test_masked_find_contacts_matches_torch_scan_small_scene():
    from lcp_physics_b200.scenes import joint_chain_specs, make_joint_chain
    from lcp_physics_b200.world import BatchedWorld
    ic = make_joint_chain(9, seed=11)
    js, nc = joint_chain_specs(ic["anchor"])
    w = BatchedWorld(ic["pos"], ic["rad"], vel=ic["vel"], mass=ic["mass"], restitution=ic["rest"], fric_coeff=ic["fric"],
                     gravity=100.0, static=[0], joints=js, no_contact=nc)
    for _ in range(3):
        _check_masked_against_torch(w)
        w.p = w.p.clone()
        w.p[:, 1:6, 1] += 12.0                      # shift the chain so that masked neighbours also overlap others
        w.find_contacts()
        _check_masked_against_torch(w)
        w.step()


def test_masked_find_contacts_matches_torch_scan_on_pile():
    """300-ball pile, ~860 touching pairs per scene; every pair of horizontal neighbours is masked."""
    from lcp_physics_b200.scenes import make_ball_pile
    from lcp_physics_b200.world import BatchedWorld
    nballs, cols = 300, 20
    ic = make_ball_pile(9, nballs=nballs, cols=cols, seed=5, gap=0.05)
    pairs = [(1 + k, 2 + k) for k in range(nballs - 1) if (k + 1) % cols] + [(0, 7), (3, 250)]
    mk = lambda nc: BatchedWorld(ic["pos"], ic["rad"], vel=ic["vel"], mass=ic["mass"], restitution=ic["rest"],
                                 fric_coeff=ic["fric"], gravity=100.0, static=[0], contact_capacity=4 * nballs,
                                 no_contact=nc)
    w, w0 = mk(pairs), mk(())
    assert int(w.skip_mask.sum()) == len(pairs)
    _check_masked_against_torch(w)
    assert int((w0.counts - w.counts).min()) > 200                            # many touching pairs were masked
    g = torch.Generator(device=w.device).manual_seed(1)
    w.p = w.p + torch.randn(w.p.shape, dtype=w.dtype, device=w.device, generator=g) * 0.3
    w.find_contacts()
    _check_masked_against_torch(w)
    # an empty mask (and NULL) gives exactly lcpb200_find_contacts' output
    ref = _find_contacts_call(w0, None, masked=False)
    empty = torch.zeros_like(w.skip_words)
    for out in (_find_contacts_call(w0, empty), _find_contacts_call(w0, None)):
        for a, b in zip(out, ref):
            assert torch.equal(a, b)


@pytest.mark.parametrize("post_stab", [False, True])
def test_total_constraint_joint_equals_static_pin(post_stab):
    from lcp_physics_b200.constraints import TotalConstraint
    from lcp_physics_b200.world import BatchedWorld
    z = np.load(os.path.join(HERE, "golden", "bworld_balls.npz"))
    t = lambda k: torch.from_numpy(z[k])
    kw = dict(vel=t("vel"), mass=t("mass"), restitution=t("rest"), fric_coeff=t("fric"), gravity=100.0, post_stab=post_stab)
    a = BatchedWorld(t("pos"), t("rad"), static=[0], **kw)
    b = BatchedWorld(t("pos"), t("rad"), gravity_mask=[False] + [True] * (t("pos").shape[1] - 1),
                     joints=[TotalConstraint(0)], **kw)
    assert a.ne == b.ne == 3 and torch.equal(a.A, b.A)
    for k in range(25):
        a.step()
        b.step()
        assert torch.equal(a.p, b.p) and torch.equal(a.v, b.v) and torch.equal(a.t, b.t), k


def _hanging_chain(vel, mass, anchor, post_stab, steps):
    """Contact-free chain of 4 overlapping links (no-contact neighbours) hung from a world joint; returns the final
    link positions."""
    from lcp_physics_b200.constraints import Joint
    from lcp_physics_b200.world import BatchedWorld
    L = 4
    pos = torch.tensor([[[300.0 + 6.0 * k, 130.0 + 25.0 * k] for k in range(L)]], dtype=torch.float64).expand(2, L, 2)
    js = [Joint(0, None, anchor)] + [Joint(k + 1, k, pos[:, k] * 0.5 + pos[:, k + 1] * 0.5) for k in range(L - 1)]
    w = BatchedWorld(pos, 15.0, vel=vel, mass=mass, gravity=100.0, joints=js,
                     no_contact=[(k, k + 1) for k in range(L - 1)], post_stab=post_stab)
    for _ in range(steps):
        w.step()
        assert int(w.counts.max()) == 0
    return w.p[:, :, 1:]


@pytest.mark.parametrize("post_stab", [False, True])
def test_joint_world_gradients_match_finite_differences(post_stab):
    """d(final link positions . weights) / d(initial velocity, link mass, anchor) over 12 steps against central
    differences (h = 1e-6 relative). Without contacts the step is a smooth function of these inputs and each LCP
    is an equality-constrained solve whose KKT system is symmetric, so the adjoint is exact; central differences
    in fp64 carry O(h^2) truncation and ~1e-16 |f| / h round-off, both far below the relative tolerance 1e-5."""
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(0)
    vel0 = (torch.randn(2, 4, 3, generator=g, dtype=torch.float64) * torch.tensor([0.2, 20.0, 20.0], dtype=torch.float64)).to(dev)
    mass0 = (0.5 + torch.rand(2, 4, generator=g, dtype=torch.float64)).to(dev)
    anchor0 = torch.tensor([[300.0, 108.0], [299.0, 106.0]], dtype=torch.float64, device=dev)
    wts = torch.randn(2, 4, 2, generator=g, dtype=torch.float64).to(dev)
    steps = 12
    f = lambda v, m, a: float((_hanging_chain(v, m, a, post_stab, steps) * wts).sum())
    leaves = [t.clone().requires_grad_(True) for t in (vel0, mass0, anchor0)]
    (_hanging_chain(*leaves, post_stab, steps) * wts).sum().backward()
    base = [vel0, mass0, anchor0]
    checks = [(0, (0, 2, 1)), (0, (1, 0, 0)), (0, (0, 3, 2)), (1, (0, 1)), (1, (1, 3)), (2, (0, 0)), (2, (1, 1))]
    with torch.no_grad():
        for which, idx in checks:
            x = base[which]
            h = 1e-6 * max(1.0, abs(float(x[idx])))
            plus, minus = [t.clone() for t in base], [t.clone() for t in base]
            plus[which][idx] += h
            minus[which][idx] -= h
            fd = (f(*plus) - f(*minus)) / (2 * h)
            an = float(leaves[which].grad[idx])
            assert abs(an - fd) <= 1e-5 * max(abs(fd), 1e-3), (which, idx, an, fd)


def test_banded_route_with_constraints_matches_oracle():
    """60-ball pile on a pinned floor ball (n = 183): X / Y / Rot constraints and a no-contact pair on the banded
    kernel (e = 6; border 3 x 3 bodies + 6 rows = 15 <= 16), against OracleJointWorld with the same constraints."""
    from lcp_physics_b200.constraints import RotConstraint, XConstraint, YConstraint
    from lcp_physics_b200.world import BatchedWorld
    from oracle.joint_world_oracle import OracleJointWorld
    z = np.load(os.path.join(HERE, "golden", "bworld_large.npz"))
    js = [XConstraint(5), RotConstraint(5), YConstraint(30)]
    nc = [(30, 39)]                                  # a pair that touches from the third step on without the mask
    t = lambda k: torch.from_numpy(z[k]).unsqueeze(0).expand(2, *z[k].shape).contiguous()
    w = BatchedWorld(t("pos"), t("rad"), vel=t("vel"), mass=t("mass"), restitution=t("rest"), fric_coeff=t("fric"),
                     gravity=100.0, static=[0], joints=js, no_contact=nc)
    assert w.large and w.ne == 6
    o = OracleJointWorld(z["pos"], z["rad"], z["vel"], z["mass"], z["rest"], z["fric"], gravity=100.0, static=(0,),
                          joints=js, no_contact=nc)
    worst_p = worst_v = 0.0
    for k in range(8):
        w.step()
        o.step()
        assert [int(c) for c in w.counts.tolist()] == [len(o.contacts)] * 2, k
        worst_p = max(worst_p, float((w.p.cpu() - o.p).abs().max()))
        worst_v = max(worst_v, float((w.v.cpu() - o.v).abs().max()))
    assert abs(float(w.t[0]) - o.t) < 1e-12
    assert worst_p < 1e-6 and worst_v < 1e-5, (worst_p, worst_v)


def test_too_many_rows_for_the_banded_kernel_raise():
    from lcp_physics_b200.constraints import XConstraint
    from lcp_physics_b200.world import BatchedWorld
    z = np.load(os.path.join(HERE, "golden", "bworld_large.npz"))
    t = lambda k: torch.from_numpy(z[k]).unsqueeze(0)
    with pytest.raises(ValueError, match="e = 18"):
        BatchedWorld(t("pos"), t("rad"), gravity=100.0, static=[0], joints=[XConstraint(k) for k in range(1, 16)])
    with pytest.raises(ValueError, match="border"):                         # 3 x 4 bodies + 6 rows > 16
        BatchedWorld(t("pos"), t("rad"), gravity=100.0, static=[0], joints=[XConstraint(k) for k in (5, 30, 44)])
