"""CPU: the world oracle with joints and no-contact pairs against trajectories recorded from the unmodified reference
(tests/golden/bworld_joints.npz, tests/golden/make_joint_world_golden.py), and the constraint specs' validation and
row table."""
import os

import numpy as np
import pytest
import torch

from lcp_physics_b200.constraints import (LEVER_X, LEVER_Y, ROT, UNIT, FixedJoint, Joint, RotConstraint,
                                          TotalConstraint, XConstraint, YConstraint, pair_mask, row_table)
from lcp_physics_b200.scenes import joint_chain_specs
from oracle.joint_world_oracle import OracleJointWorld

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bworld_joints.npz")


@pytest.mark.parametrize("post_stab", [False, True])
def test_world_oracle_with_joints_matches_reference_world(post_stab):
    z = np.load(GOLDEN)
    tag = "ps" if post_stab else "nops"
    for w in (0, 3):
        js, nc = joint_chain_specs(torch.from_numpy(z["anchor"][w]))
        world = OracleJointWorld(z["pos"][w], z["rad"][w], z["vel"][w], z["mass"][w], z["rest"][w], z["fric"][w],
                                  gravity=100.0, static=(0,), dt=1.0 / 30, post_stab=post_stab, joints=js, no_contact=nc)
        for k in range(z[tag + "_p"].shape[0]):
            world.step()
            assert len(world.contacts) == int(z[tag + "_nc"][k, w]), k
            assert np.abs(world.p.numpy() - z[tag + "_p"][k, w]).max() < 1e-8, k
            assert np.abs(world.v.numpy().reshape(-1, 3) - z[tag + "_v"][k, w]).max() < 1e-7, k
        assert abs(world.t - z[tag + "_t"][-1, w]) < 1e-12


def test_joint_golden_covers_contacts_on_jointed_bodies_and_dt_halving():
    z = np.load(GOLDEN)
    for tag in ("nops", "ps"):
        t = z[tag + "_t"]
        dts = np.diff(np.concatenate([np.zeros((1, t.shape[1])), t]), axis=0)
        assert (np.abs(dts - 1.0 / 30) > 1e-12).any()                      # at least one dt halving
        assert (z[tag + "_nc"] > 0).any()
    js, _ = joint_chain_specs(torch.from_numpy(z["anchor"][0]))
    assert any(isinstance(j, Joint) and j.i2 is not None and j.i1 > j.i2 for j in js)


def test_specs_reject_malformed_input():
    with pytest.raises(ValueError):
        Joint(2, 2, [0.0, 0.0])                      # a joint of a body with itself
    with pytest.raises(ValueError):
        FixedJoint(1, 1)
    with pytest.raises(ValueError):
        FixedJoint(1)                                # no second body
    with pytest.raises(ValueError):
        FixedJoint(1, None)
    with pytest.raises(ValueError):
        XConstraint(-1)
    with pytest.raises(ValueError):
        Joint(0, None, [1.0, 2.0, 3.0])
    with pytest.raises(ValueError):
        row_table([YConstraint(5)], nb=5)            # index out of range
    with pytest.raises(ValueError):
        row_table([Joint(0, 7, [0.0, 0.0])], nb=5)
    with pytest.raises(ValueError):
        pair_mask([(1, 1)], 4)
    with pytest.raises(ValueError):
        pair_mask([(0, 4)], 4)


def test_row_table_follows_reference_order():
    """World.Je() order (world.py:156-170): every spec's rows in list order, 2 / 3 / 1 / 1 / 1 / 3 rows."""
    specs = [TotalConstraint(0), Joint(3, 2, [1.0, 2.0]), XConstraint(4), FixedJoint(5, 6), Joint(1, None, [0.0, 0.0]),
             RotConstraint(4), YConstraint(1)]
    rows, revolute = row_table(specs, nb=7)
    assert len(rows) == 3 + 2 + 1 + 3 + 2 + 1 + 1
    assert rows == [(UNIT, 0, -1, 0), (UNIT, 0, -1, 1), (UNIT, 0, -1, 2),
                    (LEVER_X, 3, 2, 0), (LEVER_Y, 3, 2, 0),
                    (UNIT, 4, -1, 1),
                    (LEVER_X, 5, 6, -1), (LEVER_Y, 5, 6, -1), (ROT, 5, 6, -1),
                    (LEVER_X, 1, -1, 1), (LEVER_Y, 1, -1, 1),
                    (UNIT, 4, -1, 0), (UNIT, 1, -1, 2)]
    assert revolute == [specs[1], specs[4]]


def test_pair_mask_indexes_lexicographic_pairs():
    nb = 40
    mask, words = pair_mask([(3, 1), (0, 39), (38, 39)], nb)
    ii, jj = torch.triu_indices(nb, nb, 1)
    assert sorted(zip(ii[mask].tolist(), jj[mask].tolist())) == [(0, 39), (1, 3), (38, 39)]
    bits = ((words.long().unsqueeze(1) & 0xFFFFFFFF) >> torch.arange(32)) & 1
    assert torch.equal(bits.reshape(-1)[:mask.numel()].bool(), mask)
    assert int(bits.reshape(-1)[mask.numel():].sum()) == 0
