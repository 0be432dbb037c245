"""Model variants: the `FruitFly` constructor switches the reference's env factories expose (force_actuators, disable_wings,
disable_legs, joint_filter; reference fly_envs.py:100-246, fruitfly.py:204-340) compiled on demand, and the reference's walker
contracts of tests/test_flywalker.py:36-168 (all 16 use-combinations x 4 filter settings: action <-> ctrl index maps, actuator
dyntype / dynprm, ctrlrange of named actuators, force actuators, filterexact) checked on OUR compiled models -- the reference
checks them on MuJoCo's compilation of the same MJCF surgery.  Compiled from the reference's fruitfly.xml stored under
tests/golden/fruitfly_assets; every compilation is also checked against the stored one (tests/model_goldens.py)."""
import numpy as np
import pytest

import __graft_entry__ as ge
from flybody_b200 import fly_envs, stepper as st
from flybody_b200.dm_env_shim import StepType
from flybody_b200.flymodel import from_compiled

import model_goldens

JOINT_FILTER, ADHESION_FILTER = 0.0123, 0.0234                     # tests/test_flywalker.py:13-14
USES = [(i, j, k, l) for i in range(2) for j in range(2) for k in range(2) for l in range(2)]
FILTERS = [(0, 0), (JOINT_FILTER, 0), (0, ADHESION_FILTER), (JOINT_FILTER, ADHESION_FILTER)]


@pytest.fixture(scope='module')
def emu():
    ge.build()
    return ge.EMU


def _walker(use, flt, **kw):
    return from_compiled(model_goldens.compile_variant('walker', use_legs=bool(use[0]), use_wings=bool(use[1]), use_mouth=bool(use[2]),
                                                       use_antennae=bool(use[3]), joint_filter=flt[0], adhesion_filter=flt[1], **kw))


def test_fly_bulletproof_contracts_on_the_compiled_walker(emu):
    """tests/test_flywalker.py:36-121 on our compiler's output, every configuration; a subset is also stepped."""
    counts = set()
    for ui, use in enumerate(USES):
        for fi, flt in enumerate(FILTERS):
            m = _walker(use, flt)
            ci = m.meta['ctrl_indices']
            # action_spec consistency + every action class maps onto distinct, in-range ctrl slots (:62-82)
            idx = [i for key in ('adhesion', 'head', 'mouth', 'antennae', 'wings', 'abdomen', 'legs') for i in (ci.get(key) or [])]
            assert len(idx) == len(set(idx)) == m.nu and all(0 <= i < m.nu for i in idx), (use, flt)
            counts.add((use, m.nu))
            names = m.meta['actuator_names']
            for i in range(m.nu):
                trn = int(m.actuator_trntype[i])
                if trn == 0:                                       # joint actuators (:89-98)
                    assert (m.actuator_dynprm.reshape(m.nu, -1)[i, 0], int(m.actuator_dyntype[i])) == ((1.0, 0) if flt[0] == 0 else (JOINT_FILTER, 2)), names[i]
                if trn == 5:                                       # adhesion actuators (:99-107)
                    assert (m.actuator_dynprm.reshape(m.nu, -1)[i, 0], int(m.actuator_dyntype[i])) == ((1.0, 0) if flt[1] == 0 else (ADHESION_FILTER, 2)), names[i]
            # activations exist exactly for the filtered actuators
            assert m.na == int((np.asarray(m.actuator_dyntype) != 0).sum())
            if (ui * 4 + fi) % 9 == 0:                             # can compile AND step (:52-59), on the kernel source
                s = st.BatchedStepper(m, 1, lib_path=emu)
                rs = np.random.RandomState(ui)
                for k in range(2):
                    s.set_control(rs.uniform(-0.2, 0.2, (1, m.nu)).astype(np.float32)); s.step(10)
                assert np.all(np.isfinite(s.get(st.QPOS))) and int(s.get(st.FLAGS)[0, 0]) & 1 == 0
                s.close()
    nu = dict(counts)
    assert nu[(1, 1, 1, 1)] == 78 and nu[(1, 0, 0, 0)] == 59 and nu[(0, 1, 0, 0)] == 11       # tests/test_flybare.py:14, test_walking_env.py:24, flight: 11


def test_force_actuators_and_filterexact():
    """tests/test_flywalker.py:124-168 with tests/common.py:6-29 (`is_force_actuator`: gain 1, no bias on joint / tendon actuators)."""
    m = _walker((1, 1, 1, 1), (0.01, 0.02), force_actuators=True)
    gp, bp = m.actuator_gainprm.reshape(m.nu, -1), m.actuator_biasprm.reshape(m.nu, -1)
    for i in range(m.nu):
        if int(m.actuator_trntype[i]) in (0, 3):                   # joint / tendon transmissions
            assert int(m.actuator_biastype[i]) == 0 and np.all(bp[i, :3] == 0), m.meta['actuator_names'][i]
    for exact, want in ((False, 2), (True, 3)):
        m = _walker((1, 1, 1, 1), (0.01, 0.02), dyntype_filterexact=exact)
        assert all(int(m.actuator_dyntype[i]) == want for i in range(m.nu) if int(m.actuator_trntype[i]) in (0, 5))


def test_env_factories_accept_the_reference_switches(emu, tmp_path, monkeypatch):
    """walk_imitation(force_actuators / disable_wings=False / joint_filter) and flight_imitation(disable_legs=False / joint_filter):
    compiled on first use, cached, stepped; the flight env with legs gains the leg observables (tasks/base.py:360-364)."""
    monkeypatch.setenv('FLYBODY_ASSETS', model_goldens.ASSETS)
    monkeypatch.setenv('FLYBODY_B200_CACHE', str(tmp_path))
    env = fly_envs.walk_imitation(n_envs=2, lib_path=emu, disable_wings=False, terminal_com_dist=float('inf'))
    assert env.action_spec().shape == (65,) and 'wing_yaw_left' in env.action_spec().name
    ts = env.reset(); ts = env.step(np.zeros((2, 65)))
    assert ts.observation['walker/joints_pos'].shape == (2, 91) and np.all(ts.reward == 1)
    env.close()
    env = fly_envs.walk_imitation(n_envs=2, lib_path=emu, force_actuators=True, joint_filter=0.0, terminal_com_dist=float('inf'))
    assert env.action_spec().shape == (59,) and env.model.na == 6              # only the adhesion actuators keep an activation
    ts = env.reset(); ts = env.step(np.random.RandomState(0).uniform(-0.01, 0.01, (2, 59)))
    assert all(np.all(np.isfinite(v)) for v in ts.observation.values())
    env.close()
    assert (tmp_path / 'fly_walk_wings.npz').exists() and (tmp_path / 'fly_walk_force_jf0.npz').exists()
    env = fly_envs.flight_imitation(n_envs=2, lib_path=emu, disable_legs=False, joint_filter=0.0002, seed=1)
    names = list(env.observation_spec())
    assert names == ['walker/accelerometer', 'walker/actuator_activation', 'walker/appendages_pos', 'walker/force', 'walker/gyro', 'walker/joints_pos',
                     'walker/joints_vel', 'walker/touch', 'walker/velocimeter', 'walker/world_zaxis', 'walker/ref_displacement', 'walker/ref_root_quat']
    assert env.action_spec().shape == (66,)                                    # adhesion 6, head 3, wings 6, abdomen 2, legs 48 + user 1
    ts = env.reset()
    for _ in range(3):
        ts = env.step(np.random.RandomState(1).uniform(-0.2, 0.2, (2, env.action_spec().shape[0])))
    assert np.all(np.asarray(ts.step_type) == int(StepType.MID)) and all(np.all(np.isfinite(v)) for v in ts.observation.values())
    env.close()
    # the device-side task program works on a variant too
    env = fly_envs.walk_imitation(n_envs=2, lib_path=emu, disable_wings=False, device_task=True, terminal_com_dist=float('inf'))
    env.reset(); ts = env.step(np.zeros((2, 65), np.float32))
    assert np.all(ts.reward == 1)
    env.close()
    # the cached compilations against the stored ones (the switches as model_for hands them to the compiler)
    sw = dict(force_actuators=False, use_wings=None, use_legs=None, joint_filter=None)
    for name, variant, kw in (('fly_walk_wings', 'walk', dict(sw, use_wings=True)), ('fly_walk_force_jf0', 'walk', dict(sw, force_actuators=True, joint_filter=0.0)),
                              ('fly_flight_legs_jf0.0002', 'flight', dict(sw, use_legs=True, joint_filter=0.0002))):
        model_goldens.assert_matches_stored(*model_goldens.read_saved(str(tmp_path / f'{name}.npz')), variant, **kw)
