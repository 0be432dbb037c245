"""Model compiler vs the reference's goldens (tests/golden/reference_goldens.json) + ABI struct sync."""
import json
import os
import re

import numpy as np

from flybody_b200.flymodel import FIELDS, c_struct_text, load_model

import model_goldens

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'reference_goldens.json')))


def test_bare_model_sizes_match_reference_goldens():
    m = load_model('bare')     # reference tests/test_flybare.py:12-25
    exp = G['flybare_sizes']
    assert m.nq == exp['nq'] and m.nv == exp['nv'] and m.nu == exp['nu'] and m.nbody == exp['nbody']
    assert m.njnt == exp['njnt'] and m.meta['ngeom_all'] == exp['ngeom'] and m.nsensor == exp['nsensor']
    assert m.nsensordata == exp['nsensordata'] and m.nsite == exp['nsite'] and m.ntendon == exp['ntendon']
    assert m.nM == 1213        # SURVEY.md App. B


def test_bare_model_masses_match_reference_goldens():
    m = load_model('bare')     # reference tests/test_flybare.py:27-73 (np.isclose defaults: rtol 1e-5, atol 1e-8)
    n, st, bm = m.meta['body_names'], m.body_subtreemass, m.body_mass
    e = G['flybare_masses']
    assert np.isclose(st[n.index('thorax')], e['fly_mass'])
    assert np.isclose(st[n.index('head')], e['head'])
    assert np.isclose(bm[n.index('thorax')], e['thorax'])
    assert np.isclose(st[n.index('abdomen')], e['abdomen'])
    for side in ('left', 'right'):
        for k in (1, 2, 3):
            assert np.isclose(st[n.index(f'coxa_T{k}_{side}')], e[f'leg_T{k}'])
        assert np.isclose(bm[n.index(f'wing_{side}')], e['wing'])
    # tighter than the reference: the volume algorithm is pinned to ~1e-8 on the large bodies
    assert abs(st[n.index('thorax')] / e['fly_mass'] - 1) < 1e-7


def test_position_actuator_ctrlrange_equals_joint_range():
    m = load_model('bare')     # reference tests/test_flybare.py:76-88
    for i in range(m.nu):
        if m.actuator_trntype[i] == 0 and m.actuator_biastype[i] == 1:
            j = m.actuator_trnid[i]
            assert m.meta['actuator_names'][i] == m.meta['jnt_names'][j]
            assert np.all(m.actuator_ctrlrange[i] == m.jnt_range[j])


def test_walk_variant_contract():
    m = load_model('walk')
    # walker 109/108/59 + ghost free joint (SURVEY.md 8(a)); 2096 self pairs + 70 floor pairs (App. B)
    assert (m.nq, m.nv, m.nu, m.na) == (116, 114, 59, 59)
    assert m.npair == 2096 + 70
    assert np.isclose(m.opt_timestep, 2e-4)
    # filter dyntype + time constants (reference tests/test_flywalker.py:84-108, fruitfly.py:330-340)
    names = m.meta['actuator_names']
    for i, nme in enumerate(names):
        assert m.actuator_dyntype[i] == 2
        assert np.isclose(m.actuator_dynprm[i, 0], 0.007 if 'adhere' in nme else 0.01)
    # claw friction 1.0 (walk_imitation.py:70-73), floor params (base.py:398-401)
    gi = m.meta['geom_names'].index('walker/tarsal_claw_T1_left_collision')
    assert m.geom_friction[gi, 0] == 1.0 and m.geom_margin[gi] == 0.0005 and m.geom_gap[gi] == 0.0005
    assert m.meta['geom_names'][0] == 'floor' and np.allclose(m.geom_solref[0], [0.001, 1])


def test_action_order_and_ranges_match_reference_notebook():
    from flybody_b200.fly_envs import _ACTION_CLASS_ORDER
    m = load_model('walk')
    ci = m.meta['ctrl_indices']
    idx = [i for k in _ACTION_CLASS_ORDER if ci.get(k) for i in ci[k]]
    names = [m.meta['actuator_names'][i].split('/')[-1] for i in idx]
    assert names == G['action_names']                       # docs/getting-started.ipynb cell 46
    assert np.allclose(m.actuator_ctrlrange[idx, 0], G['action_minimum'])
    assert np.allclose(m.actuator_ctrlrange[idx, 1], G['action_maximum'])
    assert len(m.meta['observable_joints']) == G['walk_on_ball_obs_shapes']['walker/joints_pos'] == 85


def test_flight_variant_contract():
    m = load_model('flight')
    assert (m.nq, m.nv, m.nu, m.na) == (50, 48, 11, 0)      # SURVEY.md 8(a) F
    assert m.npair == 842 and m.nfluid == 2
    assert np.isclose(m.opt_timestep, 5e-5)
    assert len(m.meta['observable_joints']) == 25          # docs/sensory-input-tracking.ipynb:152
    # wing force actuators with gain 18 (constants.py:25)
    for i, nme in enumerate(m.meta['actuator_names']):
        if 'wing' in nme:
            assert m.actuator_gainprm[i, 0] == 18 and m.actuator_biastype[i] == 0


def test_header_struct_in_sync_with_field_table():
    hdr = open(os.path.join(ROOT, 'include', 'flybody_b200.h')).read()
    body = re.search(r'/\*@FBMODEL_BEGIN\*/\n(.*?)\n/\*@FBMODEL_END\*/', hdr, re.S).group(1)
    assert body.strip() == c_struct_text().strip()
    assert len(FIELDS) == len(set(n for n, _ in FIELDS))


def test_committed_models_reproduce_from_reference_assets():
    """the shipped models are what the compiler makes of the reference's fruitfly.xml (tests/golden/fruitfly_assets)"""
    for variant in ('walk', 'flight'):
        fresh = model_goldens.compile_variant(variant)
        m = load_model(variant)
        for k in ('body_mass', 'body_inertia', 'body_pos', 'geom_pos', 'dof_invweight0', 'actuator_gainprm'):
            assert np.allclose(fresh[k], getattr(m, k), rtol=1e-12, atol=0), k
