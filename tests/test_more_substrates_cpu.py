"""SURVEY.md section 8f, row N1: further substrates of the 8-substrate sweep that reuse existing components.

territory__open (BOUNDED 39x23 map, same territory.py components as territory__rooms) and
commons_harvest__closed (walled variant of commons_harvest__open). CPU side: the committed blobs are what
the compiler emits from the reference configs, and the oracle plays them without breaking invariants.
"""

import json

import numpy as np
import pytest

from meltingpot_b200 import blob as mpb
from meltingpot_b200 import compiler
from meltingpot_b200 import substrate
from meltingpot_b200 import substrates
from tests import reference_configs


CASES = [('territory__open', 9), ('territory__inside_out', 5), ('commons_harvest__closed', 7), ('commons_harvest__partnership', 7), ('coins', 2), ('coop_mining', 6)]


def _tables(blob):
  sec = mpb.unpack(blob)
  return sec, json.loads(mpb.section_text(sec, 'info_json'))


@pytest.mark.parametrize('name,players', CASES)
def test_registered_with_default_roles(name, players):
  assert name in substrate.SUBSTRATES
  cfg = substrate.get_config(name)
  assert tuple(cfg.default_player_roles) == ('default',) * players
  assert 'default' in set(cfg.valid_roles)


@pytest.mark.parametrize('name,players', CASES)
def test_committed_blob_is_what_the_compiler_emits(name, players):
  # compiled from the settings the reference's config builds (recorded under tests/golden)
  fresh = reference_configs.compile_recorded(name, build_seed=substrates.BUILD_SEEDS.get(name))
  assert fresh == substrates.load_blob(name, ('default',) * players)


@pytest.mark.parametrize('name,players', CASES)
def test_specs_follow_the_reference_config(name, players):
  ref = reference_configs.config(name)
  cfg = substrate.get_config(name)
  assert tuple(cfg.timestep_spec.observation['WORLD.RGB'].shape) == tuple(ref.world_rgb_shape)
  assert tuple(cfg.timestep_spec.observation['RGB'].shape) == tuple(ref.rgb_shape)
  assert cfg.action_spec.num_values == ref.num_actions


def test_territory_open_is_bounded_and_pays_for_claims(oracle):
  blob = substrates.load_blob('territory__open', ('default',) * 9)
  sec, info = _tables(blob)
  meta = sec['meta']
  assert int(meta[6]) == 0 and (int(meta[1]), int(meta[2])) == (39, 23)  # BOUNDED, 39 x 23 cells
  env = oracle.OracleEnv(blob, 5)
  env.reset()
  assert env.world_rgb().shape == (23 * 8, 39 * 8, 3)
  rng = np.random.default_rng(1)
  total = np.zeros(9)
  for _ in range(600):
    env.step(rng.integers(0, int(meta[19]), 9))
    total += env.rewards()
    av = env.avatars()
    alive = av[:, 3] != 0
    assert (av[alive, 0] >= 0).all() and (av[alive, 0] < 39).all() and (av[alive, 1] >= 0).all() and (av[alive, 1] < 23).all()
  assert total.sum() > 20  # claimed resources pay out (territory.py Resource rewardRate)


def test_commons_closed_walls_keep_the_orchard_closed(oracle):
  blob = substrates.load_blob('commons_harvest__closed', ('default',) * 7)
  sec, info = _tables(blob)
  apples, nbr = sec['ch_apple'], sec['ch_nbr']
  names = info['kind_states'][info['kinds'].index('apple')]
  env = oracle.OracleEnv(blob, 9)
  env.reset()
  rng = np.random.default_rng(2)
  eaten = 0
  for t in range(600):
    env.step(rng.integers(0, 8, 7))
    eaten += sum(1 for name, _, _ in env.events() if name == 'edible_consumed')
    if t % 100 == 99:
      for k in range(len(apples)):
        st = names[env.object_state(int(apples[k, 0]))]
        if st.startswith('appleWait_'):
          assert 0 <= int(st.split('_')[1]) <= (nbr[k] >= 0).sum()
  assert eaten > 5


def test_choice_prefabs_are_left_to_the_engine_unless_a_build_seed_fixes_them():
  # prefab_utils.lua:63-65: 'choice' is drawn with the env's random stream at every env build. Without a build seed the
  # blob carries the options (conditional objects) and the engine draws per env and episode; with one, a single draw is
  # baked into the blob (the older behaviour, still available for reproducing one fixed layout).
  from meltingpot_b200 import blob as blob_lib, substrates
  per_env = reference_configs.compile_recorded('territory__inside_out')
  sec = blob_lib.unpack(per_env)
  assert 'choice_groups' in sec and 'tr_res_cond' in sec and (sec['obj_choice'][:, 0] >= 0).sum() > 100
  assert per_env == substrates.load_blob('territory__inside_out', ('default',) * 5)  # the committed blob is this one
  a = reference_configs.compile_recorded('territory__inside_out', build_seed=1)
  b = reference_configs.compile_recorded('territory__inside_out', build_seed=2)
  assert a != b and 'choice_groups' not in blob_lib.unpack(a)
  assert a == reference_configs.compile_recorded('territory__inside_out', build_seed=1)


def test_role_tile_is_inert_for_default_roles_and_refused_when_it_would_pay(oracle):
  # component_library.lua:1098-1136: the tile pays rolesToRewards[role]; default builds carry role 'none'.
  config = reference_configs.config('commons_harvest__partnership')
  paying = reference_configs.settings('commons_harvest__partnership')
  for go in paying['simulation']['gameObjects']:
    for c in go['components']:
      if c['component'] == 'Role':
        c['kwargs']['role'] = 'putative_cooperator'
  with pytest.raises(NotImplementedError, match='RoleBasedRewardTile'):
    compiler.compile_settings(paying, config)
  blob = substrates.load_blob('commons_harvest__partnership', ('default',) * 7)
  env = oracle.OracleEnv(blob, 4)
  env.reset()
  rng = np.random.default_rng(5)
  total = 0.0
  for _ in range(400):
    env.step(rng.integers(0, 8, 7))
    r = env.rewards()
    assert (r >= 0).all()  # the -10 tile never fires for role 'none'
    total += r.sum()
  assert total > 0


def test_every_scalar_observation_id_has_a_name():
  # (a blob whose scalar observation the Python layer cannot name fails only when an env is built -- on a GPU)
  for name, counts in substrates.PRECOMPILED.items():
    for players in counts:
      sec = mpb.unpack(substrates.load_blob(name, ('default',) * players))
      info = json.loads(mpb.section_text(sec, 'info_json'))
      named = [substrate._SCALAR_NAMES[int(k)] for k in sec['scalar_obs']]  # pylint: disable=protected-access
      assert named == [n for n in info['individual_observation_names'] if n != 'RGB']
