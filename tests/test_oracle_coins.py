"""Oracle semantics for the coins family (lua/levels/coins/components.lua), SURVEY.md section 8f row N1."""

import json

import numpy as np

from meltingpot_b200 import blob as mpb
from meltingpot_b200 import substrates
from tests import reference_configs


def _tables(blob):
  sec = mpb.unpack(blob)
  return sec, json.loads(mpb.section_text(sec, 'info_json'))


def test_layout_and_specs(coins_blob):
  sec, info = _tables(coins_blob)
  meta = sec['meta']
  assert int(meta[0]) == 4 and int(meta[4]) == 2           # family coins, two players (components.lua:93-96)
  assert info['world_rgb_shape'] == [136, 136, 3]           # padded to the maximum map (coins.py:45-84, timestep_spec)
  assert info['individual_observation_names'] == ['RGB', 'MISMATCHED_COIN_COLLECTED_BY_PARTNER']
  assert len(info['action_set']) == 7                       # no zapping in coins
  ip, dp = sec['co_ip'], sec['co_dp']
  assert sorted(int(t) for t in ip[8:10]) == [0, 1]         # the two players own different coin types
  assert list(dp[4:8]) == [1.0, 1.0, 0.0, -2.0]             # self match, self mismatch, other match, other mismatch


def test_build_seed_fixes_the_python_side_randomness():
  # tests/golden records what coins' config builder returned after `random.seed(build_seed)` for build seeds 0-5
  a = reference_configs.compile_recorded('coins', build_seed=3)
  assert a == reference_configs.compile_recorded('coins', build_seed=3)
  shapes = {tuple(int(v) for v in mpb.unpack(reference_configs.compile_recorded('coins', build_seed=s))['co_ip'][:1])
            for s in range(6)}
  assert len(shapes) > 1  # different seeds draw different map sizes (coin counts)
  assert reference_configs.compile_recorded('coins', build_seed=substrates.BUILD_SEEDS['coins']) == \
      substrates.load_blob('coins', ('default',) * 2)


def test_coins_appear_are_collected_and_pay_by_type(oracle, coins_blob):
  sec, info = _tables(coins_blob)
  types = [int(t) for t in sec['co_ip'][8:10]]
  coin_kind = info['kinds'].index('coin')
  names = info['kind_states'][coin_kind]
  env = oracle.OracleEnv(coins_blob, 7)
  env.reset()
  assert all(names[env.object_state(int(o))] == 'coinWait' for o, _ in sec['co_coin'])  # every coin starts waiting
  rng = np.random.default_rng(0)
  seen = 0
  for _ in range(4000):
    if env.step(rng.integers(0, 7, 2)) == 2:
      break
    r = env.rewards()
    obs = env.scalar_obs()  # [P][n_scalar]
    mismatch_by = [False, False]
    expect = np.zeros(2)
    for name, player, matched in env.events():
      assert name == 'coin_consumed'
      seen += 1
      p = player - 1
      expect[p] += 1.0                      # rewardSelfForMatch == rewardSelfForMismatch == 1
      if not matched:
        expect[1 - p] += -2.0               # rewardOtherForMismatch
        mismatch_by[p] = True
    np.testing.assert_array_equal(r, expect)
    # MISMATCHED_COIN_COLLECTED_BY_PARTNER: set on the partner of whoever took a coin of the wrong type
    assert [bool(obs[0][0]), bool(obs[1][0])] == [mismatch_by[1], mismatch_by[0]]
  assert seen > 20
  assert sorted(types) == [0, 1]
