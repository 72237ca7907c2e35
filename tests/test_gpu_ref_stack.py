"""GPU: this repo's API mirror and its `dmlab2d` boundary module against what the reference's OWN Python stack returned.

tests/golden/ref_stack_*.json were recorded (tools/make_ref_stack_golden.py) by running the reference's unmodified
builder.py + wrapper stack + Substrate class + configs over `lab2d_env` on the CPU oracle. Here, with no reference
checkout, (1) `meltingpot.substrate.build(...)` -- this repo's mirror of that stack, over the C ABI -- must return the
same TimeSteps, specs and events, and (2) `lab2d_env.Lab2d / Environment` with the ENGINE backend, fed the flattened
settings builder.py produced, must return the same raw observations."""

import glob
import gzip
import json
import os

import numpy as np
import pytest

from tests import ref_stack

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURES = sorted(glob.glob(os.path.join(ROOT, 'tests', 'golden', 'ref_stack_*.json')))


@pytest.mark.parametrize('path', FIXTURES, ids=lambda p: os.path.basename(p)[10:-5])
def test_substrate_api_equals_the_reference_stack(path):
  from meltingpot import substrate  # the alias package: existing `from meltingpot import substrate` code resolves here
  with open(path) as f:
    want = json.load(f)
  name, players, seed = want['substrate'], want['players'], want['seed']
  config = substrate.get_config(name)
  roles = (tuple(config.default_player_roles)[0],) * players
  with substrate.build(name, roles=roles, env_seed=seed) as env:
    assert [ref_stack._spec(s) for s in env.action_spec()] == want['action_spec']
    assert [{k: ref_stack._spec(v) for k, v in sorted(o.items())} for o in env.observation_spec()] == want['observation_spec']
    assert [ref_stack._spec(s) for s in env.reward_spec()] == want['reward_spec']
    assert ref_stack._spec(env.discount_spec()) == want['discount_spec']
    assert [dict(a) for a in config.action_set] == want['action_table']
    ts = env.reset()
    assert json.loads(json.dumps(ref_stack.describe_timestep(ts, env.events()))) == want['steps'][0]
    for t, acts in enumerate(want['actions']):
      ts = env.step(acts)
      got = json.loads(json.dumps(ref_stack.describe_timestep(ts, env.events())))
      assert got == want['steps'][t + 1], f'{name} step {t}'
  # the reference rebuilds the env with the next seed on every later reset (reset_wrapper.py:37-45, builder.py:174-187)
  with substrate.build(name, roles=roles, env_seed=seed + 1) as env:
    got = json.loads(json.dumps(ref_stack.describe_timestep(env.reset(), env.events())))
    assert got == want['second_episode_first']


@pytest.mark.parametrize('name', ['clean_up', 'territory__rooms'])
def test_engine_backed_dmlab2d_module_from_flattened_settings(name):
  # The FFI hop itself: dmlab2d.Lab2d(settings_dict) + dmlab2d.Environment(...) as builder.py:182-187 calls them, served by
  # libmpengine.so: un-flatten -> compile -> engine -> flat "{i}.RGB" observations.
  from meltingpot_b200 import lab2d_env
  with open(os.path.join(ROOT, 'tests', 'golden', f'ref_stack_{name}.json')) as f:
    want = json.load(f)
  with gzip.open(os.path.join(ROOT, 'tests', 'golden', f'ref_stack_settings_{name}.json.gz')) as f:
    flat = json.loads(f.read().decode())
  lab = lab2d_env.Lab2d('', flat)
  assert lab.env_seed == want['seed']
  P = want['players']
  with lab2d_env.Environment(env=lab, observation_names=lab.observation_names(), seed=lab.env_seed) as env:
    assert isinstance(env._backend, lab2d_env.EngineBackend)  # the CUDA engine, not a stand-in
    ref_stack.check_raw_timestep(env.reset(), want['steps'][0], P)
    for t, acts in enumerate(want['actions']):
      action = {f'{i + 1}.{k}': np.int32(v) for i, a in enumerate(acts) for k, v in want['action_table'][a].items()}
      ref_stack.check_raw_timestep(env.step(action), want['steps'][t + 1], P)


def test_substrate_dmlab2d_observables_equal_the_reference_stacks_stream():
  # observables().dmlab2d (built by flat_action / flat_timestep) against the raw stream the reference's own stack
  # emitted there for the same actions (tests/golden/dmlab2d_stream_clean_up.json, tools/make_ref_stack_golden.py).
  from meltingpot import substrate
  with open(os.path.join(ROOT, 'tests', 'golden', 'dmlab2d_stream_clean_up.json')) as f:
    want = json.load(f)
  raw_ts, raw_act = [], []
  with substrate.build(want['substrate'], roles=('default',) * want['players'], env_seed=want['seed']) as env:
    env.observables().dmlab2d.timestep.subscribe(raw_ts.append)
    env.observables().dmlab2d.action.subscribe(raw_act.append)
    env.reset()
    for acts in want['actions']:
      env.step(acts)
  assert [{k: int(v) for k, v in a.items()} for a in raw_act] == want['raw_actions']
  assert len(raw_ts) == len(want['raw_timesteps'])
  for t, (ts, rec) in enumerate(zip(raw_ts, want['raw_timesteps'])):
    got = ref_stack.describe_raw_timestep(ts)
    assert (got['step_type'], got['reward'], got['discount']) == (rec['step_type'], rec['reward'], rec['discount']), t
    assert set(got['observation']) <= set(rec['observation']), t  # (the raw env offers every observation; the wrappers select)
    for key, value in got['observation'].items():
      assert value == rec['observation'][key], (t, key)
