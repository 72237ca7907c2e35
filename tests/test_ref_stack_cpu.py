"""This repo's `dmlab2d` boundary module against what the reference's own Python stack returned over it (CPU: oracle backend)."""

import gzip
import json
import os
import sys

import numpy as np
import pytest

from meltingpot_b200 import compiler, lab2d_env
from tests import ref_stack, reference_configs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_unflatten_inverts_flatten_and_str():
  settings = {'levelName': 'clean_up', 'numPlayers': 7, 'spriteSize': 8, 'topology': 'BOUNDED', 'flag': True, 'none': None,
              'simulation': {'map': '\nWW\nW \n', 'charPrefabMap': {'1': 'a', 'W': 'wall'}, 'rate': 0.05, 'tiny': 1e-05,
                             'prefabs': {'wall': {'name': 'wall', 'components': [{'component': 'Transform', 'kwargs': {}},
                                                                                 {'component': 'Appearance', 'kwargs': {'colors': [(1, 2, 3, 255)], 'names': ['Wall']}}]}},
                             'gameObjects': [{'name': 'avatar', 'components': [{'component': 'Avatar', 'kwargs': {'index': 1, 'neg': -1}}]}]}}
  flat = {k: str(v) for k, v in lab2d_env.flatten_args(settings).items()}
  assert flat['simulation.prefabs.wall.components.2.kwargs.colors.1.4'] == '255'
  back = lab2d_env.unflatten_args(flat)
  want = json.loads(json.dumps(settings))  # tuples -> lists
  del want['simulation']['prefabs']['wall']['components'][0]['kwargs']  # an empty dict has no flat key
  del back['simulation']['prefabs']['wall']['components'][0]
  del want['simulation']['prefabs']['wall']['components'][0]
  assert back == want
  assert isinstance(back['simulation']['charPrefabMap'], dict)  # digit keys, still a dict


@pytest.mark.parametrize('name,players', [('clean_up', 7), ('territory__rooms', 9), ('coins', 2)])
def test_oracle_backed_dmlab2d_module_reproduces_the_committed_fixture(name, players):
  # tests/golden/ref_stack_<name>.json is what the reference's own stack returned over lab2d_env on the CPU oracle
  # (tools/make_ref_stack_golden.py). Fed the flattened settings that stack's builder.py produced, the boundary module on
  # the oracle must return the same raw observations, rewards and events, and the next episode's first step.
  with open(os.path.join(ROOT, 'tests', 'golden', f'ref_stack_{name}.json')) as f:
    want = json.load(f)
  with gzip.open(os.path.join(ROOT, 'tests', 'golden', f'ref_stack_settings_{name}.json.gz')) as f:
    flat = json.loads(f.read().decode())
  lab = lab2d_env.Lab2d('', flat)
  assert lab.env_seed == want['seed'] and lab.num_players == players

  saved = lab2d_env.BACKEND_FACTORY
  lab2d_env.BACKEND_FACTORY = ref_stack.OracleBackend
  try:
    with lab2d_env.Environment(env=lab, observation_names=lab.observation_names(), seed=lab.env_seed) as env:
      ref_stack.check_raw_timestep(env.reset(), want['steps'][0], players, env)
      for t, acts in enumerate(want['actions']):
        action = {f'{i + 1}.{k}': np.int32(v) for i, a in enumerate(acts) for k, v in want['action_table'][a].items()}
        ref_stack.check_raw_timestep(env.step(action), want['steps'][t + 1], players, env)
    # the reference rebuilds the env with the next seed on every later reset (reset_wrapper.py:37-45, builder.py:174-187)
    with lab2d_env.Environment(env=lab, observation_names=lab.observation_names(), seed=lab.env_seed + 1) as env:
      ref_stack.check_raw_timestep(env.reset(), want['second_episode_first'], players, env)
  finally:
    lab2d_env.BACKEND_FACTORY = saved


def test_compiling_from_flattened_settings_equals_compiling_from_the_config():
  # builder.py flattens the settings to "a.b.1.c" -> str for Lua (builder.py:55-67); lab2d_env un-flattens them. The blob
  # compiled from the round-tripped settings must equal the one compiled from the config's own settings.
  config = reference_configs.config('clean_up')
  settings = reference_configs.settings('clean_up')
  flat = {k.replace('$', '.'): str(v) for k, v in lab2d_env.flatten_args(settings).items()}
  back = lab2d_env.unflatten_args(flat)
  assert compiler.compile_settings(back, config) == compiler.compile_settings(settings, config)


def test_reference_import_leaves_no_stub_modules_behind(tmp_path):
  # A stand-in checkout laid out like the reference: a config module that imports from meltingpot.utils.
  pkg = tmp_path / 'meltingpot'
  (pkg / 'configs' / 'substrates').mkdir(parents=True)
  (pkg / 'utils' / 'substrates').mkdir(parents=True)
  (pkg / 'utils' / 'substrates' / 'shapes.py').write_text("WALL = 'W'\n")
  (pkg / 'configs' / 'substrates' / '__init__.py').write_text(
      'import importlib\n\n\ndef get_config(name):\n'
      "  return importlib.import_module(f'meltingpot.configs.substrates.{name}').get_config()\n")
  (pkg / 'configs' / 'substrates' / 'clean_up.py').write_text(
      'from meltingpot.utils.substrates import shapes\n\n\ndef get_config():\n  return shapes.WALL\n')
  assert compiler.load_reference_config('clean_up', root=str(tmp_path)) == 'W'
  import meltingpot  # this repo's alias package, not a stub of the checkout
  assert 'meltingpot_b200' in (meltingpot.__doc__ or '') and hasattr(meltingpot, 'substrate')
  assert not [k for k in sys.modules if k.startswith('meltingpot.configs')]


@pytest.mark.parametrize('name,players', [('clean_up', 7), ('territory__rooms', 9)])
def test_boundary_module_compiles_builder_settings_and_refuses_to_run_without_a_gpu(name, players):
  # No reference checkout needed: the flattened settings builder.py handed to dmlab2d.Lab2d are committed. lab2d_env
  # un-flattens and compiles them; apart from the action table (full product at this boundary) the blob equals the
  # committed one. Constructing the environment needs the engine: without a CUDA device it raises, there is no CPU path.
  import torch
  from meltingpot_b200 import blob as blob_lib, engine, substrates
  with gzip.open(os.path.join(ROOT, 'tests', 'golden', f'ref_stack_settings_{name}.json.gz')) as f:
    flat = json.loads(f.read().decode())
  lab = lab2d_env.Lab2d('', flat)
  got, want = blob_lib.unpack(lab.blob), blob_lib.unpack(substrates.load_blob(name, ('default',) * players))
  for key in ('objects', 'states', 'kinds', 'comps', 'comps_f', 'init_grid', 'atlas', 'sprite_map', 'hits', 'av_table'):
    assert np.array_equal(got[key], want[key]), key
  assert got['action_table'].shape[0] == len(lab.actions.table) > want['action_table'].shape[0]
  for row in want['action_table']:  # every action of the substrate's discrete set is in the full product, at its mixed-radix index
    fields = dict(zip(['move', 'turn', 'fireZap', 'fireClean' if name == 'clean_up' else 'fireClaim'], (int(v) for v in row)))
    idx = lab.actions.index([fields[k] for k in lab.actions.order])
    assert np.array_equal(got['action_table'][idx], row)
  assert lab.observation_names()[:2] == ['1.RGB', '1.REWARD'] and lab.observation_names()[-1] == 'WORLD.RGB'
  if not torch.cuda.is_available():
    with pytest.raises(engine.EngineError, match='no CPU path'):
      lab2d_env.Environment(env=lab, observation_names=lab.observation_names(), seed=lab.env_seed)


def test_flat_views_equal_the_reference_stacks_own_dmlab2d_stream():
  # tests/golden/dmlab2d_stream_clean_up.json: what the reference's innermost ObservablesWrapper emitted
  # (observables_wrapper.py:43-58) while its stack played `actions` over lab2d_env on the CPU oracle. flat_action (what
  # this repo's Substrate emits on observables().dmlab2d.action) must rebuild the action dicts its wrappers handed to
  # dmlab2d; fed those dicts, the boundary module must return the recorded flat TimeSteps. (tests/test_gpu_ref_stack.py
  # checks flat_timestep, through the Substrate's own stream, against the same recording.)
  from meltingpot_b200 import substrate as b200_substrate
  with open(os.path.join(ROOT, 'tests', 'golden', 'dmlab2d_stream_clean_up.json')) as f:
    want = json.load(f)
  action_set = reference_configs.config('clean_up').action_set
  for acts, rec in zip(want['actions'], want['raw_actions']):
    mine = b200_substrate.flat_action(acts, action_set)
    assert all(v.dtype == np.int32 and v.shape == () for v in mine.values())
    assert {k: int(v) for k, v in mine.items()} == rec
  with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'ref_stack_settings_clean_up.json.gz')) as f:
    lab = lab2d_env.Lab2d('', json.loads(f.read().decode()))
  assert lab.env_seed == want['seed']
  saved = lab2d_env.BACKEND_FACTORY
  lab2d_env.BACKEND_FACTORY = ref_stack.OracleBackend
  try:
    with lab2d_env.Environment(env=lab, observation_names=lab.observation_names(), seed=lab.env_seed) as env:
      got = [ref_stack.describe_raw_timestep(env.reset())]
      for rec in want['raw_actions']:
        got.append(ref_stack.describe_raw_timestep(env.step({k: np.int32(v) for k, v in rec.items()})))
  finally:
    lab2d_env.BACKEND_FACTORY = saved
  assert got == want['raw_timesteps']
