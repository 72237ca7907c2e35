"""TEST INFRASTRUCTURE: runs the reference's own Python stack (UNMODIFIED builder.py, wrapper stack, Substrate class,
configs; imported from MELTINGPOT_REFERENCE_ROOT) on top of `meltingpot_b200.lab2d_env` -- the `dmlab2d` boundary
module -- with the CPU oracle plugged in as the backend, and records what that stack returns. The records become
the fixtures tests/golden/ref_stack_*.json which the GPU tests compare `meltingpot_b200.substrate.build(...)` and the
engine-backed boundary module against on the GPU box (where no reference checkout exists)."""

import contextlib
import hashlib
import random

import numpy as np

from meltingpot_b200 import compiler, lab2d_env, shims, substrates

SEED = 4242
STEPS = 48
SUBSTRATES = [(name, counts[0]) for name, counts in substrates.PRECOMPILED.items()]


class OracleBackend:
  """lab2d_env backend on the CPU oracle (tests only)."""

  def __init__(self, blob, seed):
    from oracle import binding
    binding.build()
    self._binding = binding
    self._env = binding.OracleEnv(blob, seed)
    self._code = {v: k for k, v in binding.EVENT_NAMES.items()}

  def reset(self):
    self._env.reset()

  def step(self, ids):
    self._env.step(np.asarray(ids, np.int32))

  def outputs(self):
    e = self._env
    return {'rgb': e.rgb(), 'world_rgb': e.world_rgb(), 'reward': e.rewards(), 'scalar_obs': e.scalar_obs().T.copy(),
            'step_type': int(e.step_type()), 'discount': float(e.discount())}

  def events(self):
    return np.array([(self._code[n], a, b) for n, a, b in self._env.events()], np.int32).reshape(-1, 3)

  def close(self):
    self._env.close()


@contextlib.contextmanager
def reference_stack_on_oracle():
  """Inside: `meltingpot.*` is the reference checkout, `dmlab2d` is lab2d_env with the oracle backend."""
  import sys
  shims.install()
  saved_backend = lab2d_env.BACKEND_FACTORY
  saved_dmlab2d = {k: v for k, v in sys.modules.items() if k == 'dmlab2d' or k.startswith('dmlab2d.')}
  sys.modules.update(lab2d_env.build_modules())
  lab2d_env.BACKEND_FACTORY = OracleBackend
  try:
    with compiler.reference_packages():
      yield
  finally:
    lab2d_env.BACKEND_FACTORY = saved_backend
    for k in [k for k in sys.modules if k == 'dmlab2d' or k.startswith('dmlab2d.')]:
      del sys.modules[k]
    sys.modules.update(saved_dmlab2d)


def _sha(a):
  return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def _spec(s):
  d = {'shape': list(s.shape), 'dtype': np.dtype(s.dtype).name}
  if hasattr(s, 'num_values'):
    d['num_values'] = int(s.num_values)
  return d


def describe_timestep(ts, env_events):
  """What a fixture keeps of one TimeStep of the P-player API."""
  rec = {'step_type': int(ts.step_type), 'reward': [float(r) for r in ts.reward], 'discount': float(ts.discount),
         'players': []}
  for obs in ts.observation:
    p = {}
    for k in sorted(obs):
      v = np.asarray(obs[k])
      p[k] = _sha(v) if v.ndim else float(v)
    rec['players'].append(p)
  rec['world_shared'] = all(ts.observation[0].get('WORLD.RGB') is o.get('WORLD.RGB') for o in ts.observation)
  rec['events'] = sorted([name, [float(x) if isinstance(x, np.ndarray) else x.decode() for x in payload]] for name, payload in env_events)
  return rec


def actions_for(name, players, num_actions, steps=STEPS):
  rng = np.random.default_rng(abs(hash((name, players))) % (2 ** 31) if False else sum(map(ord, name)) + players)
  return rng.integers(0, num_actions, size=(steps, players))


def _build_reference_env(name, players, seed):
  """Inside reference_stack_on_oracle(): the reference's meltingpot.substrate.build(name) with default roles and the env
  seed pinned to `seed`. Returns (config, env)."""
  import importlib
  ref_substrate = importlib.import_module('meltingpot.substrate')
  ref_builder = importlib.import_module('meltingpot.utils.substrates.builder')
  config = ref_substrate.get_config(name)
  roles = (tuple(config.default_player_roles)[0],) * players
  original = ref_builder.builder
  ref_builder.builder = lambda settings, **kw: original(settings, env_seed=seed, **kw)  # pin the seed builder.py would draw
  state = random.getstate()
  try:
    build_seed = substrates.BUILD_SEEDS.get(name)
    if build_seed is not None:
      random.seed(build_seed)  # configs that draw their map from Python's `random` (coins.py:45-84)
    return config, ref_substrate.build(name, roles=roles)
  finally:
    random.setstate(state)
    ref_builder.builder = original


def run_reference_stack(name, players, steps=STEPS, seed=SEED):
  """Builds `name` through the reference's meltingpot.substrate.build (its configs, builder.py, wrappers, Substrate) on
  the oracle-backed dmlab2d module and returns the fixture record."""
  with reference_stack_on_oracle():
    config, env = _build_reference_env(name, players, seed)
    try:
      rec = {'substrate': name, 'players': players, 'seed': seed, 'class': type(env).__module__ + '.' + type(env).__name__,
             'action_table': [dict(a) for a in compiler._plain(config.action_set)],  # pylint: disable=protected-access
             'flat_settings': dict(lab2d_env.LAST_LAB2D.flat_settings),
             'action_spec': [_spec(s) for s in env.action_spec()],
             'observation_spec': [{k: _spec(v) for k, v in sorted(o.items())} for o in env.observation_spec()],
             'reward_spec': [_spec(s) for s in env.reward_spec()], 'discount_spec': _spec(env.discount_spec()),
             'steps': []}
      acts = actions_for(name, players, env.action_spec()[0].num_values, steps)
      rec['actions'] = acts.tolist()
      ts = env.reset()
      rec['steps'].append(describe_timestep(ts, env.events()))
      for t in range(steps):
        ts = env.step([int(a) for a in acts[t]])
        rec['steps'].append(describe_timestep(ts, env.events()))
      # a second reset: the reference rebuilds the env with the next seed (reset_wrapper.py:37-45, builder.py:174-187)
      ts = env.reset()
      rec['second_episode_first'] = describe_timestep(ts, env.events())
    finally:
      env.close()
  return rec


def describe_raw_timestep(ts):
  """What a fixture keeps of one dmlab2d-level TimeStep (flat "{i}.RGB", "{i}.REWARD", ..., "WORLD.RGB" observation)."""
  return {'step_type': int(ts.step_type), 'reward': None if ts.reward is None else float(ts.reward),
          'discount': None if ts.discount is None else float(ts.discount),
          'observation': {k: _sha(v) if np.asarray(v).ndim else float(v) for k, v in sorted(ts.observation.items())}}


def record_dmlab2d_stream(name, players, steps=12, seed=SEED):
  """The raw stream the reference's innermost ObservablesWrapper emits (observables_wrapper.py:43-58) on
  observables().dmlab2d while its stack plays `actions_for(...)`: the action dicts its discrete-action and multiplayer
  wrappers hand to dmlab2d, and the flat TimeSteps dmlab2d returns."""
  with reference_stack_on_oracle():
    _, env = _build_reference_env(name, players, seed)
    raw_ts, raw_act = [], []
    env.observables().dmlab2d.timestep.subscribe(raw_ts.append)
    env.observables().dmlab2d.action.subscribe(raw_act.append)
    try:
      acts = actions_for(name, players, env.action_spec()[0].num_values, steps)
      env.reset()
      for t in range(steps):
        env.step([int(a) for a in acts[t]])
    finally:
      env.close()
  assert len(raw_ts) == steps + 1 and len(raw_act) == steps
  return {'substrate': name, 'players': players, 'seed': seed, 'actions': acts.tolist(),
          'raw_actions': [{k: int(v) for k, v in sorted(a.items())} for a in raw_act],
          'raw_timesteps': [describe_raw_timestep(ts) for ts in raw_ts]}


def check_raw_timestep(ts, rec, players, env=None):
  """A dmlab2d-level TimeStep (from lab2d_env.Environment) against one step of a ref_stack_<name>.json fixture; with
  `env`, its events() too."""
  assert int(ts.step_type) == rec['step_type']
  assert (0.0 if ts.discount is None else ts.discount) == rec['discount']
  for i in range(players):
    assert float(ts.observation[f'{i + 1}.REWARD']) == rec['reward'][i]
    for key, value in rec['players'][i].items():
      if key == 'COLLECTIVE_REWARD':  # added by the reference's wrapper stack, not the dmlab2d module
        continue
      obs = ts.observation['WORLD.RGB' if key == 'WORLD.RGB' else f'{i + 1}.{key}']
      assert (_sha(obs) if np.asarray(obs).ndim else float(obs)) == value, (key, i)
  if env is not None:
    events = sorted([n, [float(x) if isinstance(x, np.ndarray) else x.decode() for x in p]] for n, p in env.events())
    assert events == rec['events']
