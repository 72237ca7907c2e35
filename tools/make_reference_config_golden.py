"""Generates tests/golden/ref_config_<substrate>.json.gz: what the reference's Python configs hand the compiler.

For each substrate with a committed blob: the lab2d settings its `lab2d_settings_builder` returns for default roles
(one record per build seed the tests compile with) and the config fields `compiler.compile_settings` and the spec
tests read. tests/reference_configs.py compiles from these records, so the compiler tests run without a checkout.

  MELTINGPOT_REFERENCE_ROOT=<Melting Pot checkout> python tools/make_reference_config_golden.py
"""
import gzip
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from meltingpot_b200 import compiler, substrates  # noqa: E402
from tests import reference_configs  # noqa: E402

# Build seeds the tests compile with, besides the substrate's own BUILD_SEEDS entry.
EXTRA_SEEDS = {'territory__inside_out': [1, 2], 'coins': [1, 2, 3, 4, 5]}


def main():
  if compiler.reference_root() is None:
    raise SystemExit('set MELTINGPOT_REFERENCE_ROOT to a Melting Pot checkout')
  for name, counts in substrates.PRECOMPILED.items():
    players = counts[0]
    config = compiler.load_reference_config(name)
    roles = ('default',) * players
    seeds = [substrates.BUILD_SEEDS.get(name)] + EXTRA_SEEDS.get(name, [])
    settings = {}
    for seed in seeds:
      state = random.getstate()
      try:
        if seed is not None:
          random.seed(seed)
        settings[str(seed)] = compiler._plain(config.lab2d_settings_builder(roles=roles, config=config))  # pylint: disable=protected-access
      finally:
        random.setstate(state)
    rec = {
        'substrate': name, 'players': players,
        'config': {
            'action_set': [dict(a) for a in compiler._plain(config.action_set)],  # pylint: disable=protected-access
            'individual_observation_names': list(config.individual_observation_names),
            'global_observation_names': list(config.global_observation_names),
            'valid_roles': sorted(config.valid_roles),
            'default_player_roles': list(config.default_player_roles),
            'rgb_shape': list(config.timestep_spec.observation['RGB'].shape),
            'world_rgb_shape': list(config.timestep_spec.observation['WORLD.RGB'].shape),
            'num_actions': int(config.action_spec.num_values),
        },
        'settings_by_build_seed': settings,
    }
    path = reference_configs.path(name)
    with gzip.GzipFile(path, 'wb', mtime=0) as f:
      f.write(json.dumps(rec).encode())  # key order is data: it orders action_set fields
    # The recorded settings must compile to exactly what the checkout's configs compile to.
    for seed in seeds:
      want = compiler.compile_substrate(name, roles, build_seed=seed)
      assert reference_configs.compile_recorded(name, build_seed=seed) == want, (name, seed)
    print(path, os.path.getsize(path))


if __name__ == '__main__':
  main()
