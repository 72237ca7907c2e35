"""TEST INFRASTRUCTURE: the reference's substrate configs as recorded in tests/golden/ref_config_<substrate>.json.gz
(tools/make_reference_config_golden.py): the lab2d settings each config builder returned for default roles, per build
seed, and the config fields the compiler reads. Tests compile from these records instead of a reference checkout."""

import copy
import functools
import gzip
import json
import os
import types

from meltingpot_b200 import compiler

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def path(name):
  return os.path.join(ROOT, 'tests', 'golden', f'ref_config_{name}.json.gz')


@functools.lru_cache(maxsize=None)
def _record(name):
  with gzip.open(path(name)) as f:
    return json.loads(f.read().decode())


def config(name):
  """The recorded config fields (action_set, observation names, roles, spec shapes) as attributes."""
  return types.SimpleNamespace(**_record(name)['config'])


def settings(name, build_seed=None):
  """A fresh copy of the settings the config builder returned for default roles with this build seed."""
  return copy.deepcopy(_record(name)['settings_by_build_seed'][str(build_seed)])


def compile_recorded(name, build_seed=None):
  """What `compiler.compile_substrate(name, default roles, build_seed=...)` returns, from the recorded config."""
  return compiler.compile_settings(settings(name, build_seed), config(name), build_seed)
