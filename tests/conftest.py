import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)


def pytest_configure(config):
  config.addinivalue_line('markers', 'gpu: needs a real B200 (run with -m gpu)')


@pytest.fixture(scope='session')
def clean_up_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('clean_up')


@pytest.fixture(scope='session')
def oracle():
  from oracle import binding
  binding.build()
  return binding


@pytest.fixture(scope='session')
def clean_river_blob():
  with open(os.path.join(ROOT, 'tests', 'golden', 'clean_up_clean_river__7p.mpb'), 'rb') as f:
    return f.read()


@pytest.fixture(scope='session')
def commons_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('commons_harvest__open', ('default',) * 7)


@pytest.fixture(scope='session')
def commons16_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('commons_harvest__open', ('default',) * 16)


@pytest.fixture(scope='session')
def territory_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('territory__rooms', ('default',) * 9)


@pytest.fixture(scope='session')
def territory_open_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('territory__open', ('default',) * 9)


@pytest.fixture(scope='session')
def commons_closed_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('commons_harvest__closed', ('default',) * 7)


@pytest.fixture(scope='session')
def territory_inside_out_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('territory__inside_out', ('default',) * 5)


@pytest.fixture(scope='session')
def commons_partnership_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('commons_harvest__partnership', ('default',) * 7)


@pytest.fixture(scope='session')
def coins_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('coins', ('default',) * 2)


@pytest.fixture(scope='session')
def coop_mining_blob():
  from meltingpot_b200 import substrates
  return substrates.load_blob('coop_mining', ('default',) * 6)
