"""Generates tests/golden/ref_stack_<substrate>.json: what the reference's OWN Python stack (builder.py, wrappers,
Substrate, configs -- imported unmodified from the checkout) returns when the `dmlab2d` module underneath it is
`meltingpot_b200.lab2d_env` on the CPU oracle. See tests/ref_stack.py.

  python tools/make_ref_stack_golden.py
"""
import os
os.environ.setdefault('MELTINGPOT_REFERENCE_ROOT', '/root/reference')  # this tool runs where the checkout is
import json
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import ref_stack  # noqa: E402

for name, players in ref_stack.SUBSTRATES:
  rec = ref_stack.run_reference_stack(name, players)
  flat = rec.pop('flat_settings')
  if name in ('clean_up', 'territory__rooms', 'coins'):  # what builder.py handed to dmlab2d.Lab2d, for the boundary-module tests
    import gzip
    with gzip.GzipFile(os.path.join(ROOT, 'tests', 'golden', f'ref_stack_settings_{name}.json.gz'), 'wb', mtime=0) as f:
      f.write(json.dumps(flat, sort_keys=True).encode())
  path = os.path.join(ROOT, 'tests', 'golden', f'ref_stack_{name}.json')
  with open(path, 'w') as f:
    json.dump(rec, f, separators=(',', ':'))
  print(path, os.path.getsize(path), 'rewards', sum(sum(s['reward']) for s in rec['steps']), 'events', sum(len(s['events']) for s in rec['steps']))

# the raw dmlab2d-level stream (observables().dmlab2d) of the reference's stack, for the flat-view tests
path = os.path.join(ROOT, 'tests', 'golden', 'dmlab2d_stream_clean_up.json')
with open(path, 'w') as f:
  json.dump(ref_stack.record_dmlab2d_stream('clean_up', 7), f, separators=(',', ':'))
print(path, os.path.getsize(path))
