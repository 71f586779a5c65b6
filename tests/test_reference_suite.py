"""This package against the original Spriteworld package (CPU tier).

tests/reference_probes.py calls the public API both packages share with seeded inputs;
tests/golden/reference_probes.npz holds what the original package returned (written by
tests/golden/make_golden.py).  Here the same probes run against spriteworld_b200 and every record
must equal the original's.  The probes of modules that drive the engine (tasks, action spaces, the
PIL renderer, configs, environments, the gym wrapper) run on the oracle-backed double
(tests/oracle_engine.py): what is under test is this package's host layer -- task / action
compilation, scene packing, the plugin protocol, the config modules -- the device arithmetic has
its own parity tests (`-m gpu`).
"""
import importlib
import json
import math
import os

import numpy as np
import pytest

from tests import reference_probes as probes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_probes.npz')


def _ours(name):
  return importlib.import_module('spriteworld_b200.' + name)


def _same(h, w):
  """Decoded records: floats to 1e-6 relative (the Clustering reward matches the reference to
  1e-6, oracle/README.md), everything else exactly."""
  if isinstance(w, float) or isinstance(h, float):
    return (type(h) in (int, float) and type(w) in (int, float) and
            (h == w or math.isclose(h, w, rel_tol=1e-6, abs_tol=1e-12) or (h != h and w != w)))
  if isinstance(w, list):
    return isinstance(h, list) and len(h) == len(w) and all(_same(a, b) for a, b in zip(h, w))
  if isinstance(w, dict):
    return isinstance(h, dict) and sorted(h) == sorted(w) and all(_same(h[k], w[k]) for k in w)
  return type(h) is type(w) and h == w


def _compare(name):
  blob = np.load(GOLDEN, allow_pickle=False)
  want = {k.split(':', 1)[1]: blob[k] for k in blob.files if k.startswith(name + ':')}
  have = probes.run(name, _ours)
  assert want and sorted(have) == sorted(want)
  bad = []
  for key, w in sorted(want.items()):
    h = have[key]
    if w.dtype.kind == 'U':
      ok = isinstance(h, str) and _same(json.loads(h), json.loads(str(w)))
    else:
      ok = isinstance(h, np.ndarray) and h.dtype == w.dtype and np.array_equal(h, w)
    if not ok:
      bad.append('%s: %.300s != %.300s' % (key, h, w))
  assert not bad, '\n'.join(bad)


@pytest.mark.parametrize('name', sorted(probes.HOST))
def test_host_modules_match_the_reference(name):
  _compare(name)


@pytest.mark.parametrize('name', sorted(probes.ENGINE))
def test_engine_modules_match_the_reference_on_oracle_engine(monkeypatch, name):
  from tests import oracle_engine
  oracle_engine.install(monkeypatch)
  _compare(name)


def test_public_surface_of_the_reference_is_present():
  """Every public class, function, method and constructor parameter of the reference's modules
  on and around the path exists under the same name in spriteworld_b200 (demo_ui / run_demo /
  example_run_loop are out of scope, DESIGN.md section 8)."""
  import inspect
  surface = json.loads(str(np.load(GOLDEN, allow_pickle=False)['surface']))
  assert surface
  missing = []
  for m, name, attrs, params in surface:
    ours = _ours(m)
    if not hasattr(ours, name):
      missing.append('%s.%s' % (m, name))
      continue
    mine = getattr(ours, name)
    missing += ['%s.%s.%s' % (m, name, a) for a in attrs if not hasattr(mine, a)]
    if params is not None:
      have = [p for p in inspect.signature(mine.__init__ if inspect.isclass(mine) else mine).parameters
              if p != 'self']
      if params != have[:len(params)]:
        missing.append('%s.%s(%s)' % (m, name, ', '.join(params)))
  assert not missing, missing
