"""Every SQDET_* environment variable the library reads is documented in INTEGRATION.md §5, and
every variable documented there is read: a new switch cannot appear unannounced, and a removed one
cannot linger in the docs."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _code_switches():
  names = set()
  csrc = os.path.join(ROOT, 'squeezedet_b200', 'csrc')
  for path in glob.glob(os.path.join(csrc, '*.cu')) + glob.glob(os.path.join(csrc, '*.cuh')):
    with open(path) as f:
      names.update(re.findall(r'"(SQDET_[A-Z0-9_]+)"', f.read()))
  return names


def _documented_switches():
  with open(os.path.join(ROOT, 'INTEGRATION.md')) as f:
    text = f.read()
  section = re.search(r'^## 5\..*?(?=^## |\Z)', text, re.M | re.S).group(0)
  names = set()
  for line in section.splitlines():
    if line.startswith('| `SQDET_'):
      first_cell = line.split('|')[1]
      names.update(re.findall(r'`(SQDET_[A-Z0-9_]+)`', first_cell))
  return names


def test_env_switches_match_integration_table():
  code = _code_switches()
  assert code, 'no SQDET_* switch found in the sources'
  assert code == _documented_switches()
