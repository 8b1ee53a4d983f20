"""Writes tests/golden/sequence_cases.json from the reference's own SequenceAdder test vectors
(`acme/adders/reverb/sequence_test.py:25-181`, TEST_CASES).  The reference module cannot be imported here (it needs
reverb / tensorflow), so the TEST_CASES literal is cut out of the file and evaluated with this repo's dm_env shim, which
builds the same TimeSteps.  Needs a checkout of the reference:  python tools/make_sequence_golden.py <reference checkout>"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from acme_b200 import dm_env  # noqa: E402

SRC = os.path.join('acme', 'adders', 'reverb', 'sequence_test.py')


def main(reference_root):
  text = open(os.path.join(reference_root, SRC)).read()
  a = text.index('TEST_CASES = [')
  b = text.index('\n]\n', a) + 3
  ns = {'dm_env': dm_env}
  exec(text[a:b], ns)  # the literal only calls dm_env.restart / transition / termination
  out = []
  for c in ns['TEST_CASES']:
    steps = []
    for action, ts in c['steps']:
      steps.append(dict(action=action, kind='term' if ts.last() else 'mid', reward=float(ts.reward),
                        discount=float(ts.discount), observation=int(ts.observation)))
    out.append(dict(name=c['testcase_name'], sequence_length=c['sequence_length'], period=c['period'],
                    pad_end_of_episode=c.get('pad_end_of_episode', True), first=int(c['first'].observation), steps=steps,
                    expected=[[[int(o), int(a_), float(r), float(d), bool(s), list(e)] for (o, a_, r, d, s, e) in seq]
                              for seq in c['expected_sequences']]))
  path = os.path.join(ROOT, 'tests', 'golden', 'sequence_cases.json')
  json.dump(out, open(path, 'w'), indent=1)
  print('wrote', path, len(out), 'cases')


if __name__ == '__main__':
  main(sys.argv[1])
