"""Records the splits a `load_jodie_data` makes of the toy dataset of tests/jodie_utils.py (the events of every split,
the pre-sampled negatives, eval flags and seeds) into jodie_toy_splits.json, which tests/test_jodie_cpu.py compares
this package's loader with.  The file's `source` field names the loader that recorded it.

    TIGER_REFERENCE=<reference checkout> python tests/golden/make_golden_jodie.py   # the reference's own loader
    python tests/golden/make_golden_jodie.py --this-package                         # this package's loader

Record from the reference wherever a checkout of it (yzhang1918/www2023tiger) is at hand: only then does the stored
file tie the loader to the original project.  `--this-package` records today's behaviour of this package, which
catches later changes to the loader but not a difference from the reference that is already there.
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from jodie_utils import reference_splits, summarize_splits, write_toy_dataset   # noqa: E402
from www2023tiger_b200.tiger.data.data_loader import load_jodie_data          # noqa: E402

if __name__ == '__main__':
    this_package = '--this-package' in sys.argv[1:]
    reference = os.environ.get('TIGER_REFERENCE', '')
    if not this_package and not os.path.isdir(os.path.join(reference, 'tiger')):
        sys.exit('set TIGER_REFERENCE to a checkout of the reference (the directory that holds tiger/), '
                 'or pass --this-package')
    with tempfile.TemporaryDirectory() as tmp:
        write_toy_dataset(tmp)
        if this_package:
            res = summarize_splits(load_jodie_data('toy', train_seed=5, root=tmp))
            res['source'] = "this package's load_jodie_data (not the reference's)"
        else:
            res = reference_splits(reference, tmp)
            res['source'] = "the reference's load_jodie_data (yzhang1918/www2023tiger)"
    with open(os.path.join(HERE, 'jodie_toy_splits.json'), 'w') as f:
        json.dump(res, f, separators=(',', ':'))
    print('jodie_toy_splits.json written:', res['source'])
