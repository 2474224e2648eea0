"""Record tests/golden/oracle_bitwise.npz: the outputs that tests/test_oracle.py compares bit for bit with the reference's
own C library (oracle/_ref/libbhmm_ref.so), on that test's seeded inputs.

    python tests/golden/make_oracle_bitwise.py reference    # from the reference library (needs `make -C oracle ref`)
    python tests/golden/make_oracle_bitwise.py port         # from the C restatement, oracle/hmm_oracle.c

The committed file was recorded with `port`, because no reference checkout was at hand when it was made.  That gives the
reference library's outputs as long as oracle/hmm_oracle.c is the code that test_port_bitwise_equals_reference_library
pinned bit for bit to the library on these inputs: hmm_oracle.c is unchanged since commit 60a9040, which added it together
with that test.  test_reference_library_reproduces_stored_outputs checks the file against the library wherever the library
is built; re-record with `reference` there if it ever fails.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from oracle import oracle as orc  # noqa: E402
from test_oracle import bitwise_cases, bitwise_outputs  # noqa: E402


def main(kind):
    orc.build(ref=False)
    o = orc.Oracle(kind)
    out = {'recorded_with': np.array(kind)}
    for k, case in enumerate(bitwise_cases()):
        out.update(bitwise_outputs(o, case, k))
    path = os.path.join(HERE, 'oracle_bitwise.npz')
    np.savez_compressed(path, **out)
    print('%s: %d arrays, %d bytes' % (path, len(out), os.path.getsize(path)))


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else 'reference')
