"""Records tests/golden/ref_pins.json: digests of the oracle's values that tests/test_ref_pins.py compares with the reference's own
shader text.  With the whole reference present (libref.so, libref_b6.so, libref_legacy_b{2,12}.so or the source tree they are built
from) the pins run against it and the file is rewritten only if every test passed.  Without it a recording cannot change a digest: it
only adds the slice digests of values whose digest is unchanged, and fails otherwise.
usage: python tests/golden/make_ref_pins.py [pytest args, e.g. -k legacy]"""
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

if __name__ == "__main__":
    os.environ["RTX_RECORD_REF_PINS"] = "1"
    sys.exit(pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(os.path.dirname(HERE), "test_ref_pins.py")] + sys.argv[1:]))
