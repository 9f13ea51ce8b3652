"""Generator of tests/golden/reference_record.npz:  python tests/golden/make_reference_record.py

The tests in test_circles_host.py, test_gridfit_host.py, test_oracle_geometry.py,
test_oracle_paths.py (stitch, flat-field) and test_reader_host.py (extract_paths) compare this
package with functions of the reference (FordyceLab/magnify), loaded in place by
oracle/_refload.py when a checkout of it is present.  Those comparisons assert equality, bit for
bit, or within the stated rtol for the grid line fits.  The reference is not part of this
repository, so this file records this package's side of each comparison (each module's
`record()`), written at a commit where every one of the comparisons passed against the
reference.  The tests check this package against the record always, and the reference against
the same record whenever it is present (MAGNIFY_REFERENCE_ROOT).
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
for path in (TESTS, os.path.dirname(TESTS)):
    if path not in sys.path:
        sys.path.insert(0, path)

import test_circles_host  # noqa: E402
import test_gridfit_host  # noqa: E402
import test_oracle_geometry  # noqa: E402
import test_oracle_paths  # noqa: E402
import test_reader_host  # noqa: E402


def main():
    out = {}
    for module in (test_circles_host, test_gridfit_host, test_oracle_geometry, test_oracle_paths):
        out.update(module.record())
    with tempfile.TemporaryDirectory(prefix="mgb_paths_") as tmpdir:
        out.update(test_reader_host.record(tmpdir))
    path = os.path.join(HERE, "reference_record.npz")
    np.savez_compressed(path, **out)
    print(path, len(out), "arrays,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
