#!/usr/bin/env python
"""Regenerates tests/golden/reference_digests.json: what the reference tools and functions give in
the tests that compare with them (tests/refgold.py), as sha256 digests or, for the command-line
errors, the exit status, stdout and stderr themselves.

    python tests/golden/make_reference_digests.py               # from the reference (oracle/_ref)
    python tests/golden/make_reference_digests.py --from-oracle # from this repository's side

With oracle/_ref built, the values recorded are the reference's own.  --from-oracle records the
values of this repository's side of each comparison instead; that is the reference's only where
those comparisons last passed against the reference binaries with the same inputs and the same
code.  The committed table was made that way: oracle/dx_oracle.c is unchanged since it was pinned
to the reference tools on these cases and fuzz seeds (DESIGN.md section 2), and the command-line
tools and libdexcompat matched the reference on these calls."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import orc          # noqa: E402

TESTS = ["tests/test_oracle_vs_ref.py", "tests/test_oracle_fuzz.py", "tests/test_oracle_functions.py",
         "tests/test_cli_errors.py::test_tool_errors_match_the_reference",
         "tests/test_compat_errors.py::test_path_helpers_match_the_reference",
         "tests/test_compat_errors.py::test_line_reader_matches_the_interactive_reference",
         "tests/test_compat_errors.py::test_coding_header_io_matches_the_reference_functions",
         "tests/test_gpu_dbapi.py::test_dex2db_write_order_and_load_qventry"]         # needs a GPU


def main():
    if not orc.have_ref() and "--from-oracle" not in sys.argv:
        sys.exit("oracle/_ref is not built (make -C oracle ref); see --from-oracle")
    out = os.path.join(HERE, "reference_digests.json")
    tmp = out + ".new"
    if os.path.exists(tmp):
        os.remove(tmp)
    env = dict(os.environ, DX_RECORD_REFERENCE=tmp)
    if "--from-oracle" in sys.argv:
        env["DX_RECORD_FROM_THIS_REPOSITORY"] = "1"
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *TESTS],
                          cwd=ROOT, env=env)
    os.replace(tmp, out)
    print("wrote", out)


if __name__ == "__main__":
    main()
