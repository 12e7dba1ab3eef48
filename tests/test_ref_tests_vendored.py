"""CPU suite: the vendored copies of the reference's test files are still byte-identical to the reference's own.
golden/ref_tests/SHA256SUMS holds the SHA-256 of each file as it is in the reference's tests/ directory
(zombie-einstein/bourse 0.4.0), keyed by its path there."""
import hashlib
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REF_TESTS = os.path.join(HERE, "golden", "ref_tests")
PAIRS = {"test_order_book.py": "test_order_book.py", "test_env.py": "test_step_sim/test_env.py",
         "test_numpy_api.py": "test_step_sim/test_numpy_api.py", "test_agents.py": "test_step_sim/test_agents.py"}


def reference_digests() -> dict:
    with open(os.path.join(REF_TESTS, "SHA256SUMS")) as f:
        return {path: digest for digest, path in (line.split() for line in f if line.strip())}


@pytest.mark.parametrize("ours,theirs", sorted(PAIRS.items()))
def test_vendored_reference_tests_are_unmodified(ours, theirs):
    with open(os.path.join(REF_TESTS, ours), "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == reference_digests()[theirs]
