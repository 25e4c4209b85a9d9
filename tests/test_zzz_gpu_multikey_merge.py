"""GPU variants of the multi-key merge checks (``tests/test_fifth_batch.py::_sixth_batch_checks``: both front doors
against ``tests/golden/ext6_multikey_merge.npz`` from the unmodified reference) and of the float-key groupby checks
(``_seventh_batch_checks``: the Modin front door against ``ext7_float_keys.npz``).

Kept in a file of its own that sorts LAST: the feature was written after the round's GPU minutes were spent, so unlike
everything else under ``-m gpu`` it has run on the numpy device double only (it is composed from kernels that are
verified on the B200 -- the column maps of ``groupkeys.pack``, the join tables, the gathers -- but the composition is
not), and a failure here must not stop a ``pytest -x`` run before the verified tests.
"""

import os

import pytest

from tests.test_alignment_merge import REF, _modin
from tests.test_fifth_batch import _seventh_batch_checks, _sixth_batch_checks

UNTRIED = pytest.mark.xfail(strict=False, reason="written after the round's last GPU minute: has run on the numpy "
                           "device double only, never on a B200 (an XPASS is the first hardware evidence)")


@pytest.mark.gpu
@UNTRIED
def test_multi_key_merge_on_b200():
    import modin_b200.pandas as bpd

    _sixth_batch_checks(bpd)
    if os.path.isdir(os.path.join(REF, "modin")):
        _sixth_batch_checks(_modin())


@pytest.mark.gpu
@UNTRIED
def test_float_key_groupby_on_b200():
    if not os.path.isdir(os.path.join(REF, "modin")):
        pytest.skip("oracle/_ref (the unmodified reference) is not installed on this box")
    _seventh_batch_checks(_modin())


@pytest.mark.gpu
@UNTRIED
def test_groupby_level_on_b200():
    if not os.path.isdir(os.path.join(REF, "modin")):
        pytest.skip("oracle/_ref (the unmodified reference) is not installed on this box")
    from tests.test_modin_plugin import _level_scenarios

    _level_scenarios(_modin())
