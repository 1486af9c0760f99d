"""Record ``reference_contracts.npz``: what the reference's own functions return on the inputs of the tests that compare
the drop-ins with them.

  test_host_module.py::test_load_data_matches_reference                        loadData
  test_host_module.py::test_helpers_match_reference                            doyToMonth, applyScaling, genEmptyArrays
  test_host_module.py::test_drift_regridders_match_reference                   utils.int_smooth_drifts_v2/v3
  test_host_module.py::test_per_function_operators_have_the_reference_contracts  the eight functions of calcBudget
  test_final_products.py::test_oracle_matches_reference_writer                 utils.OutputSnowModelFinal

Those tests used to run the reference verbatim (``oracle/ref_loader.py``), which needs the reference's source tree next
to this repository.  The drop-ins they check (``nesosim_b200/NESOSIM.py``, ``nesosim_b200/drift_smoothing.py``,
``oracle/final_products.py``) were identical to the reference on every one of these inputs, and this script records
their outputs at that revision, so the file holds the reference's values.  The tests' own functions build the inputs
and collect the outputs, so the file and the tests cannot drift apart.  Re-record only after comparing the drop-ins
with the reference again:   python tests/golden/make_reference_contracts.py
"""
import os
import sys
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import test_final_products as TF      # noqa: E402
import test_host_module as TH         # noqa: E402


def main():
    out = {}
    TH.N.VERBOSE = False
    with tempfile.TemporaryDirectory() as root:
        out.update(TH.load_data_outputs(TH.load_data_tree(root)))
    out.update(TH.helper_outputs())
    out.update(TH.drift_regridder_outputs())
    with pytest.MonkeyPatch.context() as mp:
        TH.use_stand_in_ops(mp)
        out.update(TH.operator_outputs())
    out.update(TF.writer_digests())
    path = os.path.join(HERE, TH.CONTRACTS)
    np.savez_compressed(path, **out)
    print(TH.CONTRACTS, len(out), "arrays,", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
