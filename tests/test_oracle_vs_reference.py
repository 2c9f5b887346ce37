"""Bit-equality of the oracle with the unmodified reference: its pixels and poses on fixed seeds, stored by
tests/golden/make_goldens.py (the reference's forward under the seed protocol of tests/_cases.py)."""
import numpy as np
import pytest
import torch

import _cases
import _harness


@pytest.fixture
def golden_threads():
    saved = torch.get_num_threads()
    torch.set_num_threads(_cases.GOLDEN_THREADS)
    yield
    torch.set_num_threads(saved)


@pytest.mark.parametrize("name", ["a_small", "a_small_noise", "a_nohier_softplus", "a_lockview_uniform", "b_small", "c_small", "d_small",
                                  "a_hier_softplus", "b_noise_b2", "a_cam_hybrid", "a_cam_hybrid2", "a_cam_truncgauss",
                                  "a_cam_spherical", "s_small", "f_small", "g_small", "h_small"])
def test_oracle_is_bit_exact_with_reference(name, golden_threads):
    case = _cases.CASE_BY_NAME[name]
    gold = np.load(_cases.golden_path(case))
    px_ref, poses_ref = torch.from_numpy(gold["pixels"]), torch.from_numpy(gold["poses"])
    run = _harness.oracle_run(case, keep_stages=False)
    assert torch.equal(run["out"]["pixels"], px_ref), float((run["out"]["pixels"] - px_ref).abs().max())
    assert torch.equal(run["out"]["poses"], poses_ref)
