"""Host-side checks of the joint posterior sampler: the Philox4x64-10 stream its normals come from, and the
ThompsonSampling acquisition's value semantics.  The device path is in test_posterior_sample_gpu.py."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sample_reference as ref  # noqa: E402


def test_philox_known_answer():
    assert ref.philox4x64_10((1, 0, 0, 0), (12345, 0)) == [
        0xa5792c0a0ed6a560, 0xc63666ba8b756514, 0xc953e311f634209d, 0x28db5404d83fac91]


@pytest.mark.parametrize("seed,s", [(12345, 0), (0, 7), (2 ** 64 - 1, 4095), (0xDEADBEEF, 1)])
def test_numpy_philox_blocks_are_counter_j_plus_one(seed, s):
    w = ref.philox_words(seed, s, 9)
    for j in range(9):
        assert [int(v) for v in w[j]] == ref.philox4x64_10((j + 1, 0, 0, 0), (seed, s)), j


def test_normals_follow_the_box_muller_recipe():
    m = 10
    w = ref.philox_words(3, 5, 3)
    z = ref.philox_normals(3, 5, m)
    for i in range(m):
        j, q = divmod(i, 4)
        u = [((int(w[j][a]) >> 11) + 0.5) * 2.0 ** -53 for a in range(4)]
        r = np.sqrt(-2 * np.log(u[0 if q < 2 else 2]))
        a = 2 * np.pi * u[1 if q < 2 else 3]
        assert abs(z[i] - (r * np.cos(a) if q % 2 == 0 else r * np.sin(a))) <= 4e-16 * max(1.0, abs(z[i]))
    # a draw's normals do not depend on how many candidates are asked for
    assert np.array_equal(ref.philox_normals(3, 5, 7), z[:7])
    Z = ref.normals(11, 64, 4001)
    assert abs(Z.mean()) < 0.01 and abs(Z.var() - 1) < 0.01 and abs(np.corrcoef(Z[0], Z[1])[0, 1]) < 0.06


def test_thompson_sampling_value_semantics():
    import abo_b200 as abo
    ts = abo.ThompsonSampling(7)
    assert abo.update(ts, np.zeros(3), None) == abo.ThompsonSampling(8)
    assert ts.update(None, None).update(None, None).seed == 9
    c = abo.copy(ts)
    assert c == ts and c is not ts
    with pytest.raises(TypeError):
        ts.value_and_grad(None, np.zeros((2, 2)))
    assert not ts.has_gradient and abo.ExpectedImprovement(0.0, 1.0).has_gradient
    with pytest.raises(Exception):
        ts.seed = 3                                   # frozen
    for name in ("posterior_sample", "thompson_batch", "ThompsonSampling"):
        assert hasattr(abo, name), name


def test_sampler_signature_is_checked_with_its_unsigned_seed():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("check_ffi", os.path.join(root, "tools", "check_ffi_signatures.py"))
    chk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(chk)
    protos = chk.c_prototypes()
    assert protos["abo_gp_posterior_sample"][1] == ["ptr:void", "ptr:double", "int64", "int64", "uint64", "double",
                                                     "ptr:double", "ptr:int64", "ptr:double", "ptr:double"]
    assert "abo_gp_posterior_sample" in {c[0] for c in chk.julia_ccalls()}
    broken = dict(protos)
    broken["abo_gp_posterior_sample"] = ("int32", protos["abo_gp_posterior_sample"][1][:4] + ["int64"] +
                                         protos["abo_gp_posterior_sample"][1][5:])
    _, errs = chk.check_julia(broken)
    assert any("abo_gp_posterior_sample" in e and "argument 5" in e for e in errs)
