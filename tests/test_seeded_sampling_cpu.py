"""CPU checks of seeded sampling: the numpy oracle of the draw contract against Random123's known-answer vectors and the
normal distribution, the argument checks of the three _ex entry points (before any launch) and of the Python keywords."""
import numpy as np
import pytest
import torch
from scipy import stats

import normalizing_flow as nf
from normalizing_flow import _engine as E
from normalizing_flow import _native as N
import philox_oracle as PO


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(w) for w in PO.philox4x32_10(ctr, key)) == want


def test_uniforms_stay_inside_the_unit_interval():
    w = np.array([0, 255, 256, 0x7fffff00, 0xffffff00, 0xffffffff], dtype=np.uint32)
    u = PO.uniforms(w)
    assert u.dtype == np.float32
    assert u[0] == np.float32(2.0 ** -25) and u[1] == u[0] and u[2] == np.float32(1.5 * 2.0 ** -24)
    assert bool((u > 0).all()) and bool((u <= 1).all())


def test_oracle_normals_are_standard_normal():
    n = 1 << 20
    seeds = np.array([0, 1, -1, 2 ** 62 + 12345], dtype=np.int64)
    z = PO.normals(seeds, 3, n // 4).reshape(-1)
    assert z.size == n and np.isfinite(z).all()
    ks = stats.kstest(z, "norm")
    assert ks.pvalue > 1e-3, ks
    assert abs(z.mean()) <= 5.0 / np.sqrt(n)
    assert abs(z.var() - 1.0) <= 5.0 * np.sqrt(2.0 / n)


def test_oracle_draw_is_a_function_of_seed_stream_and_element():
    a = PO.normals(np.array([7, 8], dtype=np.int64), 0, 37)
    b = PO.normals(np.array([8], dtype=np.int64), 0, 41)
    assert np.array_equal(a[1], b[0, :37])                          # neither the batch nor the tensor size matters
    assert not np.array_equal(a[0], a[1])
    assert not np.array_equal(PO.normals(np.array([7]), 1, 37), a[:1])          # the draw site does


def _err():
    return N.lib.nfdpm_last_error_string()


def test_ex_entry_points_check_arguments_before_any_launch():
    # (h, ldh, bias, logs, eps, seeds, stream_id, T, temp_b, eps_out, y, ybs, B, C, H, W, stream)
    sp = N.lib.nfdpm_split_prior_sample_ex
    assert sp(None, 0, None, None, 8, None, 0, 1.0, None, None, None, 8, 1, 4, 2, 2, None) != 0
    assert b"nfdpm_split_prior_sample_ex: null pointer" in _err()
    assert sp(None, 0, None, None, 8, 8, 0, 1.0, None, None, 8, 8, 1, 4, 2, 2, None) != 0
    assert b"exactly one of eps / seeds" in _err()
    assert sp(None, 0, None, None, None, None, 0, 1.0, None, None, 8, 8, 1, 4, 2, 2, None) != 0
    assert b"exactly one of eps / seeds" in _err()
    assert sp(None, 0, None, None, 8, None, 3, 1.0, None, None, 8, 8, 1, 4, 2, 2, None) != 0
    assert b"stream_id / eps_out need seeds" in _err()
    assert sp(None, 0, None, None, 8, None, 0, 1.0, None, 8, 8, 8, 1, 4, 2, 2, None) != 0
    assert b"stream_id / eps_out need seeds" in _err()
    assert sp(None, 0, None, None, None, 8, 0, 1.0, None, None, 8, 8, 1, 3, 2, 2, None) != 0
    assert b"nfdpm_split_prior_sample_ex: bad shape" in _err()
    assert sp(None, 0, None, None, None, 8, 0, 1.0, None, None, 8, 8, 0, 4, 2, 2, None) != 0
    assert b"nfdpm_split_prior_sample_ex: bad shape" in _err()
    assert sp(8, 2, None, None, None, 8, 0, 1.0, None, None, 8, 8, 1, 4, 2, 2, None) != 0
    assert b"learned prior needs bias/logs/ldh" in _err()
    assert sp(None, 0, None, None, None, 8, 0, 1.0, None, None, 8, 8, 1, 2, 65536, 65537, None) != 0
    assert b"more than 2^32" in _err()
    # (eps, seeds, stream_id, bias, logs, T, temp_b, eps_out, out, B, C, P, stream)
    gs = N.lib.nfdpm_gauss_sample_const_ex
    assert gs(None, 8, 0, None, None, 1.0, None, None, None, 1, 4, 4, None) != 0
    assert b"nfdpm_gauss_sample_const_ex: null pointer" in _err()
    assert gs(8, 8, 0, None, None, 1.0, None, None, 8, 1, 4, 4, None) != 0
    assert b"exactly one of eps / seeds" in _err()
    assert gs(None, None, 0, None, None, 1.0, None, None, 8, 1, 4, 4, None) != 0
    assert b"exactly one of eps / seeds" in _err()
    assert gs(8, None, 0xFFFFFFFF, None, None, 1.0, None, None, 8, 1, 4, 4, None) != 0
    assert b"stream_id / eps_out need seeds" in _err()
    assert gs(None, 8, 0, 8, None, 1.0, None, None, 8, 1, 4, 4, None) != 0
    assert b"bias/logs must both be set" in _err()
    assert gs(None, 8, 0, None, None, 1.0, None, None, 8, 1, 4, 0, None) != 0
    assert b"nfdpm_gauss_sample_const_ex: bad shape" in _err()
    # (dz, dz_bs, eps, T, temp_b, dlp, h, ldh, bias, logs, dh, dpar, B, C, H, W, stream)
    sb = N.lib.nfdpm_split_sample_bwd_ex
    assert sb(8, 0, None, 1.0, 8, None, None, 0, 8, 8, None, 8, 1, 2, 1, 1, None) != 0
    assert b"nfdpm_split_sample_bwd_ex: null pointer" in _err()
    assert sb(8, 0, 8, 1.0, 8, None, 8, 1, 8, 8, 8, 8, 1, 2, 1, 1, None) != 0
    assert b"needs dh with ldh >= C" in _err()
    assert sb(8, 0, 8, 1.0, 8, None, None, 0, 8, 8, None, 8, 1, 3, 1, 1, None) != 0
    assert b"nfdpm_split_sample_bwd_ex: bad shape" in _err()


def test_sampling_keywords_are_checked_before_any_launch():
    before = N.launch_count
    assert E.sampling_inputs(0.7, None, 4, "cpu") == (0.7, None)
    with pytest.raises(RuntimeError, match="CUDA"):
        E.sampling_inputs(1.0, torch.zeros(4, dtype=torch.int64), 4, "cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        E.sampling_inputs(torch.ones(4), None, 4, "cpu")
    with pytest.raises(TypeError, match="seeds"):
        E.sampling_inputs(1.0, [1, 2, 3, 4], 4, "cpu")
    g = nf.Glow(3, 2, 1)
    lat = [torch.zeros(2, 48, 2, 2)]
    with pytest.raises(RuntimeError, match="CUDA"):
        g.invert(lat, 1.0, seeds=torch.zeros(2, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="CUDA"):
        nf.GaussianPrior(48).sample((2, 48, 2, 2), torch.ones(2), seeds=torch.zeros(2, dtype=torch.int64))
    assert N.launch_count == before
