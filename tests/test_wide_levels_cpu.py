"""Levels wider than 192 channels, CPU side: the 1024-channel bound of the calls and of the C ABI, checked before any
launch, and the oracle's own fp64 round trip at the L6 / L7 geometries the GPU tests compare against."""
import pytest
import torch

import normalizing_flow as nf
from normalizing_flow import _native as N
from oracle import glow_oracle as O

FAKE = 256        # a non-null device address: a call that got past its checks would launch on it


def test_glow_wider_than_1024_is_refused_before_init():
    """L8 on RGB has a 1536-channel final level: the constructor accepts it (a checkpoint still loads), the calls raise
    ValueError before the data-dependent initialisation touches a parameter."""
    flow = nf.Glow(3, 8, 1)
    sd = {k: v.clone() for k, v in flow.state_dict().items()}
    flow.load_state_dict(sd)
    x = torch.randn(1, 3, 256, 256)
    with pytest.raises(ValueError, match="1536 channels"):
        flow.transform(x, torch.zeros(1), torch.zeros(1))
    with pytest.raises(ValueError, match="1536 channels"):
        flow.invert([torch.zeros(1, 1536, 1, 1)])
    with pytest.raises(ValueError, match="1536 channels"):
        flow.sample([torch.zeros(1, 1536, 1, 1)])
    with pytest.raises(ValueError, match="1536 channels"):
        flow.invert_with_density([torch.zeros(1, 1536, 1, 1)], 1.0, torch.zeros(1))
    assert all(int(m.is_initialized) == 0 for m in flow.modules() if isinstance(m, nf.ActNorm))
    assert all(torch.equal(v, sd[k]) for k, v in flow.state_dict().items())
    nf.Glow(3, 7, 1)            # 768 channels: no refusal at construction either


@pytest.mark.parametrize("make,shape", [(lambda: nf.InvConv2d(1536), (1, 1536, 1, 1)),
                                        (lambda: nf.ActNorm(1536), (1, 1536, 1, 1)),
                                        (lambda: nf.StepFlow(1536), (1, 1536, 1, 1)),
                                        (lambda: nf.Split(1536), (1, 1536, 1, 1))])
def test_modules_wider_than_1024_are_refused(make, shape):
    mod = make()
    with pytest.raises(ValueError, match="1536 channels"):
        mod.transform(torch.zeros(shape), torch.zeros(1), torch.zeros(1))
    half = (shape[0], shape[1] // 2) + shape[2:] if isinstance(mod, nf.Split) else shape
    with pytest.raises(ValueError, match="1536 channels"):
        mod.invert(torch.zeros(half))


def test_glow_block_wider_than_1024_is_refused():
    blk = nf.GlowBlock(in_channels=384, K=1)
    with pytest.raises(ValueError, match="1536 channels"):
        blk.transform(torch.zeros(1, 384, 2, 2), torch.zeros(1), torch.zeros(1))
    with pytest.raises(ValueError, match="1536 channels"):
        blk.invert(torch.zeros(1, 768, 1, 1))


def test_abi_rejects_1025_channels_before_any_launch():
    rc = N.lib.nfdpm_channel_mix(None, None, None, None, 1, 1025, 1, 1025, 1025, None)
    assert rc != 0 and b"null pointer" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_channel_mix(FAKE, FAKE, FAKE, FAKE, 1, 1025, 1, 1025, 1025, None)
    assert rc != 0 and b"C=1025 > 1024" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_mix_bwd(None, 1025, None, 0, None, 1025, None, None, 1025, None, 1, 1025, 1, 1, None)
    assert rc != 0 and b"null pointer" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_mix_bwd(FAKE, 1025, None, 0, FAKE, 1025, FAKE, FAKE, 1025, FAKE, 1, 1025, 1, 1, None)
    assert rc != 0 and b"C=1025 > 1024" in N.lib.nfdpm_last_error_string()
    item = N.MixGradItem(part=FAKE, B=1, C=1025, weight=None, scale=None, bias=None, winv=FAKE, dld_sum=None, P=1.0,
                         pad_=0, d_weight=None, d_scale=None, d_bias=FAKE, scratch=FAKE)
    arr = (N.MixGradItem * 1)(item)
    rc = N.lib.nfdpm_mix_inv_param_grad(arr, 1, None)
    assert rc != 0 and b"C=1025 > 1024" in N.lib.nfdpm_last_error_string()


def test_mix_bwd_tiles_of_wide_levels():
    """One partial row per image above 192 channels; the single-pass kernel's tiles below are unchanged."""
    assert [N.mix_bwd_tiles(C, 4, 4) for C in (193, 384, 768, 1024)] == [1] * 4
    assert N.mix_bwd_tiles(384, 64, 64) == 1
    assert N.mix_bwd_tiles(12, 64, 64) == 16 and N.mix_bwd_tiles(192, 4, 4) == 1


@pytest.mark.parametrize("L,K,S", [(6, 1, 64), (7, 1, 128)])
def test_oracle_fp64_round_trip(L, K, S):
    """The oracle the GPU tests compare against inverts its own transform at these depths (384 / 768 channels)."""
    sd, _ = O.seeded_state(3, L, K, 7)
    sd = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    x = O.seeded_input((2, 3, S, S), 8).double()
    ld, lp = torch.zeros(2, dtype=torch.float64), torch.zeros(2, dtype=torch.float64)
    with torch.no_grad():
        zs, ld, lp = O.glow_transform(sd, x, L, K, ld, lp)
        assert [tuple(z.shape[1:]) for z in zs] == [tuple(s) for s in O.output_shapes(L, 3, S)]
        assert max(z.shape[1] for z in zs) == 2 ** (L + 1) * 3
        xr = O.glow_invert(sd, zs, L, K)
    assert bool(torch.isfinite(ld).all() and torch.isfinite(lp).all())
    # not exact: the reference's coupling multiplies by s and divides by s + 1e-6, an asymmetry that grows with the
    # number of steps (measured 1.2e-5 at L6, 6.6e-4 at L7 with these weights)
    assert float((xr - x).abs().max()) < (1e-4 if L == 6 else 1e-3)
