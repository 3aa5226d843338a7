"""16-bit storage of the data shard (params.a_storage; dtype codes DNMF_A_F16 / DNMF_A_BF16): the checks that need no
GPU -- validation of the knob, the rejections PyNMF / PyNMFk make before touching the device, and the C-ABI's argument
checks (only the entry points that read A accept the 16-bit codes)."""
import numpy as np
import pytest
import torch

from pydnmfk_b200 import _lib as L
from pydnmfk_b200.pyDNMF import PyNMF, a_storage_dtype


class _Params:
    pass


def _params(**kw):
    p = _Params()
    p.init, p.k, p.p_r, p.p_c, p.grid = 'rand', 4, 1, 1, None
    for key, val in kw.items():
        setattr(p, key, val)
    return p


def test_default_changes_nothing():
    assert a_storage_dtype(None, np.zeros((4, 4), np.float32)) is None
    assert a_storage_dtype(None, np.zeros((4, 4), np.float64)) is None


@pytest.mark.parametrize('fmt,dt', [('float16', torch.float16), ('bfloat16', torch.bfloat16)])
def test_float32_data_is_accepted(fmt, dt):
    assert a_storage_dtype(fmt, np.zeros((4, 4), np.float32)) is dt
    assert a_storage_dtype(fmt, torch.zeros((4, 4), dtype=torch.float32)) is dt


@pytest.mark.parametrize('bad', ['half', 'fp16', 'float32', 16, True])
def test_unknown_format_is_rejected(bad):
    with pytest.raises(ValueError, match='a_storage'):
        a_storage_dtype(bad, np.zeros((4, 4), np.float32))


@pytest.mark.parametrize('data', [np.zeros((4, 4), np.float64), np.zeros((4, 4), np.float16),
                                  torch.zeros((4, 4), dtype=torch.float64),
                                  torch.zeros((4, 4), dtype=torch.float16)])     # a host tensor is not "already on the device"
def test_other_data_dtypes_are_rejected(data):
    with pytest.raises(ValueError, match='a_storage'):
        a_storage_dtype('float16', data)


def test_pynmf_rejects_before_using_a_device():
    with pytest.raises(ValueError, match='a_storage'):
        PyNMF(np.ones((8, 8), np.float64), params=_params(a_storage='float16'))
    with pytest.raises(ValueError, match='nnsvd'):
        PyNMF(np.ones((8, 8), np.float32), params=_params(a_storage='bfloat16', init='nnsvd'))


def test_pynmfk_rejects_the_knob():
    from pydnmfk_b200.pyDNMFk import PyNMFk
    with pytest.raises(ValueError, match='a_storage'):
        PyNMFk(np.ones((8, 8), np.float32), params=_params(a_storage='float16'))


def test_host_rounding_is_nearest_even():
    """PyNMF rounds host data with torch's CPU cast: for float16 that is exactly numpy's astype (ties to even,
    subnormals, overflow to inf)."""
    rs = np.random.RandomState(0)
    x = np.concatenate([rs.rand(100000) * 10.0 ** rs.randint(-9, 6, size=100000),
                        np.float32([0.0, -0.0, 65504.0, 65519.9, 65520.0, 1e-8, 2.0 ** -24, 3 * 2.0 ** -25,
                                    1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 2049.0, 2051.0])]).astype(np.float32)
    got = torch.from_numpy(x).to(torch.float16).numpy()
    with np.errstate(over='ignore'):
        want = x.astype(np.float16)
    assert np.array_equal(got.view(np.uint16), want.view(np.uint16))


A16 = [L.A_F16, L.A_BF16]


def test_codes_match_the_header():
    import os
    import re
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'dnmf.h')).read()
    codes = dict(re.findall(r'#define (DNMF_A_F16|DNMF_A_BF16|DNMF_I64) (\d+)', src))
    assert (int(codes['DNMF_A_F16']), int(codes['DNMF_A_BF16'])) == (L.A_F16, L.A_BF16)
    assert int(codes['DNMF_I64']) not in A16          # the collectives accept DNMF_I64


@pytest.mark.parametrize('dt', A16)
def test_a_reading_entry_points_accept_the_codes(dt):
    """Argument checks pass (the workspace query needs no device); k > DNMF_MAX_K is still refused on these codes."""
    for op in (L.OP_AH, L.OP_WTA, L.OP_KL_UHT, L.OP_KL_WTU, L.OP_RESIDUAL, L.OP_AH_RESIDUAL, L.OP_NNZ):
        assert L.workspace_bytes(op, 4096, 4096, 32, dt) > 0
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_ah', 1, 8, 1, 8, 1, 8, 8, 8, L.MAX_K + 1, dt, 0, None, 0, None)
    assert e.value.status == -2 and 'DNMF_MAX_K' in str(e.value)
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_wta', 1, 8, 1, 8, 1, 8, 8, 8, L.MAX_K + 1, 0, dt, 0, None, 0, None)
    assert e.value.status == -2


@pytest.mark.parametrize('dt', A16)
def test_other_entry_points_reject_the_codes(dt):
    """Factor-only entry points keep rejecting 16-bit codes at argument-check level, with their current message."""
    calls = [
        ('dnmf_gram', (1, 8, 8, 4, 0, 1, dt, None, 0, None)),
        ('dnmf_mu_update_w', (1, 8, 1, 8, 1, 8, 4, 1e-7, dt, None)),
        ('dnmf_mu_update_h', (1, 8, 1, 8, 1, 1, 4, 8, 1e-7, 0, dt, None)),
        ('dnmf_clamp_min', (1, 8, 8, 8, 0.0, dt, None)),
        ('dnmf_colsum', (1, 8, 8, 8, 1, dt, None, 0, None)),
        ('dnmf_normalize', (1, 4, 8, 1, 8, 8, 4, 1, 1e-7, dt, None)),
        ('dnmf_axpby', (1, 1, 1, 1.0, 0.0, 8, dt, None)),
        ('dnmf_hals_h', (1, 8, 1, 8, 1, 1, 4, 8, 1e-7, dt, None)),
        ('dnmf_perturb_uniform', (1, 1, 1, 8, 0.03, dt, None)),
        ('dnmf_scatter_rows', (1, 8, 1, 8, 8, 1, 8, dt, None)),
    ]
    for name, args in calls:
        with pytest.raises(L.DnmfError) as e:
            L.call(name, *args)
        assert e.value.status == -1 and 'dtype must be DNMF_F32 or DNMF_F64' in str(e.value), name
    # the _p updates read fp32 partials: the factor dtype is DNMF_F32, never a 16-bit code
    view = (L.i64 * 4)(1, 32, 1, 0)
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_mu_update_w_p', 1, 8, view, 1, 8, 4, 1e-7, dt, None)
    assert e.value.status == -1
