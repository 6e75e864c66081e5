"""CPU: the shared-memory plans of the bf16-latent (DVQ_Z_BF16) tcgen05 VQ kernels, through the host-only
dvq_debug_tc_layout_ex.  Every bf16 plan fits the 227 KB budget, the kernel variant is the one the fp32 call
gets (it is chosen on (N, K, D) alone), and flags = 0 reproduces dvq_debug_tc_layout / dvq_debug_tc_pair_layout."""
import ctypes
import os

import pytest

KS = (512, 1024, 2048, 4096, 8192, 16384)
DS = (16, 32, 64, 128, 256, 512)
NS = (129, 1 << 20, 1 << 24)


def _ex(N, K, D, flags):
    from dvq import _cabi
    out = (ctypes.c_int * 8)()
    _cabi.check(_cabi.lib.dvq_debug_tc_layout_ex(N, K, D, flags, out), "dvq_debug_tc_layout_ex")
    return list(out)


def _old(N, K, D):
    from dvq import _cabi
    single, pair = (ctypes.c_int * 8)(), (ctypes.c_int * 8)()
    _cabi.check(_cabi.lib.dvq_debug_tc_layout(K, D, single), "dvq_debug_tc_layout")
    _cabi.check(_cabi.lib.dvq_debug_tc_pair_layout(N, K, D, pair), "dvq_debug_tc_pair_layout")
    return list(single), list(pair)


def test_flags_zero_reproduces_the_fp32_plans():
    for N in NS:
        for K in KS:
            for D in DS:
                single, pair = _old(N, K, D)
                assert _ex(N, K, D, 0) == (pair if pair[0] == 1 else single), (N, K, D)


def test_every_bf16_plan_fits_and_keeps_the_fp32_variant():
    from dvq import _cabi
    for N in NS:
        for K in KS:
            for D in DS:
                single, pair = _old(N, K, D)
                p32 = _ex(N, K, D, 0)
                p16 = _ex(N, K, D, _cabi.DVQ_Z_BF16)
                is_pair = pair[0] == 1
                assert p16[0] == p32[0] == 1, (N, K, D)          # handled by the tensor-core path, pair kernel iff fp32's
                assert p16[1:3] == p32[1:3], (N, K, D)           # same slice width and slice count
                assert p16[6] <= 227 * 1024, (N, K, D, p16)
                assert 1 <= p16[3] <= 2 and 1 <= p16[5] <= 2 and 2 <= p16[4] <= (8 if is_pair else 4)
                if is_pair:
                    assert p16[7] == 128
                elif (K + 255) // 256 * p32[2] <= 2:
                    # resident operand image: the same plan with half the staging bytes
                    assert p16[3:6] == p32[3:6] and p16[7] == p32[7], (K, D, p16, p32)
                    assert p32[6] - p16[6] == p32[5] * 128 * p32[1] * 2, (K, D, p16, p32)


def test_bf16_plan_of_config2():
    """Config 2 (K = 512, e_dim 64): resident image, two A images, two z staging slots of 128 x 64 bf16 (16 KiB each)."""
    from dvq import _cabi
    p32 = _ex(1 << 22, 512, 64, 0)
    p16 = _ex(1 << 22, 512, 64, _cabi.DVQ_Z_BF16)
    assert p16[:6] == p32[:6] == [1, 64, 1, 2, 2, 2]
    assert p32[6] - p16[6] == 2 * 128 * 64 * 2


@pytest.mark.skipif(bool(os.environ.get("DVQ_TC_PAIR")), reason="DVQ_TC_PAIR overrides the selection rule")
def test_layout_ex_rejects_bad_arguments():
    from dvq import _cabi
    out = (ctypes.c_int * 8)()
    assert _cabi.lib.dvq_debug_tc_layout_ex(1024, 0, 64, 0, out) == -1
    assert _cabi.lib.dvq_debug_tc_layout_ex(1024, 512, 64, 0, None) == -7
    assert _ex(1024, 500, 64, _cabi.DVQ_Z_BF16)[0] == 0      # K not a multiple of 32: not a tensor-core shape


def test_host_path_and_ex_entries_validate_the_flag_without_a_device():
    """dvq_vq_forward_host takes fp32 rows only; the _ex entries accept DVQ_Z_BF16 and nothing else."""
    from dvq import _cabi
    assert _cabi.DVQ_Z_BF16 == 0x400
    buf = (ctypes.c_float * 64)()
    a = ctypes.addressof(buf)
    assert _cabi.lib.dvq_vq_backward_ex(a, a, a, None, a, a, 4, 4, 8, 1.0, 0.25, 0x1, a, a, None) == -7
    assert _cabi.lib.dvq_vq_code_sums_ex(a, a, 4, 4, 8, 0x1, a, None) == -7
    assert _cabi.lib.dvq_vq_code_sums_ex(a, a, 4, 4, 6, _cabi.DVQ_Z_BF16, a, None) == -1
