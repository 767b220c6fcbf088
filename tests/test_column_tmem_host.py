"""Host side of the TMA column kernel's tensor-memory stash (no GPU needed): the columns a CTA allocates for its
parked levels, and the shared-memory padding that keeps the CTAs resident on an SM within its 512 columns."""
import ctypes as C

import pytest

SMEM_PER_SM, SMEM_RESERVED_PER_CTA, TMEM_COLS_PER_SM = 228 * 1024, 1024, 512
K = 19        # plev19


def _layout(nplev, nlev, np_):
    from pgw4era5_b200 import _native as N
    cols, smem = C.c_int(0), C.c_longlong(0)
    rc = N.lib.pgw_column_tma_layout(nplev, nlev, np_, C.byref(cols), C.byref(smem))
    return rc, cols.value, smem.value


@pytest.mark.parametrize("np_, cols", [(2, 32), (16, 32), (18, 64), (32, 64), (56, 128), (64, 128), (66, 256),
                                       (128, 256), (130, 512), (160, 512)])
def test_columns_are_the_next_power_of_two_of_the_stash(np_, cols):
    rc, c, _ = _layout(K, 160, np_)
    assert rc == 0 and c == cols and c >= 2 * np_


@pytest.mark.parametrize("np_", [2, 16, 56, 64, 66, 100, 128, 130, 160])
def test_shared_memory_bounds_resident_ctas_by_tensor_memory(np_):
    _, cols, smem = _layout(K, 160, np_)
    ctas = SMEM_PER_SM // (smem + SMEM_RESERVED_PER_CTA)
    assert ctas * cols <= TMEM_COLS_PER_SM
    # and no tighter than that: up to 128 columns the registers (4 CTAs of 256 threads) bind, 256 leave two, 512 one
    assert min(ctas, 4) == min(4, TMEM_COLS_PER_SM // cols)
    assert smem <= SMEM_PER_SM - SMEM_RESERVED_PER_CTA


def test_era5_l137_plan_runs_four_ctas_per_sm():
    # 56 parked levels (p_ref = 300 hPa): 112 columns of (T_pgw, e_pgw) in a 128-column allocation
    _, cols, smem = _layout(K, 137, 56)
    assert cols == 128
    assert SMEM_PER_SM // (smem + SMEM_RESERVED_PER_CTA) == 4


def test_padding_covers_the_ring_and_tables():
    # ring, level and node tables stay well inside a quarter of the SM at any node count
    _, _, small = _layout(2, 137, 56)
    _, _, large = _layout(64, 137, 56)
    assert small == large == SMEM_PER_SM // 4 - SMEM_RESERVED_PER_CTA


@pytest.mark.parametrize("args", [(1, 137, 56), (65, 137, 56), (19, 161, 56), (19, 137, 0), (19, 137, 57),
                                  (19, 137, 138)])
def test_rejects_out_of_range(args):
    from pgw4era5_b200 import _native as N
    assert _layout(*args)[0] == N.PGW_E_INVALID
