"""mgym_rollout_final's argument checks that need no device (the GPU tests are in test_gpu_rollout_final.py)."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from modurl_gym_b200 import build as b

    b.build()
    import modurl_gym_b200

    return modurl_gym_b200.load_library()


def test_null_handle_is_a_bad_argument(lib):
    for K in (0, 8):
        assert lib.mgym_rollout_final(None, K, None, None, None, None, None, None, None) == -1  # MGYM_ERR_BAD_ARGUMENT
        assert b"mgym_rollout_final" in lib.mgym_last_error()
