"""mgym_step_episodes / mgym_rollout_episodes argument checks that need no device (the GPU tests are in
test_gpu_episodes.py)."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from modurl_gym_b200 import build as b

    b.build()
    import modurl_gym_b200

    return modurl_gym_b200.load_library()


def test_null_handle_is_a_bad_argument(lib):
    assert lib.mgym_step_episodes(None, None, None, None, None, None, None, None, None) == -1  # MGYM_ERR_BAD_ARGUMENT
    assert b"mgym_step_episodes" in lib.mgym_last_error()
    for K in (0, 8):
        assert lib.mgym_rollout_episodes(None, K, None, None, None, None, None, None, None, None, None) == -1
        assert b"mgym_rollout_episodes" in lib.mgym_last_error()
