"""CPU tier of the batched frame step: the workspace query of klt_frame_step_batch needs no GPU."""


def test_frame_step_workspace_query(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    ws = L.klt_frame_step_ws_bytes
    assert ws(1241, 376, 1, 0) > 0
    assert ws(1241, 376, 4, 2000) > ws(1241, 376, 4, 1000) > ws(1241, 376, 4, 0)
    assert ws(1241, 376, 8, 2000) > ws(1241, 376, 4, 2000)
    # keys, eigenvalues, mask and the corner scans' scratch of every frame at least
    assert ws(1241, 376, 4, 0) >= 4 * 1241 * 376 * (8 + 4 + 1) + L.klt_corner_ws_bytes(1241, 376, 4)
    for bad in [(0, 376, 1, 10), (1241, 0, 1, 10), (1241, 376, 0, 10), (1241, 376, 1, -1)]:
        assert ws(*bad) == 0
