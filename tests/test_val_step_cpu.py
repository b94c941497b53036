"""CPU: the validation step's C entry point rejects bad arguments before any CUDA call, its workspace query, the choice
between the one-launch kernel and the composed kernels in ``HeatmapHotPath.val_step``, and the rows -> dicts helper."""
import pytest
import torch

GT, BASIC = 0, 2


@pytest.fixture(scope="module")
def lib():
    from simple_pose_b200 import build, _abi
    build.build()
    return _abi.lib()


def val_args(lib, B=1, K=17, H=64, W=48, mode=GT, ksize=11):
    ws_bytes = lib.sp_val_step_workspace_bytes(B, K)
    # joints, pred, trans_inv, blur_w, mode, weights, loss, acc, rows, coords, maxval, pred_xy, label_xy, ws, ws_bytes,
    # B, K, H, W, sigma, ksize, distance_thresh, norm_frac, stream
    return [16, 16, 16, 16, mode, 16, 16, 16, 16, 16, 16, None, None, 16, ws_bytes, B, K, H, W, 2.0, ksize, 0.5, 10.0, None]


def with_(args, **kw):
    names = ["joints", "pred", "trans_inv", "blur_w", "mode", "weights", "loss", "acc", "rows", "coords", "maxval",
             "pred_xy", "label_xy", "ws", "ws_bytes", "B", "K", "H", "W", "sigma", "ksize", "thresh", "norm_frac", "stream"]
    out = list(args)
    for k, v in kw.items():
        out[names.index(k)] = v
    return out


def test_val_step_argument_errors(lib):
    ok = val_args(lib)
    call = lambda a: lib.sp_val_step_f32(*a)
    for mode in (1, 3, 4, -1):                                          # argmax-only, DarkPose original, unknown
        assert call(with_(ok, mode=mode)) == -1
    for name in ("joints", "pred", "loss", "acc", "rows", "ws"):
        assert call(with_(ok, **{name: None})) == -1, name
    assert call(with_(ok, blur_w=None)) == -1                           # GaussTaylor needs the blur weights
    assert call(with_(ok, coords=None)) == -1                           # coords without maxval
    assert call(with_(ok, pred_xy=16)) == -1                            # pred_xy without label_xy
    assert call(with_(ok, B=0)) == -1 and call(with_(ok, K=0)) == -1 and call(with_(ok, sigma=0.0)) == -1
    assert call(with_(ok, norm_frac=0.0)) == -1
    assert call(with_(ok, W=50)) == -4                                  # W % 4 != 0
    assert call(with_(ok, ksize=9)) == -4                               # GaussTaylor: only the 11 x 11 blur
    assert call(with_(ok, H=4096, W=4096)) == -4                        # map larger than the 2^24 pixel limit
    assert call(with_(ok, ws_bytes=ok[14] - 1)) == -3                   # workspace too small
    assert call(with_(ok, ws=24)) == -2                                 # misaligned workspace
    assert call(with_(ok, pred=24)) == -2                               # misaligned pred
    assert call(with_(ok, coords=24)) == -2                             # misaligned coords
    assert call(with_(ok, pred_xy=24, label_xy=16)) == -2               # misaligned axes
    # Basic needs no blur weights and takes any ksize, but the same shape limits apply
    basic = val_args(lib, mode=BASIC)
    assert call(with_(basic, W=50, blur_w=None, ksize=0)) == -4
    assert call(with_(basic, blur_w=None, ksize=0, ws_bytes=8)) == -3
    assert call(with_(basic, blur_w=None, ksize=0, pred=24)) == -2


def test_val_step_workspace_bytes(lib):
    base = lib.sp_mse_workspace_bytes()
    counters = lambda b: (4 * b + 15) // 16 * 16
    for b, k in ((1, 17), (128, 17), (1024, 17), (3, 5), (7, 1)):
        assert lib.sp_val_step_workspace_bytes(b, k) == (base + 15) // 16 * 16 + counters(b) + 16 * b * k
        assert lib.sp_val_step_workspace_bytes(b, k) % 16 == 0
    assert lib.sp_val_step_workspace_bytes(0, 17) == (base + 15) // 16 * 16


@pytest.mark.parametrize("h,w,ksize,decoder,want", [
    (64, 48, 11, "gauss_taylor", True), (64, 48, 11, "basic", True), (96, 72, 11, "gauss_taylor", True),
    (64, 48, 9, "gauss_taylor", False), (64, 48, 9, "basic", True),            # Basic has no blur
    (63, 50, 11, "gauss_taylor", False), (63, 50, 11, "basic", False),         # W % 4 != 0
    (256, 256, 11, "basic", False),                                            # one map does not fit in shared memory
])
def test_val_step_path_selection(h, w, ksize, decoder, want):
    from simple_pose_b200.pipeline import HeatmapHotPath
    assert HeatmapHotPath.val_one_launch_supported(h, w, ksize, decoder) is want


def test_rows_to_dicts_is_kps_to_dict_loop():
    from simple_pose_b200.metrics.pose_metrics import rows_to_dicts
    rows = torch.tensor([[1.0, 2.0, 0.5, 3.0, 4.0, 0.25, 0.875], [5.0, 6.0, 0.0, 7.0, 8.0, 1.0, 1.5]])
    out = [{"image_id": 0}]
    rows_to_dicts(rows, [11, 12], out)
    assert out[1:] == [{"image_id": 11, "score": 0.875, "category_id": 1, "keypoints": [1.0, 2.0, 0.5, 3.0, 4.0, 0.25]},
                       {"image_id": 12, "score": 1.5, "category_id": 1, "keypoints": [5.0, 6.0, 0.0, 7.0, 8.0, 1.0]}]
