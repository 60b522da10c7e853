"""GPU: the CROP kernel's TMA box loads against its per-row vector loads (crop_load = 1), byte for byte.

Both paths run the same arithmetic, so every cloud must be identical, and neither may write outside its frame's
points: each output frame sits between canary bytes that must come back untouched.  Batches are large enough
that the launch keeps 4 / 6 / 8 rows per unit (a lone small frame falls back to 2-row units and per-row loads).
"""
import numpy as np
import pytest
import torch

from disparity_to_point_cloud_b200 import synth

pytestmark = pytest.mark.gpu

CANARY = 0xA5
PAD = 4096  # canary bytes before and after every output frame


@pytest.fixture(scope="module")
def ctx():
    import disparity_to_point_cloud_b200 as d2pc
    with d2pc.Context() as c:
        yield c


def _frames(w, h, f, step, frame_stride):
    """f float frames of w x h (S3 data, rolled per frame) at the given row and frame strides, on the device."""
    base = synth.s3_float(h, w, 11)
    buf = torch.zeros(f * frame_stride // 4 + 64, dtype=torch.float32, device="cuda")
    for i in range(f):
        v = buf[i * frame_stride // 4: i * frame_stride // 4 + h * step // 4].view(h, step // 4)
        v[:, :w] = torch.from_numpy(np.roll(base, 37 * i, axis=1)).cuda()
    return buf


def _run(ctx, buf, offset, f, w, h, step, frame_stride, crop_load, rows):
    n = (w - 80) * (h - 80)
    stride = n * 16 + 2 * PAD
    out = torch.full((f * stride + PAD,), CANARY, dtype=torch.uint8, device="cuda")
    ctx.set_tuning("crop_load", crop_load)
    ctx.set_tuning("rows_per_unit", rows)
    try:
        ctx.reproject_f32_device(buf.data_ptr() + offset, f, w, h, step, frame_stride, out.data_ptr() + PAD, stride)
        torch.cuda.synchronize()
    finally:
        ctx.set_tuning("crop_load", 0)
        ctx.set_tuning("rows_per_unit", 0)
    o = out.cpu().numpy()
    clouds = np.stack([o[PAD + i * stride: PAD + i * stride + n * 16] for i in range(f)])
    canary = np.concatenate([o[:PAD]] + [o[PAD + i * stride + n * 16: PAD + (i + 1) * stride] for i in range(f)])
    assert (canary == CANARY).all(), "a store landed outside the frame's points"
    return clouds


CASES = [
    # (w, h, frames, extra row bytes, extra frame bytes, rows per unit)
    (3840, 2160, 16, 0, 0, 0),      # config 4: 3760 = 29 x 128 + 48, the last segment is partial
    (1280, 720, 64, 0, 0, 0),
    (640, 480, 32, 0, 0, 0),
    (752, 480, 32, 0, 0, 0),        # 672 = 5 x 128 + 32
    (1280, 725, 64, 0, 0, 6),       # 645 crop rows: the last row block of each frame is partial at 4 / 6 / 8
    (1280, 725, 64, 0, 0, 4),
    (1280, 725, 64, 0, 0, 8),
    (1024, 600, 32, 0, 0, 4),       # 944 = 7 x 128 + 48
    (1280, 720, 64, 256, 4096, 6),  # pitched rows, frame_stride > h * step
    (1328, 720, 48, 0, 1 << 20, 8),  # 1248 = 9 x 128 + 96, frames 1 MB apart
]


@pytest.mark.parametrize("w,h,f,row_pad,frame_pad,rows", CASES)
def test_tma_equals_ldg(ctx, w, h, f, row_pad, frame_pad, rows):
    step = 4 * w + row_pad
    frame_stride = h * step + frame_pad
    buf = _frames(w, h, f, step, frame_stride)
    tma = _run(ctx, buf, 0, f, w, h, step, frame_stride, 0, rows)
    ldg = _run(ctx, buf, 0, f, w, h, step, frame_stride, 1, rows)
    assert tma.tobytes() == ldg.tobytes()
    assert (tma.view(np.float32).reshape(f, -1, 4)[:, :, 3] == 1.0).all()


def test_unaligned_base_takes_the_fallback(ctx):
    """A base 4 bytes off the 16-byte grid cannot be described by the map: the scalar path serves it, with the same
    points as an aligned copy of the same frames."""
    w, h, f = 1280, 720, 32
    step = 4 * w + 16
    frame_stride = h * step
    buf = _frames(w, h, f, step, frame_stride)
    shifted = torch.zeros(buf.numel() + 4, dtype=torch.float32, device="cuda")
    shifted[1:1 + buf.numel()] = buf
    want = _run(ctx, buf, 0, f, w, h, step, frame_stride, 0, 8)
    got = _run(ctx, shifted, 4, f, w, h, step, frame_stride, 0, 8)
    assert got.tobytes() == want.tobytes()
