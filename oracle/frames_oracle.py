"""numpy statement of v2ce_assemble_windows (csrc/frames.cu): colour -> gray, center crop, window gather.

Gray conversion is OpenCV's cvtColor(COLOR_{BGR,RGB,BGRA,RGBA}2GRAY) for 8-bit input, the conversion the reference's
video reader applies (scripts/video_reader.py:66-67).  The coefficients are 15-bit fixed point, rounded half up; they
were derived from cv2 and tests/test_frames_oracle.py pins them against the installed cv2 over all 2^24 colours."""
import numpy as np

B2Y, G2Y, R2Y, SHIFT = 3735, 19235, 9798, 15

# color name -> (channels, index of blue, index of green, index of red)
COLORS = {'gray': (1, 0, 0, 0), 'bgr': (3, 0, 1, 2), 'rgb': (3, 2, 1, 0), 'bgra': (4, 0, 1, 2), 'rgba': (4, 2, 1, 0)}


def to_gray(frame, color):
    """(..., H, W) gray or (..., H, W, C) colour uint8 -> (..., H, W) uint8."""
    c, ib, ig, ir = COLORS[color]
    f = np.asarray(frame)
    if c == 1:
        return f.copy()
    assert f.shape[-1] == c, (f.shape, color)
    f = f.astype(np.int32)
    v = f[..., ib] * B2Y + f[..., ig] * G2Y + f[..., ir] * R2Y + (1 << (SHIFT - 1))
    return (v >> SHIFT).astype(np.uint8)


def assemble_windows(frames, slots, color='gray', x0=0, out_width=None):
    """frames: sequence of source frames; slots (n_windows, L+1) source index per output frame ->
    (n_windows, L+1, H, out_width) uint8, columns x0 .. x0 + out_width of each gray frame."""
    slots = np.asarray(slots)
    gray = [to_gray(f, color) for f in frames]
    W = gray[0].shape[1]
    out_width = W - x0 if out_width is None else out_width
    return np.stack([np.stack([gray[s][:, x0:x0 + out_width] for s in row]) for row in slots])
