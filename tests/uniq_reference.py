"""The uniqueness ratio of the winner-takes-all (opt-in, include/vppstereo_b200.h) as a literal NumPy restatement of its
definition: a full scan of each pixel's candidates c[0..end], no online state.  Test infrastructure for test_uniqueness_cpu.py and
test_gpu_uniqueness.py.

  left view  c[d] = S[y][x][d],     end = min(D-1, x)
  right view c[k] = S[y][x+k][k],   end = min(D-1, W-1-x)
  b = the first arg-min, c2 = min{c[d] : |d - b| >= 2}, f = (uint32)(1024.0f * u);
  accepted iff no such d exists or 1024 * c[b] <= f * c2; a rejected pixel is -10.
"""
import numpy as np

_OUT = np.int64(1) << 40          # outside every candidate range (costs are uint16)


def factor(u):
    return int(np.float32(1024.0) * np.float32(u))


def _pick(c, u):
    """c: int64 [..., D] candidates with _OUT past `end` -> float32 [...] disparities (-10 = rejected)"""
    D = c.shape[-1]
    b = np.argmin(c, axis=-1)
    cb = np.take_along_axis(c, b[..., None], axis=-1)[..., 0]
    d = np.arange(D)
    rival = (np.abs(d - b[..., None]) >= 2) & (c < _OUT)
    c2 = np.where(rival, c, _OUT).min(axis=-1)
    ok = ~rival.any(axis=-1) | (1024 * cb <= factor(u) * c2)
    return np.where(ok, b, -10).astype(np.float32)


def wta_left(S, u):
    """S uint16 [H, W, D] (or [N, H, W, D]) -> the left raw disparities with the uniqueness test"""
    S = np.asarray(S).astype(np.int64)
    W, D = S.shape[-2], S.shape[-1]
    x = np.arange(W)[:, None]
    c = np.where(np.arange(D)[None, :] <= np.minimum(D - 1, x), S, _OUT)
    return _pick(c, u)


def wta_right(S, u):
    """S uint16 [H, W, D] (or [N, H, W, D]) -> the right raw disparities with the uniqueness test"""
    S = np.asarray(S).astype(np.int64)
    W, D = S.shape[-2], S.shape[-1]
    x, k = np.arange(W)[:, None], np.arange(D)[None, :]
    src = x + k                                              # column of candidate k of target x
    inside = src <= W - 1
    c = S[..., np.minimum(src, W - 1), k]
    c = np.where(inside, c, _OUT)
    return _pick(c, u)
