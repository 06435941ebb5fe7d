"""Seeded synthetic inputs shaped like the reference's data (SURVEY.md §8d).

G1  ``blob_stack``   — the paraboloid blob of the reference's ``tests/test_flow.py:203-204,317`` scaled to
                       100x100 and rolled one pixel per frame.
G2  ``bt_sequence``  — brightness-temperature-like float32 ``(T, H, W)``: a smooth periodic field advected
                       by (+1, +2) px/frame, a warm clear-sky plateau at 285 K, growing cold cores, and the
                       NaN patterns of ``tobac_flow/dataloader.py:288-357`` (bad pixels, a missing stripe,
                       a whole missing frame).
G3  ``moving_texture`` — an analytic texture under prescribed, per-pair motion (shifts, rotation, zoom, a
                       discontinuity), exact in every frame: flow tests against OpenCV beyond a constant roll.

``bt_sequence`` works on numpy (tests, CPU baseline) and on torch tensors (bench, on the GPU) from the
same seeded base field, so the CPU baseline and the CUDA path see identical inputs.
"""
import numpy as np


def blob_stack(T: int = 10, n: int = 100) -> np.ndarray:
    xx, yy = np.meshgrid(np.arange(n), np.arange(n))
    c = (n - 1) / 2
    blob = ((c ** 2 - (xx - c) ** 2) * (c ** 2 - (yy - c) ** 2)).astype(np.float32)
    return np.stack([np.roll(blob, (t, t), (0, 1)) for t in range(T)])


def base_field(H: int, W: int, seed: int, sigma_px: float = 12.0) -> np.ndarray:
    """Periodic smooth field in [0, 1]: white noise through a Gaussian spectral filter."""
    rng = np.random.default_rng(seed)
    noise = rng.standard_normal((H, W)).astype(np.float32)
    fy = np.fft.fftfreq(H)[:, None]
    fx = np.fft.rfftfreq(W)[None, :]
    filt = np.exp(-2.0 * (np.pi * sigma_px) ** 2 * (fx * fx + fy * fy))
    f = np.fft.irfft2(np.fft.rfft2(noise) * filt, s=(H, W))
    f = (f - f.min()) / (f.max() - f.min())
    return f.astype(np.float32)


def core_table(T: int, H: int, W: int, seed: int):
    """Seeded growing cold cores: (y, x, t_start) rows; 8 per 3.75 Mpx, at least 2."""
    rng = np.random.default_rng(seed + 7919)
    n = max(2, int(round(8 * H * W / 3.75e6)))
    ys = rng.integers(H // 8, max(H - H // 8, H // 8 + 1), n)
    xs = rng.integers(W // 8, max(W - W // 8, W // 8 + 1), n)
    ts = rng.integers(0, max(T - 6, 1), n)
    return np.stack([ys, xs, ts], -1)


def nan_plan(T: int, H: int, W: int, seed: int, frac: float = 5e-4):
    """Which frames get a 16-row stripe / go entirely missing, and the bad-pixel fraction."""
    stripe_frames = list(range(5, T, 48))
    missing_frames = [t for t in range(71, T, 144)]
    return dict(frac=frac, stripe_frames=stripe_frames, missing_frames=missing_frames,
                stripe_row=(H // 3) if H > 48 else 1, seed=seed + 104729)


def bt_frame(base, t: int, cores, plan, T: int):
    """One BT frame from the base field; ``base`` may be a numpy array or a torch tensor."""
    is_torch = not isinstance(base, np.ndarray)
    H, W = base.shape
    if is_torch:
        import torch
        f = torch.roll(base, shifts=(t, 2 * t), dims=(0, 1))
        bt = 200.0 + 100.0 * f
        yy = torch.arange(H, device=base.device, dtype=torch.float32)[:, None]
        xx = torch.arange(W, device=base.device, dtype=torch.float32)[None, :]
        exp, clamp_max = torch.exp, lambda a, m: torch.clamp(a, max=m)
    else:
        f = np.roll(base, (t, 2 * t), (0, 1))
        bt = np.float32(200.0) + np.float32(100.0) * f
        yy = np.arange(H, dtype=np.float32)[:, None]
        xx = np.arange(W, dtype=np.float32)[None, :]
        exp, clamp_max = np.exp, lambda a, m: np.minimum(a, np.float32(m))
    bt = clamp_max(bt, 285.0)
    for cy, cx, t0 in cores:
        age = t - int(t0)
        if age <= 0:
            continue
        g = min(age, 12) / 12.0
        sig = 6.0 + 6.0 * g
        # cores drift with the background advection so they can be tracked
        py = float((int(cy) + age) % H)
        px = float((int(cx) + 2 * age) % W)
        d2 = (yy - py) ** 2 + (xx - px) ** 2
        bt = bt - (40.0 * g) * exp(-d2 / (2.0 * sig * sig))
    if is_torch:
        bt = bt.to(torch.float32)
    else:
        bt = bt.astype(np.float32)
    # NaN injection
    if plan is not None:
        rng = np.random.default_rng(plan["seed"] + t)
        n_bad = int(plan["frac"] * H * W)
        if n_bad:
            idx = rng.integers(0, H * W, n_bad)
            if is_torch:
                import torch
                bt.view(-1)[torch.as_tensor(idx, device=bt.device)] = float("nan")
            else:
                bt.reshape(-1)[idx] = np.nan
        if t in plan["stripe_frames"]:
            r = plan["stripe_row"]
            bt[r:r + 16] = float("nan")
        if t in plan["missing_frames"]:
            bt[:] = float("nan")
    return bt


def bt_sequence(T: int, H: int, W: int, seed: int = 1234, nans: bool = True, device=None):
    """(T, H, W) float32; numpy when ``device`` is None, else a torch tensor on ``device``."""
    base = base_field(H, W, seed)
    cores = core_table(T, H, W, seed)
    plan = nan_plan(T, H, W, seed) if nans else None
    if device is None:
        return np.stack([bt_frame(base, t, cores, plan, T) for t in range(T)])
    import torch
    base_t = torch.as_tensor(base, device=device)
    out = torch.empty((T, H, W), dtype=torch.float32, device=device)
    for t in range(T):
        out[t] = bt_frame(base_t, t, cores, plan, T)
    return out


def texture(x, y, seed: int = 0):
    """Analytic texture: 12 seeded sinusoids (wavelengths 10-45 px) around 250 K, float64 at arbitrary (x, y)."""
    rng = np.random.default_rng(seed)
    f = np.full(np.broadcast(x, y).shape, 250.0)
    for _ in range(12):
        k = 2.0 * np.pi / rng.uniform(10.0, 45.0)
        th = rng.uniform(0.0, 2.0 * np.pi)
        f += rng.uniform(1.5, 4.0) * np.sin(k * np.cos(th) * x + k * np.sin(th) * y + rng.uniform(0.0, 2.0 * np.pi))
    return f


# motions d(x, y, H, W) -> (u, v) for moving_texture: frame k + 1 at x shows frame k at x - d(x), so the forward flow
# of the pair is ~ d
def shift_motion(u: float, v: float):
    return lambda x, y, H, W: (np.full_like(x, u), np.full_like(y, v))


def rotation_motion(deg: float):
    """Rotation by ``deg`` about the frame centre."""
    def d(x, y, H, W):
        cx, cy, a = (W - 1) / 2.0, (H - 1) / 2.0, np.deg2rad(deg)
        rx = cx + np.cos(a) * (x - cx) + np.sin(a) * (y - cy)       # the point that rotates onto (x, y)
        ry = cy - np.sin(a) * (x - cx) + np.cos(a) * (y - cy)
        return x - rx, y - ry
    return d


def zoom_motion(factor: float):
    """Magnification by ``factor`` about the frame centre (outward flow for factor > 1)."""
    def d(x, y, H, W):
        cx, cy = (W - 1) / 2.0, (H - 1) / 2.0
        return (x - cx) * (1.0 - 1.0 / factor), (y - cy) * (1.0 - 1.0 / factor)
    return d


def split_motion(s: float):
    """+s px along x left of the centre column, -s px right of it: a motion discontinuity."""
    return lambda x, y, H, W: (np.where(x < (W - 1) / 2.0, s, -s), np.zeros_like(y))


def moving_texture(H: int, W: int, motions, seed: int = 0) -> np.ndarray:
    """(len(motions) + 1, H, W) float32 frames of ``texture``, each pair with its own motion.

    Frame k is the texture at p_k(x), p_0 the identity and p_k(x) = p_{k-1}(x - d_k(x)), evaluated in float64: no frame
    carries interpolation error."""
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    frames = []
    for k in range(len(motions) + 1):
        px, py = x, y
        for m in reversed(motions[:k]):
            u, v = m(px, py, H, W)
            px, py = px - u, py - v
        frames.append(texture(px, py, seed))
    return np.stack(frames).astype(np.float32)


def wvd_from_bt(bt):
    """A monotone map of BT into a water-vapour-difference-like range [-30, +2] K (colder -> larger)."""
    return (2.0 - (bt - 200.0) * (32.0 / 85.0))
