"""Image scenes for the robust velocity solve: a ground-plane pair (synth.make_pair) with a textured object that moves
on its own, pasted into both frames at positions that differ by the object's displacement."""
import numpy as np

import synth


def moving_patch_pair(h, w, seed, frac, shift=(9.0, -7.0), max_disp=6.0):
    """-> (prev, next, motion, (y0, x0, ph, pw)): frame 2 is the ground moved by the plane model of `motion`; a square
    patch covering `frac` of the frame sits at (y0, x0) in frame 1 and `shift` px (x, y, whole pixels) further in
    frame 2, so its features track with status 1 but move unlike the ground."""
    a, b, mo = synth.make_pair(h, w, seed, seed, max_disp=max_disp)
    side = int(round(np.sqrt(frac * h * w)))
    patch = synth.texture(side, side, 500 + seed)
    rng = np.random.default_rng(seed)
    dx, dy = int(round(shift[0])), int(round(shift[1]))
    y0 = int(rng.integers(20 + max(0, -dy), h - side - 20 - max(0, dy)))
    x0 = int(rng.integers(20 + max(0, -dx), w - side - 20 - max(0, dx)))
    a = a.copy()
    b = b.copy()
    a[y0:y0 + side, x0:x0 + side] = patch
    b[y0 + dy:y0 + dy + side, x0 + dx:x0 + dx + side] = patch
    return a, b, mo, (y0, x0, side, side)


def in_patch(pts, box, margin=0.0):
    y0, x0, ph, pw = box
    return ((pts[:, 0] >= x0 - margin) & (pts[:, 0] < x0 + pw + margin) &
            (pts[:, 1] >= y0 - margin) & (pts[:, 1] < y0 + ph + margin))
