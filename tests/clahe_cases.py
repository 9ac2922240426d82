"""Inputs of the CLAHE tests (tests/test_clahe_cpu.py, tests/test_gpu_clahe.py): images, clip limits and tile grids, all
generated from seeds."""
import numpy as np

from visual_odom_pipeline_b200 import synth as S

SHAPES = {                       # (h, w)
    "kitti": (376, 1241),
    "parking": (480, 640),
    "malaga": (768, 1024),
    "4k crop": (2160, 1536),
    "odd": (101, 37),
    "odd small": (9, 17),
    "tiny": (3, 3),
    "pixel": (1, 1),
    "one row": (1, 50),
    "one column": (50, 1),
    "two rows": (2, 7),
}
LARGE = ("kitti", "parking", "malaga", "4k crop")
# (1, 1); the reference front ends' (8, 8); grids that divide neither axis; more tiles than pixels along an axis
GRIDS = [(1, 1), (8, 8), (7, 5), (16, 3), (20, 20)]
CLIPS = [0.0, -2.0, 1.0, 3.0, 40.0, 5000.0]
KINDS = ("noise", "texture", "levels", "constant")


def image(kind, h, w, seed):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "texture":
        # a dim texture, as in an under-exposed frame
        return np.clip(S.texture(max(h, 2), max(w, 2), seed=seed)[:h, :w] * 0.45 + 10, 0, 255).astype(np.uint8)
    if kind == "levels":
        # 3-4 grey levels: most bins empty, the clipped excess and its remainder large
        return (rng.integers(0, 3 + seed % 2, (h, w)) * 60 + 20).astype(np.uint8)
    return np.full((h, w), 77, np.uint8)


def cases(shapes=None):
    """-> [(name, img, clip, grid)]: every shape x grid x image kind, with the clip limits taken in turn, and on the KITTI
    shape every clip limit with the (8, 8) grid on the texture."""
    out = []
    i = 0
    for sname, (h, w) in SHAPES.items():
        if shapes is not None and sname not in shapes:
            continue
        for grid in GRIDS:
            for kind in KINDS:
                if sname in LARGE and kind == "constant" and grid != (8, 8):
                    continue
                clip = CLIPS[i % len(CLIPS)]
                i += 1
                out.append(("%s %s %s clip %g" % (sname, kind, grid, clip), image(kind, h, w, i), clip, grid))
    if shapes is None or "kitti" in shapes:
        for clip in CLIPS:
            out.append(("kitti texture (8, 8) clip %g" % clip, image("texture", 376, 1241, 900), clip, (8, 8)))
    return out
