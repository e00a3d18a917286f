"""Training-time data augmentation on the GPU (Eigen, Puhrsch & Fergus, NIPS 2014, section 3.3), beyond the reference.

`Augment` holds the ranges; the nets draw one transform per image and step on the device (a3d_augment_draw, from the
device step counter, so a replayed CUDA graph draws fresh parameters) and apply it inside the resize that opens every
step (a3d_resize_affine_tf1_s2d / a3d_resize_affine_tf1).  No host work and no extra host->device bytes.
"""
from __future__ import annotations

import dataclasses
import math

from . import _lib as L


@dataclasses.dataclass(frozen=True)
class Augment:
    """Ranges of the per-image transform (a3d_augment_desc, include/a3d.h):
    scale s ~ U[scale_lo, scale_hi] (the window spans crop_fraction/s of the frame, depths are divided by s),
    rotation ~ U[-max_rotation_deg, max_rotation_deg], a random crop centre that keeps the unrotated window inside the
    frame, a horizontal flip with probability flip_prob, and an RGB factor ~ U[color_lo, color_hi]^3.  `aspect` is the
    height/width of the frame the rotation is a rotation of."""
    scale_lo: float = 1.0
    scale_hi: float = 1.0
    max_rotation_deg: float = 0.0
    crop_fraction: float = 1.0
    flip_prob: float = 0.0
    color_lo: float = 1.0
    color_hi: float = 1.0
    aspect: float = 0.75

    def __post_init__(self):
        for f in dataclasses.fields(self):
            v = getattr(self, f.name)
            if not isinstance(v, (int, float)) or not math.isfinite(v):
                raise ValueError(f"Augment.{f.name} must be a finite number, got {v!r}")
        if not 0 < self.scale_lo <= self.scale_hi:
            raise ValueError("Augment needs 0 < scale_lo <= scale_hi")
        if not 0 < self.crop_fraction <= 1:
            raise ValueError("Augment needs 0 < crop_fraction <= 1")
        if not 0 <= self.flip_prob <= 1:
            raise ValueError("Augment needs flip_prob in [0, 1]")
        if not self.color_lo <= self.color_hi:
            raise ValueError("Augment needs color_lo <= color_hi")
        if self.max_rotation_deg < 0:
            raise ValueError("Augment needs max_rotation_deg >= 0")
        if self.aspect <= 0:
            raise ValueError("Augment needs aspect > 0")

    @classmethod
    def eigen_nyu(cls) -> "Augment":
        """The NYU Depth v2 preset of Eigen et al. (2014, section 3.3): s in [1, 1.5], r in [-5, 5] degrees, a 304x228
        crop of the 320x240 frame (f = 304/320 = 0.95), c in [0.8, 1.2]^3, flips with probability 0.5."""
        return cls(scale_lo=1.0, scale_hi=1.5, max_rotation_deg=5.0, crop_fraction=0.95, flip_prob=0.5, color_lo=0.8,
                   color_hi=1.2, aspect=0.75)

    def desc(self) -> L.AugmentDesc:
        d = L.AugmentDesc()
        for f in dataclasses.fields(self):
            setattr(d, f.name, float(getattr(self, f.name)))
        return d

    def ranges(self) -> dict:
        return dataclasses.asdict(self)


PRESETS = {"none": None, "eigen": Augment.eigen_nyu}


def from_flag(name: str) -> Augment | None:
    """`--augment` value -> Augment (or None: no augmentation)."""
    if name not in PRESETS:
        raise ValueError(f"unknown augmentation {name!r} (choose from {sorted(PRESETS)})")
    make = PRESETS[name]
    return make() if make else None
