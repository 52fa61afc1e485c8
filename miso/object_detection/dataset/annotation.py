"""Rectangle annotation: the fields and derived geometry the hot path reads
(ref:miso/object_detection/dataset/annotation.py:33-127). Values keep the numpy scalar type they
are given (np.float32 from inference), so x + width is rounded in fp32 exactly like the reference."""
from __future__ import annotations

import numpy as np


class RectangleAnnotation:
    def __init__(self, x, y, width, height, label, score=1.0, annotator=None, validator=None, uid=None, mask=None):
        self.x, self.y, self.width, self.height = x, y, width, height
        self.label, self.score = label, score
        self.annotator, self.validator, self.uid = annotator, validator, uid
        self.mask = mask        # np.uint8 [h, w] instance mask (0 / 255) over the crop rectangle, or None

    @property
    def bounds(self):
        return self.x, self.y, self.width, self.height

    @property
    def coords(self):
        return self.x, self.y, self.x + self.width, self.y + self.height

    @property
    def coords_int(self):
        return tuple(int(np.round(c)) for c in self.coords)      # round half to even

    @property
    def bounds_int(self):
        return tuple(int(np.round(c)) for c in self.bounds)

    def __str__(self):
        return f"{self.label} - x: {self.x}, y: {self.y}, w: {self.width}, h: {self.height}"
