"""Oracle restatement of the FID InceptionV3 (pytorch-fid's ``InceptionV3([pool3])``, the network of the
reference's ``fid/inception.py`` / ``fid/fid_score_v.py``) for any dtype.  TEST INFRASTRUCTURE: imported by tests
and tools only.

torchvision's ``Inception3`` trunk (``transform_input=False``, BatchNorm eps 1e-3, no aux head) with the FID blocks
of pytorch-fid: the branch pool of Mixed_5b..5d (InceptionA), Mixed_6b..6e (InceptionC) and Mixed_7b (InceptionE)
is ``avg_pool2d(3, 1, 1, count_include_pad=False)``, that of Mixed_7c ``max_pool2d(3, 1, 1)``.  Preprocessing:
``input_range`` -> [0, 1], bilinear resize to 299 x 299 (align_corners=False, no antialias), [0, 1] -> [-1, 1];
output: the 2048 features after the global average pool.
"""
import torch
import torch.nn.functional as F
from torchvision.models import inception as tvi


class FIDInceptionA(tvi.InceptionA):
    def forward(self, x):
        b1 = self.branch1x1(x)
        b5 = self.branch5x5_2(self.branch5x5_1(x))
        b3 = self.branch3x3dbl_3(self.branch3x3dbl_2(self.branch3x3dbl_1(x)))
        bp = self.branch_pool(F.avg_pool2d(x, 3, 1, 1, count_include_pad=False))
        return torch.cat([b1, b5, b3, bp], 1)


class FIDInceptionC(tvi.InceptionC):
    def forward(self, x):
        b1 = self.branch1x1(x)
        b7 = self.branch7x7_3(self.branch7x7_2(self.branch7x7_1(x)))
        d = x
        for m in (self.branch7x7dbl_1, self.branch7x7dbl_2, self.branch7x7dbl_3, self.branch7x7dbl_4,
                  self.branch7x7dbl_5):
            d = m(d)
        bp = self.branch_pool(F.avg_pool2d(x, 3, 1, 1, count_include_pad=False))
        return torch.cat([b1, b7, d, bp], 1)


class _FIDInceptionE(tvi.InceptionE):
    def _pool(self, x):
        raise NotImplementedError

    def forward(self, x):
        b1 = self.branch1x1(x)
        b3 = self.branch3x3_1(x)
        b3 = torch.cat([self.branch3x3_2a(b3), self.branch3x3_2b(b3)], 1)
        d = self.branch3x3dbl_2(self.branch3x3dbl_1(x))
        d = torch.cat([self.branch3x3dbl_3a(d), self.branch3x3dbl_3b(d)], 1)
        bp = self.branch_pool(self._pool(x))
        return torch.cat([b1, b3, d, bp], 1)


class FIDInceptionE1(_FIDInceptionE):
    def _pool(self, x):
        return F.avg_pool2d(x, 3, 1, 1, count_include_pad=False)


class FIDInceptionE2(_FIDInceptionE):
    def _pool(self, x):
        return F.max_pool2d(x, 3, 1, 1)


class FIDInception(tvi.Inception3):
    """torchvision Inception3 with the FID blocks; ``features(frames)`` is the pool3 forward.  Its state_dict names
    are torchvision's ``inception_v3`` names without ``AuxLogits``."""

    def __init__(self, input_range=(-1.0, 1.0)):
        super().__init__(num_classes=1008, aux_logits=False, transform_input=False, init_weights=True)
        self.input_range = input_range
        self.Mixed_5b = FIDInceptionA(192, 32)
        self.Mixed_5c = FIDInceptionA(256, 64)
        self.Mixed_5d = FIDInceptionA(288, 64)
        self.Mixed_6b = FIDInceptionC(768, 128)
        self.Mixed_6c = FIDInceptionC(768, 160)
        self.Mixed_6d = FIDInceptionC(768, 160)
        self.Mixed_6e = FIDInceptionC(768, 192)
        self.Mixed_7b = FIDInceptionE1(1280)
        self.Mixed_7c = FIDInceptionE2(2048)

    def features(self, frames):
        lo, hi = self.input_range
        x = (frames.to(self.Conv2d_1a_3x3.conv.weight.dtype) - lo) / (hi - lo)
        x = F.interpolate(x, size=(299, 299), mode="bilinear", align_corners=False)
        x = 2 * x - 1
        x = self.Conv2d_2b_3x3(self.Conv2d_2a_3x3(self.Conv2d_1a_3x3(x)))
        x = self.Conv2d_4a_3x3(self.Conv2d_3b_1x1(self.maxpool1(x)))
        x = self.maxpool2(x)
        for name in ("Mixed_5b", "Mixed_5c", "Mixed_5d", "Mixed_6a", "Mixed_6b", "Mixed_6c", "Mixed_6d", "Mixed_6e",
                     "Mixed_7a", "Mixed_7b", "Mixed_7c"):
            x = getattr(self, name)(x)
        return x.mean((2, 3))
