"""Output buffers surrounded by canaries: a kernel's result is written into a view of a larger buffer whose every other
byte holds a NaN with a payload, so a store outside the view (a spilled tile, a wrong row stride, a neighbouring column
slice) is seen as changed bytes."""
import torch

_BITS = {torch.float32: torch.int32, torch.bfloat16: torch.int16}
_CANARY = {torch.float32: 0x7FC00000, torch.bfloat16: 0x7FA5}   # an f32 NaN and a bf16 NaN with payload


class Buf:
    """[rows, cols] view with row stride ld inside a canary-filled buffer: `off` elements and one full row before it, two
    rows after it, ld - cols columns beside every row."""

    def __init__(self, rows, cols, ld, dtype, off=0):
        self.buf = torch.empty(off + (rows + 3) * ld, dtype=dtype, device="cuda")
        self.buf.view(_BITS[dtype]).fill_(_CANARY[dtype])
        self.shape, self.stride, self.start = (rows, cols), (ld, 1), off + ld
        self.view = torch.as_strided(self.buf, self.shape, self.stride, self.start)
        self.before = None

    def snapshot(self):
        self.before = self.buf.view(_BITS[self.buf.dtype]).clone()

    def outside_unchanged(self, views=None):
        """Every byte outside the view (or outside each of `views`, column slices of it) is as at snapshot()."""
        now = self.buf.view(_BITS[self.buf.dtype]).clone()
        before = self.before.clone()
        for v in views if views is not None else [self.view]:
            off = v.storage_offset() - self.buf.storage_offset()
            for t in (now, before):
                torch.as_strided(t, v.shape, v.stride(), off).zero_()
        return torch.equal(now, before)

    def unchanged(self):
        return torch.equal(self.buf.view(_BITS[self.buf.dtype]), self.before)
