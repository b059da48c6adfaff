"""Interleaved 8-bit test images for yk_set_image_interleaved[_device]: the bytes of int32 planes laid out as a decoder
would hand them over, in a buffer that ends exactly at the last pixel's last byte (so that AddressSanitizer catches any
read past it), with optional garbage row padding and a base that is `offset` bytes past a 16-byte boundary."""
import numpy as np

PAD_BYTE = 0xA5


class Interleaved:
    def __init__(self, planes: np.ndarray, channels=None, pad=0, offset=0):
        c, h, w = planes.shape
        ch = channels or c
        self.w, self.h, self.channels = w, h, ch
        self.row_bytes = w * ch + pad
        span = self.row_bytes * (h - 1) + w * ch
        front = offset
        for _ in range(16):          # the allocation's own alignment is not known in advance
            self.raw = np.empty(front + span, np.uint8)
            f = (offset - self.raw.ctypes.data) % 16
            if f == front:
                break
            front = f
        assert (self.raw.ctypes.data + front) % 16 == offset
        self.raw[:] = PAD_BYTE
        px = np.empty((h, w, ch), np.uint8)
        px[:, :, :min(c, ch)] = np.transpose(planes[:ch], (1, 2, 0))
        if ch > c:
            px[:, :, c:] = np.uint8(0x5A)         # an alpha channel the slot is told to ignore
        rows = np.lib.stride_tricks.as_strided(self.raw[front:], shape=(h, w * ch), strides=(self.row_bytes, 1))
        rows[:] = px.reshape(h, w * ch)
        self.ptr = self.raw.ctypes.data + front

    def array(self):
        """The image as an H x W x C uint8 view with the buffer's row stride."""
        base = self.raw[self.ptr - self.raw.ctypes.data:]
        return np.lib.stride_tricks.as_strided(base, shape=(self.h, self.w, self.channels), strides=(self.row_bytes, self.channels, 1))


def loader(variant, channels=None, pad=0, offset=0):
    """A parity.check_image `load` hook: the planes go in through the host ("host") or device ("device") entry point.  In the
    CPU-emulated build host memory stands for device memory, so "device" hands over the buffer itself."""
    keep = []

    def load(ctx, planes, slot):
        c = planes.shape[0]
        img = Interleaved(planes, channels, pad, offset)
        keep.append(img)
        if variant == "host":
            ctx.set_image_interleaved_ptr(img.ptr, img.row_bytes, img.channels, c, img.w, img.h, slot)
        else:
            ctx.set_image_interleaved_device(img.ptr, img.row_bytes, img.channels, c, img.w, img.h, slot)
        ctx.sync()
    return load
