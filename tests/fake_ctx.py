"""An in-memory stand-in for device.Context: engines plan, load weights and enqueue whole steps against it on the CPU.

Buffers are host byte arrays at deterministic fake addresses (handed out in allocation order), so weight I/O round-trips
through real bytes and two engines built the same way see the same pointers. `call` runs nothing; it records the
entry-point name in `trace` and the name with its arguments in `calls`."""
import ctypes as C

import numpy as np


class FakeBuffer:
    def __init__(self, ptr, nbytes):
        self.ptr, self.nbytes = ptr, int(nbytes)
        self.data = bytearray(self.nbytes)

    @property
    def p(self):
        return C.c_void_p(self.ptr)

    def at(self, byte_offset):
        return C.c_void_p(self.ptr + int(byte_offset))

    def upload(self, arr, stream=None, byte_offset=0):
        b = np.ascontiguousarray(arr).tobytes()
        assert byte_offset + len(b) <= self.nbytes, (len(b), self.nbytes)
        self.data[byte_offset:byte_offset + len(b)] = b
        return self

    def download(self, dtype, shape, stream=None, byte_offset=0):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        assert byte_offset + n <= self.nbytes, (n, self.nbytes)
        return np.frombuffer(bytes(self.data[byte_offset:byte_offset + n]), dtype).reshape(shape).copy()

    def zero(self, stream=None):
        self.data[:] = bytes(self.nbytes)
        return self

    def free(self):
        pass


class _FakeLib:
    """Workspace queries and shape checks of the library: every query answers 256."""

    def __getattr__(self, name):
        return lambda *args: 256


class FakeContext:
    def __init__(self):
        self.trace, self.calls, self.allocs = [], [], []
        self._next = 1 << 20
        self._streams = 1
        self.h = None
        self.tag = ""
        self._prof = None
        self.stream = C.c_void_p(1)
        self.lib = _FakeLib()

    def alloc(self, nbytes):
        b = FakeBuffer(self._next, nbytes)
        self._next += (int(nbytes) + 255) // 256 * 256
        self.allocs.append(int(nbytes))
        return b

    def call(self, name, *args):
        self.trace.append(name)
        self.calls.append((name, args))
        return 0

    def new_event(self):
        return C.c_void_p(2)

    def new_stream(self):
        self._streams += 1
        return C.c_void_p(1 << 10 | self._streams)

    def record(self, ev, stream=None):
        pass

    def sync(self, stream=None):
        pass

    def attach_comm(self, rank, world, unique_id):
        pass
