"""Input contract of the reference (`src/data.py:28-55,70-86`): `inputs(datadir, dataset, batch_size)`
returns `(images [B,480,640,3], depths [B,h,w,1])`, float32 in [0,1], NHWC -- here as CUDA tensors that
are refilled in place by `next_batch()` (the reference's queue runners do the same behind the graph).

Two sources:
  * synthetic (default when `<datadir>/<dataset>/<split>.tfrecords` is absent): U[0,1) images and
    U[0.05,1) depths, the shapes of BASELINE.json's configs;
  * TFRecords written by the reference's `tools/data_tf_converter.py:41-53`: `tf.train.Example`s with
    raw float32 `image` / `depth` bytes stored as value/255 - 0.5 (read back with +0.5, src/data.py:84-85)
    and six int64 dims.  Parsed with a minimal pure-Python TFRecord + protobuf reader (no TensorFlow).
"""
from __future__ import annotations

import os
import queue
import struct
import threading

import torch


def _read_varint(buf, pos):
    result, shift = 0, 0
    while True:
        b = buf[pos]
        pos += 1
        result |= (b & 0x7F) << shift
        if not b & 0x80:
            return result, pos
        shift += 7


def _parse_fields(buf):
    """Yield (field_number, wire_type, value) of one protobuf message (`buf`: bytes or memoryview -- payload slices of a
    memoryview are views, so the multi-megabyte image bytes are not copied on the way down the message tree)."""
    pos, end = 0, len(buf)
    while pos < end:
        key, pos = _read_varint(buf, pos)
        field, wt = key >> 3, key & 7
        if wt == 0:
            v, pos = _read_varint(buf, pos)
        elif wt == 2:
            n, pos = _read_varint(buf, pos)
            v = buf[pos:pos + n]
            pos += n
        elif wt == 1:
            v = buf[pos:pos + 8]
            pos += 8
        elif wt == 5:
            v = buf[pos:pos + 4]
            pos += 4
        else:
            raise ValueError(f"unsupported protobuf wire type {wt}")
        yield field, wt, v


def parse_example(record: bytes) -> dict:
    """tf.train.Example -> {name: bytes | [int]} for BytesList / Int64List features."""
    out = {}
    for f, _, features in _parse_fields(record):                 # Example.features = 1
        if f != 1:
            continue
        for f2, _, entry in _parse_fields(features):             # Features.feature (map entry) = 1
            if f2 != 1:
                continue
            key, val = None, None
            for f3, _, v in _parse_fields(entry):
                if f3 == 1:
                    key = bytes(v).decode()
                elif f3 == 2:
                    for f4, _, lst in _parse_fields(v):           # Feature: bytes_list=1, int64_list=3
                        if f4 == 1:
                            # a memoryview record (the loader's path) keeps zero-copy views of the payload bytes
                            val = [x if isinstance(x, memoryview) else bytes(x)
                                   for f5, _, x in _parse_fields(lst) if f5 == 1]
                            val = val[0] if len(val) == 1 else val
                        elif f4 == 3:
                            ints = []
                            for f5, wt5, x in _parse_fields(lst):
                                if wt5 == 0:
                                    ints.append(x)
                                else:                              # packed
                                    p = 0
                                    while p < len(x):
                                        iv, p = _read_varint(x, p)
                                        ints.append(iv)
                            val = ints
            out[key] = val
    return out


def tfrecord_iterator(path, verify="length"):
    """Yields the raw records of a TFRecord file: u64 length, masked CRC-32C of the length, data, masked CRC-32C of the
    data (the framing `tools/data_tf_converter.py:41-53` writes through `tf.python_io.TFRecordWriter`).
    verify = "length" (default): the length CRC of every record is checked -- a corrupted length would otherwise send
    the reader to a garbage offset -- and the data CRC of records up to 64 KB; "full": every data CRC too (pure-Python
    CRC-32C, about 1 s per MB); None: nothing.  A truncated record raises instead of ending the iteration silently."""
    from .summary import masked_crc32c
    with open(path, "rb") as f:
        index = 0
        while True:
            head = f.read(12)
            if not head:
                return
            if len(head) < 12:
                raise IOError(f"{path}: truncated header of record {index}")
            (n,) = struct.unpack("<Q", head[:8])
            if verify and struct.unpack("<I", head[8:12])[0] != masked_crc32c(head[:8]):
                raise IOError(f"{path}: corrupted length of record {index}")
            data = f.read(n)
            tail = f.read(4)
            if len(data) < n or len(tail) < 4:
                raise IOError(f"{path}: truncated record {index} ({len(data)} of {n} bytes)")
            if (verify == "full" or (verify and n <= 65536)) and struct.unpack("<I", tail)[0] != masked_crc32c(data):
                raise IOError(f"{path}: corrupted data of record {index}")
            index += 1
            yield data


def tfrecord_index(path):
    """[(payload offset, payload length)] of every record, from the headers alone (the payloads are not read)."""
    from .summary import masked_crc32c
    out = []
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        pos = 0
        while pos < size:
            head = f.read(12)
            if len(head) < 12:
                raise IOError(f"{path}: truncated header of record {len(out)}")
            (n,) = struct.unpack("<Q", head[:8])
            if struct.unpack("<I", head[8:12])[0] != masked_crc32c(head[:8]):
                raise IOError(f"{path}: corrupted length of record {len(out)}")
            if pos + 12 + n + 4 > size:
                raise IOError(f"{path}: truncated record {len(out)}")
            out.append((pos + 12, n))
            pos += 12 + n + 4
            f.seek(pos)
    return out


class _SyntheticSource:
    """U[0,1) images and U[0.05,1) depths (the shapes of BASELINE.json's configs), generated on the host."""

    def __init__(self, seed):
        self.gen = torch.Generator().manual_seed(seed)
        self.lock = threading.Lock()

    def fill(self, images, depths):
        with self.lock:                               # one generator: batches come out in a reproducible order
            torch.rand(images.shape, generator=self.gen, out=images)
            torch.rand(depths.shape, generator=self.gen, out=depths)
        depths.mul_(0.95).add_(0.05)


class _RecordSource:
    """`tf.train.shuffle_batch(capacity=20*B, min_after_dequeue=5*B)` over the records of one TFRecord file read in
    file order, epoch after epoch (src/data.py:33-55): a pool of up to 20*B pending records is refilled from the file and
    a uniformly random one is dequeued while the pool holds more than 5*B.  The pool keeps record OFFSETS; a payload
    (3.7 MB per 640x480 image) is read and parsed only when its record is dequeued."""

    def __init__(self, path, batch, seed):
        self.path, self.index = path, tfrecord_index(path)
        if not self.index:
            raise IOError(f"{path}: no records")
        self.gen = torch.Generator().manual_seed(seed)
        self.capacity, self.min_after = 20 * batch, 5 * batch
        self.pool, self.cursor = [], 0
        self.lock = threading.Lock()
        self.local = threading.local()
        e = self.read(0)
        self.image_hw = (e["image_height"][0], e["image_width"][0])
        self.depth_hw = (e["depth_height"][0], e["depth_width"][0])

    def read(self, i):
        f = getattr(self.local, "f", None)
        if f is None:
            f = self.local.f = open(self.path, "rb")
        off, n = self.index[i]
        f.seek(off)
        buf = bytearray(n)                       # writable: torch.frombuffer can wrap the payload without a copy
        if f.readinto(buf) != n:
            raise IOError(f"{self.path}: short read of record {i}")
        return parse_example(memoryview(buf))

    def _dequeue(self):
        with self.lock:
            while len(self.pool) < self.capacity:
                self.pool.append(self.cursor)
                self.cursor = (self.cursor + 1) % len(self.index)        # epochs=None: the file repeats forever
                if len(self.pool) > self.min_after and len(self.pool) >= len(self.index):
                    break
            j = int(torch.randint(len(self.pool), (1,), generator=self.gen))
            self.pool[j], self.pool[-1] = self.pool[-1], self.pool[j]
            return self.pool.pop()

    def fill(self, images, depths):
        for i in range(images.shape[0]):
            e = self.read(self._dequeue())
            im = torch.frombuffer(e["image"], dtype=torch.float32)
            dp = torch.frombuffer(e["depth"], dtype=torch.float32)
            torch.add(im.view(images.shape[1:]), 0.5, out=images[i])        # src/data.py:84-85
            torch.add(dp.view(depths.shape[1:]), 0.5, out=depths[i])


class _SequentialSource(_RecordSource):
    """One pass over the records of a TFRecord file in file order, no shuffle pool (evaluation on the test split):
    shard (r, n) takes records r, r + n, r + 2n, ...  `fill` returns how many rows it wrote (0 at the end)."""

    def __init__(self, path, batch, shard=(0, 1)):
        super().__init__(path, batch, 0)
        rank, world = shard
        if not 0 <= rank < world:
            raise ValueError(f"shard {shard}: need 0 <= rank < world")
        self.order = list(range(rank, len(self.index), world))
        self.cursor = 0

    def _dequeue(self):
        with self.lock:
            if self.cursor >= len(self.order):
                return None
            self.cursor += 1
            return self.order[self.cursor - 1]

    def fill(self, images, depths):
        for i in range(images.shape[0]):
            j = self._dequeue()
            if j is None:
                return i
            e = self.read(j)
            im = torch.frombuffer(e["image"], dtype=torch.float32)
            dp = torch.frombuffer(e["depth"], dtype=torch.float32)
            torch.add(im.view(images.shape[1:]), 0.5, out=images[i])
            torch.add(dp.view(depths.shape[1:]), 0.5, out=depths[i])
        return images.shape[0]


class Inputs:
    """`images`, `depths`: persistent CUDA buffers (the op's input tensors); `next_batch()` refills them in place.

    The reference feeds its graph from queue-runner threads (`shuffle_batch(num_threads=2)`, src/data.py:51-55).  Here:
    `num_threads` worker threads fill a ring of pinned host batches; `next_batch()` takes the oldest one, starts its
    host->device copy on a copy stream into one of two device staging buffers -- that copy overlaps the step the caller
    enqueued before -- and copies the previous staging buffer into `images` / `depths` on the caller's stream (device to
    device, ~60 us).  The loop therefore runs at max(step, PCIe copy, host fill / num_threads), not at their sum.
    `synthetic="device"`: without a TFRecord file the batch is drawn on the GPU straight into `images` / `depths`
    (no host work at all: the train loop then runs at the benchmark's device-resident speed).

    `epochs=1` (evaluation; beyond the reference): every record of the file (of the shard `(rank, world)`: records rank,
    rank + world, ...) exactly once, in file order, one reader thread; no batch is taken at construction.
    `next_batch()` then returns the number of rows it filled -- the last batch may be partial (its trailing rows are
    stale) -- and 0 once the file is exhausted.  The file must exist."""

    def __init__(self, datadir, dataset, batch_size=32, train_or_test="train", device="cuda", seed=0,
                 image_hw=(480, 640), depth_hw=(55, 73), synthetic="device", num_threads=2, host_slots=3, epochs=None,
                 shard=(0, 1)):
        self.B, self.device = batch_size, torch.device(device)
        self.path = os.path.join(datadir, dataset, f"{train_or_test}.tfrecords")      # src/data.py:58-59
        self.source = None
        if epochs not in (None, 1):
            raise ValueError("epochs must be None (repeat forever, shuffled) or 1 (one ordered pass)")
        self.single_pass, self._exhausted = epochs == 1, False
        if self.single_pass:
            if not os.path.exists(self.path):
                raise FileNotFoundError(f"{self.path} not found")
            self.source = _SequentialSource(self.path, batch_size, shard)
            image_hw, depth_hw = self.source.image_hw, self.source.depth_hw
            num_threads = 1                            # batches must come out in file order
        elif os.path.exists(self.path):
            self.source = _RecordSource(self.path, batch_size, seed)
            image_hw, depth_hw = self.source.image_hw, self.source.depth_hw
        elif synthetic == "host":
            self.source = _SyntheticSource(seed)
        self.image_hw, self.depth_hw = image_hw, depth_hw
        self.images = torch.empty(batch_size, *image_hw, 3, device=self.device)
        self.depths = torch.empty(batch_size, *depth_hw, 1, device=self.device)
        self._threads, self._closed = [], False
        if self.source is None:
            self.gen = torch.Generator(device=self.device).manual_seed(seed)
        else:
            pin = self.device.type == "cuda"
            self._h = [(torch.empty(batch_size, *image_hw, 3, pin_memory=pin), torch.empty(batch_size, *depth_hw, 1, pin_memory=pin))
                       for _ in range(max(host_slots, 2))]
            self._free, self._ready = queue.Queue(), queue.Queue(maxsize=len(self._h))
            for k in range(len(self._h)):
                self._free.put(k)
            if pin:
                self._d = [(torch.empty_like(self.images), torch.empty_like(self.depths)) for _ in range(2)]
                self._copy_stream = torch.cuda.Stream(device=self.device)
                self._staged = [torch.cuda.Event() for _ in range(2)]        # H2D into staging buffer j finished
                self._drained = [torch.cuda.Event() for _ in range(2)]       # staging buffer j was copied out
                for ev in self._drained:
                    ev.record(torch.cuda.current_stream())
            self._inflight = None            # (host slot, staging index) whose H2D is under way
            self._rows = [batch_size] * len(self._h)        # rows the last fill of each host slot wrote
            self._n = 0
            for _ in range(max(num_threads, 1)):
                t = threading.Thread(target=self._worker, daemon=True)
                t.start()
                self._threads.append(t)
            self._prefetch()
        if not self.single_pass:
            self.next_batch()

    # ---- worker threads: host batches
    def _worker(self):
        while not self._closed:
            try:
                k = self._free.get(timeout=0.1)
            except queue.Empty:
                continue
            try:
                rows = self.source.fill(*self._h[k])
                self._rows[k] = self.B if rows is None else rows
                self._ready.put((k, None))
                if rows == 0:                                        # single pass: nothing left to read
                    return
            except Exception as e:                                   # surface reader errors in the training thread
                self._ready.put((k, e))
                return

    def _take_ready(self):
        while True:
            try:
                k, err = self._ready.get(timeout=0.1)
                break
            except queue.Empty:
                # a worker exits after its first error (or at the end of a single pass); once none is left, nothing
                # will arrive -- fail instead of waiting forever
                if not any(t.is_alive() for t in self._threads) and self._ready.empty():
                    raise IOError(f"{self.path}: no reader thread left (an earlier read failed)")
        if err is not None:
            raise err
        return k

    def _prefetch(self):
        """Start the host->device copy of the next host batch (waits for a worker only if none is ready yet)."""
        k = self._take_ready()
        if self.device.type != "cuda":
            self._inflight = (k, None)
            return
        j = self._n % 2
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._drained[j])
            self._d[j][0].copy_(self._h[k][0], non_blocking=True)
            self._d[j][1].copy_(self._h[k][1], non_blocking=True)
            self._staged[j].record(self._copy_stream)
        self._inflight = (k, j)
        self._n += 1

    def next_batch(self):
        if self.source is None:                        # synthetic, drawn on the device
            self.images.uniform_(0.0, 1.0, generator=self.gen)
            self.depths.uniform_(0.05, 1.0, generator=self.gen)
            return self.images, self.depths
        if self._exhausted:
            return 0
        k, j = self._inflight
        rows = self._rows[k]
        if j is None:                                  # CPU tensors (tests): plain copies
            self.images.copy_(self._h[k][0])
            self.depths.copy_(self._h[k][1])
            self._free.put(k)
        else:
            cur = torch.cuda.current_stream()
            cur.wait_event(self._staged[j])
            self.images.copy_(self._d[j][0], non_blocking=True)
            self.depths.copy_(self._d[j][1], non_blocking=True)
            self._drained[j].record(cur)
            self._staged[j].synchronize()              # the H2D has read the pinned batch: hand it back to the workers
            self._free.put(k)
        if self.single_pass:
            if rows == 0:
                self._exhausted = True
                return 0
            self._prefetch()
            return rows
        self._prefetch()                               # overlaps the step the caller enqueues next
        return self.images, self.depths

    def close(self):
        self._closed = True
        for t in self._threads:
            t.join(timeout=2.0)
        self._threads = []

    def __del__(self):
        self._closed = True


def inputs(datadir, dataset, batch_size=32, train_or_test="train", epochs=None, **kw):
    """Same call as the reference's `data.inputs` (src/data.py:28-29); returns an `Inputs` object whose
    `.images` / `.depths` are the tensors to hand to `models.<model>(images, depths)`.  `epochs=1` (with `shard=(rank,
    world)`): one ordered pass for evaluation, see `Inputs`."""
    return Inputs(datadir, dataset, batch_size, train_or_test, epochs=epochs, **kw)
