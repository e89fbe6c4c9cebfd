"""Device-side batch assembly for ``AudioDataset``: the host copies raw PCM bytes, one kernel decodes them on the GPU.

The stock input path (``AudioDataset`` + ``torch.utils.data.DataLoader``) opens and seeks a WAV file per item with the
``wave`` module, converts the samples to fp32 with numpy, concatenates the parts of items that cross files, collates
the batch through worker shared memory and pins it -- about 0.6 ms of one host core per e24 item, several cores per
B200.  ``DeviceBatchLoader`` yields the same batches, bit for bit, from three steps:

1. ``SegmentPlanner`` maps a dataset index to the frame ranges ``AudioDataset.__getitem__`` reads (its quirks included:
   the bisect of ``get_position``, the ``item_length + 1`` frames ``load_sample`` reads when they fit, the last frame of
   every file an item leaves, ``cross_files=False``, the final ``[:item_length]``) using the dataset object's own
   ``start_samples`` and ``unique_length``;
2. a background thread copies those frames -- whole interleaved frames, contiguous byte ranges of memory-mapped files --
   into a pinned staging slot, behind the slot's segment table (numpy copies, which run without the GIL);
3. the consuming thread uploads the slot with one asynchronous host-to-device copy on a side stream, and the current
   stream waits for it and runs ``ops.pcm_assemble`` (cpc_pcm_assemble), which writes the (B, L) fp32 batch.

A slot is refilled only after an event recorded behind the kernel that read it has completed, so ``prefetch`` slots
keep that many batches in flight.  Integer PCM WAV files (8/16/24/32-bit, any channel count, first channel read, also
WAVE_FORMAT_EXTENSIBLE with the PCM sub-format) are served; anything ``read_wav`` does not decode natively is refused
when the loader is built.
"""
import collections
import os
import queue
import struct
import threading
import wave

import numpy as np
import torch

from . import ddp, ops
from .audio_dataset import AudioDataset, AudioTestingDataset

_WAVE_FORMAT_PCM = 0x0001
_WAVE_FORMAT_EXTENSIBLE = 0xFFFE
_KSDATAFORMAT_SUBTYPE_PCM = b"\x01\x00\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
_TABLE_ALIGN = 256                                     # raw bytes start this far into a slot

WavInfo = collections.namedtuple("WavInfo", "path data_offset channels sample_width block_align frames")


def parse_wav(path):
    """RIFF ``fmt `` / ``data`` chunks of an integer PCM WAV file -> ``WavInfo`` (byte offset of the first frame, channels,
    bytes per sample, bytes per frame, frames).  Frames are counted as the ``wave`` module counts them: the data chunk's
    size over channels * sample width.  Raises ValueError for anything else (IEEE float, compressed, truncated)."""
    size = os.path.getsize(path)
    with open(path, "rb") as fh:
        head = fh.read(12)
        if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise ValueError("not a RIFF WAVE file")
        fmt, pos = None, 12
        while pos + 8 <= size:
            fh.seek(pos)
            cid, csize = struct.unpack("<4sI", fh.read(8))
            if cid == b"fmt ":
                body = fh.read(min(csize, 40))
                if len(body) < 16:
                    raise ValueError("short fmt chunk")
                tag, channels, _, _, _, bits = struct.unpack_from("<HHIIHH", body)
                if tag == _WAVE_FORMAT_EXTENSIBLE:
                    if len(body) < 40 or body[24:40] != _KSDATAFORMAT_SUBTYPE_PCM:
                        raise ValueError("WAVE_FORMAT_EXTENSIBLE with a sub-format other than integer PCM")
                elif tag != _WAVE_FORMAT_PCM:
                    raise ValueError("format tag 0x%04x is not integer PCM (3 = IEEE float)" % tag)
                width = (bits + 7) // 8
                if channels < 1 or not 1 <= width <= 4:
                    raise ValueError("%d channels of %d-bit samples" % (channels, bits))
                fmt = (channels, width)
            elif cid == b"data":
                if fmt is None:
                    raise ValueError("data chunk before fmt chunk")
                channels, width = fmt
                frames = csize // (channels * width)
                if pos + 8 + frames * channels * width > size:
                    raise ValueError("data chunk runs past the end of the file")
                return WavInfo(str(path), pos + 8, channels, width, channels * width, frames)
            pos += 8 + csize + (csize & 1)                  # chunks are padded to an even size
    raise ValueError("fmt chunk and/or data chunk missing")


def _index_file(path):
    """``parse_wav`` checked against what ``wave`` (and so ``read_wav``) reports for the same file."""
    if os.path.splitext(str(path))[1].lower() != ".wav":
        raise ValueError("not a .wav file (decoded by torchaudio on the stock path)")
    info = parse_wav(path)
    try:
        with wave.open(str(path), "rb") as fh:
            seen = (fh.getnchannels(), fh.getsampwidth(), fh.getnframes())
    except (wave.Error, EOFError) as exc:
        raise ValueError("the wave module cannot open it (%s)" % exc)
    if seen != (info.channels, info.sample_width, info.frames):
        raise ValueError("header parsed as %s, wave reports %s" % ((info.channels, info.sample_width, info.frames), seen))
    return info


class SegmentPlanner:
    """The frame ranges of ``AudioDataset`` items and the staging of whole batches.  Construction indexes every file of
    the dataset and raises ValueError, listing the offending files, for what the device path cannot reproduce."""

    def __init__(self, dataset, max_open_files=32):
        if not isinstance(dataset, AudioDataset):
            raise ValueError("device loading serves AudioDataset / AudioTestingDataset, got %s" % type(dataset).__name__)
        if dataset.dummy_load:
            raise ValueError("device loading cannot serve a dataset with dummy_load (random items, no files)")
        if dataset.dtype is not torch.FloatTensor:
            raise ValueError("device loading produces float32 batches; the dataset's dtype is %s" % (dataset.dtype,))
        self.dataset = dataset
        self.labels = isinstance(dataset, AudioTestingDataset)
        self.files, bad = [], []
        for path in dataset.files[:dataset.max_file_count]:
            try:
                self.files.append(_index_file(path))
            except (ValueError, OSError, struct.error) as exc:
                bad.append("%s: %s" % (path, exc))
        if bad:
            raise ValueError("device loading reads integer PCM WAV files only; cannot serve:\n  " + "\n  ".join(bad))
        self.max_open_files = max(1, int(max_open_files))
        self._maps = collections.OrderedDict()            # file index -> np.memmap, least recently used first

    @property
    def item_length(self):
        return self.dataset.item_length

    def item_pieces(self, idx):
        """[(file index, first frame, frames)] whose first channels, concatenated, are ``dataset[idx]``
        (``AudioDataset.__getitem__`` -> ``load_sample`` -> ``read_wav``, with read_wav's clamping to the file)."""
        ds, length = self.dataset, self.dataset.item_length
        starts = ds.start_samples
        file_index, position = ds.get_position(idx)
        pieces, n = [], length
        while True:
            if file_index + 1 >= len(starts):
                raise ValueError("item %d runs past the last file of the dataset" % idx)
            remaining = position + n + 1 - (starts[file_index + 1] - starts[file_index])
            frames = n + 1 if remaining < 0 else n - remaining
            total = self.files[file_index].frames
            first = max(0, min(int(position), total))
            count = total - first if frames < 0 else max(0, min(int(frames), total - first))
            pieces.append((file_index, first, count))
            if remaining < 0:
                break
            file_index, position, n = file_index + 1, 0, remaining
        out, have = [], 0                                     # the final [:item_length]
        for fi, first, count in pieces:
            count = min(count, length - have)
            if count > 0:
                out.append((fi, first, count))
                have += count
        if have < length:
            raise ValueError("item %d has %d of its %d samples (the stock path fails in collate)" % (idx, have, length))
        return out

    def plan(self, indices):
        """Segment table (ops.PCM_SEGMENT_DTYPE, byte offsets relative to the start of the raw area) and the file byte
        ranges [(file index, byte offset, bytes)] to copy there, in order, for the batch ``indices``."""
        rows, copies, cursor = [], [], 0
        for item, idx in enumerate(indices):
            offset = 0
            for fi, first, count in self.item_pieces(int(idx)):
                info = self.files[fi]
                nbytes = count * info.block_align
                rows.append((cursor, count, info.sample_width, info.block_align, item, offset))
                copies.append((fi, info.data_offset + first * info.block_align, nbytes))
                cursor += nbytes
                offset += count
        return np.array(rows, dtype=ops.PCM_SEGMENT_DTYPE), copies, cursor

    def _map(self, fi):
        mm = self._maps.pop(fi, None)
        if mm is None:
            while len(self._maps) >= self.max_open_files:
                self._maps.popitem(last=False)
            mm = np.memmap(self.files[fi].path, dtype=np.uint8, mode="r")
        self._maps[fi] = mm
        return mm

    def stage(self, indices, buffer_for):
        """Plan ``indices`` and copy their frames into the buffer ``buffer_for(nbytes)`` returns (a uint8 numpy array of
        at least nbytes): the segment table at offset 0, the raw frames from ``header_bytes(len(table))`` on.
        Returns (table, header bytes, total bytes)."""
        table, copies, raw_bytes = self.plan(indices)
        header = header_bytes(len(table))
        buf = buffer_for(header + raw_bytes)
        buf[:table.nbytes] = table.view(np.uint8)
        at = header
        for fi, src, nbytes in copies:
            np.copyto(buf[at:at + nbytes], self._map(fi)[src:src + nbytes])   # releases the GIL
            at += nbytes
        return table, header, header + raw_bytes

    def file_labels(self, indices):
        """AudioTestingDataset's second output: the file index of each item."""
        return [self.dataset.get_position(int(i))[0] for i in indices]

    def close(self):
        self._maps.clear()


def header_bytes(n_segments):
    return -(-n_segments * ops.PCM_SEGMENT_DTYPE.itemsize // _TABLE_ALIGN) * _TABLE_ALIGN


class _Slot:
    """One staging slot: a (pinned) host buffer, its device twin, and the event behind the last kernel that read it."""

    def __init__(self, pin):
        self.pin, self.host, self.dev, self.done = pin, None, None, None

    def host_buffer(self, nbytes):
        if self.host is None or self.host.numel() < nbytes:
            self.host = torch.empty(max(nbytes, 1 << 20) * 5 // 4, dtype=torch.uint8, pin_memory=self.pin)
        return self.host.numpy()

    def wait(self):
        if self.done is not None:
            self.done.synchronize()


_END = object()


class _Failure:
    def __init__(self, exc):
        self.exc = exc


class StagingThread:
    """Background producer: stages each batch of ``batches`` into a free slot and queues (slot, table, header bytes, total
    bytes, batch).  A slot comes back through ``release``; it is refilled after ``slot.wait()``.  ``close`` stops and
    joins the thread; it is also called when the batches are exhausted or the producer fails."""

    def __init__(self, planner, batches, slots, device=None):
        self.planner, self.batches, self.device = planner, batches, device
        self.free, self.ready = queue.Queue(), queue.Queue()
        for s in slots:
            self.free.put(s)
        self.stop = threading.Event()
        self.thread = threading.Thread(target=self._run, name="cpc-device-loader", daemon=True)
        self.thread.start()

    def _run(self):
        try:
            if self.device is not None:
                torch.cuda.set_device(self.device)         # pinned allocations and event waits on the loader's device
            for batch in self.batches:
                slot = None
                while slot is None:
                    if self.stop.is_set():
                        return
                    try:
                        slot = self.free.get(timeout=0.05)
                    except queue.Empty:
                        pass
                slot.wait()
                table, header, total = self.planner.stage(batch, slot.host_buffer)
                self.ready.put((slot, table, header, total, batch))
            self.ready.put(_END)
        except BaseException as exc:                      # noqa: BLE001 -- handed to the consumer, raised there
            self.ready.put(_Failure(exc))

    def next(self):
        """The next staged batch, or None at the end; re-raises a failure of the producer.  The thread is joined in
        both of those cases."""
        item = self.ready.get()
        if item is _END or isinstance(item, _Failure):
            self.close()
            if item is _END:
                return None
            raise item.exc
        return item

    def release(self, slot):
        self.free.put(slot)

    def close(self):
        self.stop.set()
        if self.thread.is_alive() and self.thread is not threading.current_thread():
            self.thread.join()


class DeviceBatchLoader:
    """Iterates like ``DataLoader(dataset, batch_sampler=batch_sampler)`` followed by ``.to(device)``: CUDA (B/W, L)
    float32 batches (and, for AudioTestingDataset, the (B/W,) int64 file labels), bit-identical to
    ``torch.stack([dataset[i] for i in batch])``.

    With ``world`` > 1, rank 0 iterates ``batch_sampler`` and the epoch's batches are broadcast
    (``ddp.ShardedBatchSampler``); each rank plans, copies and decodes only its contiguous shard.  The sampler is iterated
    in the calling thread when an epoch starts, as the DataLoader does, so its use of Python's ``random`` is unchanged.
    ``prefetch``: staging slots, i.e. batches staged ahead of the consumer.  ``max_open_files``: memory maps kept open.
    Raises ValueError at construction for a non-CUDA device or a dataset it cannot serve (``SegmentPlanner``).
    The producer thread is joined when an epoch ends, when it fails, and on ``close()``."""

    def __init__(self, dataset, batch_sampler, device, rank=0, world=1, prefetch=2, max_open_files=32):
        device = torch.device(device) if device is not None else None
        if device is None or device.type != "cuda":
            raise ValueError("device loading decodes on a CUDA device, got device %r" % (device,))
        if prefetch < 1:
            raise ValueError("prefetch must be at least 1, got %d" % prefetch)
        self.planner = SegmentPlanner(dataset, max_open_files)
        self.device = device if device.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.batch_sampler = ddp.ShardedBatchSampler(batch_sampler, rank, world) if world > 1 else batch_sampler
        self.slots = [_Slot(pin=True) for _ in range(prefetch)]
        self._side = None
        self._producer = None

    def __len__(self):
        return len(self.batch_sampler)

    def __iter__(self):
        self.close()                                      # an unfinished earlier epoch
        batches = [list(b) for b in iter(self.batch_sampler)]
        self._producer = StagingThread(self.planner, batches, self.slots, self.device)
        return _Epoch(self, self._producer)

    def _launch(self, staged):
        slot, table, header, total, batch = staged
        cur = torch.cuda.current_stream(self.device)
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        side = self._side
        if slot.dev is None or slot.dev.numel() < total:
            slot.dev = torch.empty(slot.host.numel(), dtype=torch.uint8, device=self.device)
            side.wait_stream(cur)                        # a fresh block may still be in use by earlier work on cur
        elif slot.done is not None:
            side.wait_event(slot.done)                   # the last kernel that read slot.dev has finished
        with torch.cuda.stream(side):
            slot.dev[:total].copy_(slot.host[:total], non_blocking=True)
        slot.dev.record_stream(side)
        uploaded = torch.cuda.Event()
        uploaded.record(side)
        cur.wait_event(uploaded)
        out = torch.empty((len(batch), self.planner.item_length), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            ops.pcm_assemble(table, slot.dev[:table.nbytes], slot.dev[header:total], out)
        slot.done = torch.cuda.Event()
        slot.done.record(cur)
        self._producer.release(slot)
        if self.planner.labels:
            labels = torch.tensor(self.planner.file_labels(batch), dtype=torch.int64).to(self.device)
            return out, labels
        return out

    def close(self):
        """Stop and join the producer thread of the current epoch (no-op when none is running)."""
        if self._producer is not None:
            self._producer.close()
            self._producer = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:                                 # noqa: BLE001 -- interpreter shutdown
            pass


class _Epoch:
    def __init__(self, loader, producer):
        self.loader, self.producer = loader, producer

    def __iter__(self):
        return self

    def __next__(self):
        if self.producer is None or self.loader._producer is not self.producer:
            raise StopIteration                          # closed
        try:
            staged = self.producer.next()
            if staged is None:
                raise StopIteration
            return self.loader._launch(staged)
        except BaseException:
            self.close()
            raise

    def close(self):
        if self.producer is not None:
            self.producer.close()
            if self.loader._producer is self.producer:
                self.loader._producer = None
            self.producer = None
