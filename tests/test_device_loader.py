"""Device-side batch assembly from PCM WAV files (cpc_b200.device_loader, cpc_pcm_assemble).

CPU: the segment planner against ``AudioDataset.__getitem__`` (its staged bytes decoded with read_wav's arithmetic),
refusals, C-ABI rejections, trainer refusals, the producer thread's lifetime and that its copies run without the GIL.
One GPU: every batch of several sampler epochs bit-identical to ``torch.stack([ds[i] for i in batch])``, strided output
rows, ``train`` / ``validate`` with ``device_loading=True`` against the DataLoader path.  Two GPUs (skips on one):
tests/device_loader_worker.py.
"""
import ctypes
import os
import random
import struct
import subprocess
import sys
import threading
import time
import wave

import numpy as np
import pytest
import torch

from cpc_b200 import device_loader as DL
from cpc_b200.audio_dataset import AudioDataset, AudioTestingDataset
from cpc_b200.sampler import FileBatchSampler

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "device_loader_worker.py")


# ---------------------------------------------------------------------------------------------------
# synthetic WAV folders
# ---------------------------------------------------------------------------------------------------

def _samples(rng, frames, channels, width):
    """Random integer samples over the whole range of the width, extremes included."""
    if width == 1:
        x = rng.integers(0, 256, size=(frames, channels), dtype=np.int64)
        x.flat[:2] = (0, 255)
        return x
    lo, hi = -(1 << (8 * width - 1)), (1 << (8 * width - 1)) - 1
    x = rng.integers(lo, hi + 1, size=(frames, channels), dtype=np.int64)
    if frames * channels >= 4:
        x.flat[:4] = (lo, hi, -1, (1 << 24) + 1 if width == 4 else 0)   # 2^24 + 1 rounds in int32 -> fp32
    return x


def _pcm_bytes(x, width):
    if width == 1:
        return x.astype(np.uint8).tobytes()
    if width == 3:
        v = x.astype(np.int64) & 0xFFFFFF
        return np.stack([v & 0xFF, (v >> 8) & 0xFF, (v >> 16) & 0xFF], axis=-1).astype(np.uint8).tobytes()
    return x.astype({2: "<i2", 4: "<i4"}[width]).tobytes()


def write_wav(path, frames, channels=1, width=2, seed=0):
    x = _samples(np.random.default_rng(seed), frames, channels, width)
    with wave.open(str(path), "wb") as fh:
        fh.setnchannels(channels)
        fh.setsampwidth(width)
        fh.setframerate(16000)
        fh.writeframes(_pcm_bytes(x, width))


def write_raw_wav(path, tag, channels, bits, payload, subformat=None, extra_chunk=False):
    """A RIFF WAVE file written by hand: any format tag, WAVE_FORMAT_EXTENSIBLE, a chunk before ``fmt ``."""
    block = channels * ((bits + 7) // 8)
    fmt = struct.pack("<HHIIHH", tag, channels, 16000, 16000 * block, block, bits)
    if subformat is not None:
        fmt += struct.pack("<HHI", 22, bits, 0) + subformat
    body = b"WAVE"
    if extra_chunk:
        body += b"LIST" + struct.pack("<I", 3) + b"abc\x00"          # odd size: padded to even
    body += b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(payload)) + payload
    with open(path, "wb") as fh:
        fh.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def make_folder(root, lengths, channels=1, width=2, seed=0):
    root.mkdir(parents=True, exist_ok=True)
    for i, n in enumerate(lengths):
        write_wav(root / ("f%02d.wav" % i), n, channels, width, seed + i)
    return root


# ---------------------------------------------------------------------------------------------------
# read_wav's arithmetic on staged bytes (what the kernel computes)
# ---------------------------------------------------------------------------------------------------

def decode_staged(buf, table, header, batch, length):
    out = np.full((batch, length), np.nan, dtype=np.float32)
    for s in table:
        n, w, a = int(s["frames"]), int(s["sample_width"]), int(s["block_align"])
        at = header + int(s["src_byte_offset"])
        raw = np.frombuffer(buf[at:at + n * a].tobytes(), dtype=np.uint8).reshape(n, a)[:, :w]
        if w == 1:
            v = (raw[:, 0].astype(np.float32) - 128.0) / 128.0
        elif w == 2:
            v = raw.copy().view("<i2")[:, 0].astype(np.float32) / 32768.0
        elif w == 3:
            b = raw.astype(np.int32)
            u = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
            v = (u - ((u & 0x800000) << 1)).astype(np.float32) / 8388608.0
        else:
            v = raw.copy().view("<i4")[:, 0].astype(np.float32) / 2147483648.0
        o = int(s["dst_offset"])
        out[int(s["dst_item"]), o:o + n] = v
    return torch.from_numpy(out)


def staged_batch(planner, indices):
    holder = {}

    def buffer_for(nbytes):
        holder["buf"] = np.zeros(nbytes, dtype=np.uint8)
        return holder["buf"]
    table, header, total = planner.stage(indices, buffer_for)
    assert total == len(holder["buf"])
    return decode_staged(holder["buf"], table, header, len(indices), planner.item_length), table


def stock_item(ds, i):
    item = ds[i]
    return item[0] if isinstance(item, tuple) else item


def assert_planner_matches(ds):
    planner = DL.SegmentPlanner(ds)
    n = len(ds)
    assert n >= 2
    order = list(range(n))
    random.Random(n).shuffle(order)
    for start in range(0, n, 5):                                    # batches of up to 5 items, last item included
        idx = order[start:start + 5]
        got, table = staged_batch(planner, idx)
        want = torch.stack([stock_item(ds, i) for i in idx])
        assert got.dtype == want.dtype == torch.float32
        assert torch.equal(got, want), idx
    return planner


# (file lengths, item_length, unique_length): several files per item, overlapping items, a long file
LAYOUTS = {"spans": ([700, 150, 90, 60, 1200, 333, 97, 500], 256, 256),
           "overlap": ([700, 150, 90, 60, 1200, 333, 97, 500], 300, 113)}


# ---------------------------------------------------------------------------------------------------
# CPU: planner, refusals
# ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("channels", [1, 3])
@pytest.mark.parametrize("width", [1, 2, 3, 4])
def test_planner_reproduces_getitem(tmp_path, width, channels, layout):
    lengths, item, unique = LAYOUTS[layout]
    root = make_folder(tmp_path / "d", lengths, channels, width, seed=width * 10 + channels)
    ds = AudioDataset(root, item_length=item, unique_length=unique)
    planner = assert_planner_matches(ds)
    assert max(len(planner.item_pieces(i)) for i in range(len(ds))) >= 3    # an item spans >= 3 files
    info = planner.files[0]
    assert (info.channels, info.sample_width, info.block_align) == (channels, width, channels * width)


@pytest.mark.parametrize("testing", [False, True])
def test_planner_without_crossing_files(tmp_path, testing):
    root = make_folder(tmp_path / "d", [900, 640, 1500, 700], 1, 2, seed=3)
    cls = AudioTestingDataset if testing else AudioDataset
    ds = cls(root, item_length=200, unique_length=150, cross_files=False)
    planner = assert_planner_matches(ds)
    assert planner.labels == testing
    idx = list(range(len(ds)))
    if testing:
        assert planner.file_labels(idx) == [int(ds[i][1]) for i in idx]


def test_planner_short_items_and_the_last_item(tmp_path):
    """Many tiny files: items that cross many boundaries lose one frame per file left, so near the end the stock path
    returns a short item (or indexes past the last file).  The planner reproduces every full item and raises ValueError
    exactly where the stock item is not full."""
    root = make_folder(tmp_path / "d", [40] * 12 + [2] * 12, 1, 2, seed=5)
    ds = AudioDataset(root, item_length=64, unique_length=48)
    planner = DL.SegmentPlanner(ds)
    short = 0
    for i in range(len(ds)):
        try:
            want = ds[i]
            full = want.shape[0] == ds.item_length
        except IndexError:
            full = False
        if full:
            got, _ = staged_batch(planner, [i])
            assert torch.equal(got[0], want), i
        else:
            short += 1
            with pytest.raises(ValueError):
                planner.item_pieces(i)
    assert short >= 1 and len(ds) - short >= 3


def test_wav_index_reads_extensible_pcm_and_skips_padded_chunks(tmp_path):
    x = _samples(np.random.default_rng(1), 300, 2, 3)
    sub = DL._KSDATAFORMAT_SUBTYPE_PCM
    write_raw_wav(tmp_path / "a.wav", 0xFFFE, 2, 24, _pcm_bytes(x, 3), subformat=sub, extra_chunk=True)
    write_raw_wav(tmp_path / "b.wav", 1, 2, 24, _pcm_bytes(x[::-1].copy(), 3), extra_chunk=True)
    info = DL.parse_wav(tmp_path / "a.wav")
    assert (info.channels, info.sample_width, info.block_align, info.frames) == (2, 3, 6, 300)
    assert_planner_matches(AudioDataset(tmp_path, item_length=128, unique_length=100))


def test_refusals_list_the_offending_files(tmp_path):
    good = make_folder(tmp_path / "mixed", [500, 500], 1, 2)
    write_raw_wav(good / "float.wav", 3, 1, 32, np.zeros(400, "<f4").tobytes())
    write_raw_wav(good / "ext_float.wav", 0xFFFE, 1, 32, np.zeros(400, "<f4").tobytes(),
                  subformat=b"\x03\x00\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71")
    (good / "song.mp3").write_bytes(b"ID3" + bytes(200))
    ds = AudioDataset.__new__(AudioDataset)                         # the stock constructor would try to decode them
    ds.files, ds.max_file_count, ds.dummy_load, ds.dtype = sorted(good.iterdir()), 5, False, torch.FloatTensor
    with pytest.raises(ValueError) as err:
        DL.SegmentPlanner(ds)
    msg = str(err.value)
    for name in ("float.wav", "ext_float.wav", "song.mp3"):
        assert name in msg, msg
    assert "f00.wav" not in msg and "f01.wav" not in msg

    ok = AudioDataset(make_folder(tmp_path / "ok", [500, 500]), item_length=100)
    ok.dummy_load = True
    with pytest.raises(ValueError, match="dummy_load"):
        DL.SegmentPlanner(ok)
    ok.dummy_load = False
    ok.dtype = torch.DoubleTensor
    with pytest.raises(ValueError, match="dtype"):
        DL.SegmentPlanner(ok)
    with pytest.raises(ValueError, match="AudioDataset"):
        DL.SegmentPlanner(torch.utils.data.TensorDataset(torch.zeros(3)))
    with pytest.raises(ValueError, match="CUDA"):
        DL.DeviceBatchLoader(AudioDataset(tmp_path / "ok", item_length=100), [[0]], "cpu")


# ---------------------------------------------------------------------------------------------------
# CPU: C-ABI rejections (no device touched)
# ---------------------------------------------------------------------------------------------------

def _table(rows):
    from cpc_b200 import ops
    return np.array(rows, dtype=ops.PCM_SEGMENT_DTYPE)


def test_segment_layout_matches_the_c_struct():
    from cpc_b200 import _lib, ops
    assert ctypes.sizeof(_lib.PcmSegment) == ops.PCM_SEGMENT_DTYPE.itemsize == 32
    for name, _ in _lib.PcmSegment._fields_:
        assert getattr(_lib.PcmSegment, name).offset == ops.PCM_SEGMENT_DTYPE.fields[name][1], name
    assert ctypes.sizeof(_lib.PcmParams) == 24


def test_pcm_assemble_rejects_bad_tables_before_the_device(built_lib):
    from cpc_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                                     # never dereferenced: every call below is refused

    def call(rows, batch=2, length=10, stride=None, seg_dev=fake, raw=fake, out=fake, host=True, params=True):
        t = _table(rows)
        p = _lib.PcmParams()
        p.batch, p.item_length, p.out_row_stride, p.n_segments = batch, length, length if stride is None else stride, len(t)
        return lib.cpc_pcm_assemble(ctypes.byref(p) if params else None, ctypes.c_void_p(t.ctypes.data) if host else None,
                                    seg_dev, raw, out, None)

    ok = [(0, 6, 2, 2, 0, 0), (12, 4, 2, 2, 0, 6), (20, 10, 2, 2, 1, 0)]
    bad = {
        "width 0": [(0, 6, 0, 2, 0, 0)] + ok[1:], "width 5": [(0, 6, 5, 5, 0, 0)] + ok[1:],
        "block_align < width": [(0, 6, 2, 1, 0, 0)] + ok[1:],
        "negative frames": [(0, -1, 2, 2, 0, 0)] + ok,
        "negative src offset": [(-2, 6, 2, 2, 0, 0)] + ok[1:],
        "negative dst offset": [(0, 6, 2, 2, 0, -1)] + ok[1:],
        "past item_length": ok[:2] + [(20, 11, 2, 2, 1, 0)],
        "dst_item past batch": ok + [(40, 10, 2, 2, 2, 0)],
        "negative dst_item": [(0, 10, 2, 2, -1, 0)] + ok,
        "gap": [(0, 5, 2, 2, 0, 0), (12, 4, 2, 2, 0, 6), (20, 10, 2, 2, 1, 0)],
        "overlap": [(0, 7, 2, 2, 0, 0), (12, 4, 2, 2, 0, 6), (20, 10, 2, 2, 1, 0)],
        "short item": [(0, 6, 2, 2, 0, 0), (20, 10, 2, 2, 1, 0)],
        "missing item": ok[:2],
        "items out of order": [ok[2], ok[0], ok[1]],
        "offsets out of order": [ok[1], ok[0], ok[2]],
    }
    for case, rows in bad.items():
        assert call(rows) == -1, case
    assert call(ok, stride=9) == -1                                 # row stride < item_length
    assert call(ok, batch=0) == -1 and call(ok, length=0) == -1
    assert call([]) == -1                                           # no segments
    assert call(ok, params=False) == -7 and call(ok, host=False) == -7
    for kw in (dict(seg_dev=None), dict(raw=None), dict(out=None)):
        assert call(ok, **kw) == -7, kw
    assert call(ok, seg_dev=ctypes.c_void_p(260)) == -2             # the table needs 8-byte alignment
    assert call(ok, out=ctypes.c_void_p(258)) == -2


# ---------------------------------------------------------------------------------------------------
# CPU: trainer refusals
# ---------------------------------------------------------------------------------------------------

def _refusing_trainer(tmp_path, device, dummy=False, world=1):
    from cpc_b200 import trainer as T
    ds = AudioDataset(make_folder(tmp_path / "t", [600, 600]), item_length=128)
    ds.dummy_load = dummy
    model = torch.nn.Linear(2, 2)
    t = T.ContrastiveEstimationTrainer(model=model, dataset=ds, validation_set=ds, device=device,
                                       score_function=T.linear_score_function, verbose=False)
    t.rank, t.world = 0, world
    return t


@pytest.mark.parametrize("world", [1, 2])
def test_trainer_refusals_come_before_any_collective(tmp_path, world):
    """With two ranks configured but no process group, a collective would fail with a different error: each refusal
    is a ValueError raised before anything is broadcast."""
    for device, dummy, msg in (("cpu", False, "CUDA"), (None, False, "CUDA"), ("cuda:0", True, "dummy_load")):
        t = _refusing_trainer(tmp_path, device, dummy, world)
        with pytest.raises(ValueError, match=msg):
            t.train(batch_size=2, epochs=1, device_loading=True)
        with pytest.raises(ValueError, match=msg):
            t.validate(batch_size=2, device_loading=True)
        if device is not None and device.startswith("cuda"):
            with pytest.raises(ValueError, match=msg):
                t.validate(batch_size=2, device_loading=True, shard_over_ranks=True)
        assert t.model.training


# ---------------------------------------------------------------------------------------------------
# CPU: the producer thread
# ---------------------------------------------------------------------------------------------------

def _loader_threads():
    return [t for t in threading.enumerate() if t.name == "cpc-device-loader"]


def _drain(producer):
    out = []
    while True:
        staged = producer.next()
        if staged is None:
            return out
        slot, table, header, total, batch = staged
        buf = slot.host.numpy()[:total].copy()
        out.append((batch, decode_staged(buf, table, header, len(batch), producer.planner.item_length)))
        producer.release(slot)


def test_producer_thread_is_joined_at_the_end_on_failure_and_on_close(tmp_path):
    ds = AudioDataset(make_folder(tmp_path / "d", [700, 150, 90, 60, 1200]), item_length=128, unique_length=100)
    planner = DL.SegmentPlanner(ds)
    batches = [[0, 3, 5], [1, 2, 4], [7, 6, 8]]
    assert not _loader_threads()
    p = DL.StagingThread(planner, batches, [DL._Slot(pin=False) for _ in range(2)])
    for batch, got in _drain(p):                                   # normal end
        assert torch.equal(got, torch.stack([ds[i] for i in batch]))
    assert not p.thread.is_alive() and not _loader_threads()
    p = DL.StagingThread(planner, batches[:1] + [[0, len(ds) + 50]], [DL._Slot(pin=False)])
    slot = p.next()[0]
    p.release(slot)
    with pytest.raises(ValueError):                                # an index past the end: the producer's failure
        p.next()
    assert not p.thread.is_alive() and not _loader_threads()
    p = DL.StagingThread(planner, batches * 5, [DL._Slot(pin=False)])
    p.next()                                                       # slot never released: the producer waits for one
    time.sleep(0.1)
    p.close()
    assert not p.thread.is_alive() and not _loader_threads()


def test_staging_copies_run_without_the_gil(tmp_path):
    """While the producer copies one 88 MB item out of a memory-mapped file, this thread keeps running Python: its
    longest stall is a small fraction of the copy.  A copy that held the GIL would stall it for the whole copy."""
    root = tmp_path / "big"
    root.mkdir()
    write_wav(root / "a.wav", 12_000_000, 2, 4, seed=1)            # 96 MB of frames
    ds = AudioDataset(root, item_length=11_000_000, unique_length=11_000_000)
    planner = DL.SegmentPlanner(ds)
    buf = np.ones(100_000_000, dtype=np.uint8)                    # faulted in: the timed copy is the memcpy alone
    planner.stage([0], lambda n: buf[:n])                          # map opened, file pages cached
    took = {}

    def copy():
        t0 = time.perf_counter()
        planner.stage([0], lambda n: buf[:n])
        took["s"] = time.perf_counter() - t0
    worker = threading.Thread(target=copy)
    last, stall = time.perf_counter(), 0.0
    worker.start()
    while worker.is_alive():
        now = time.perf_counter()
        stall, last = max(stall, now - last), now
    worker.join()
    assert took["s"] > 0.004, took
    assert stall < 0.5 * took["s"], (stall, took["s"])


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cpc(built_lib):
    import cpc_b200
    assert cpc_b200._lib.load().cpc_runtime_check() == 0, "device is not a B200 (sm_100)"
    return cpc_b200


class RecordingSampler(torch.utils.data.Sampler):
    def __init__(self, inner):
        self.inner, self.batches = inner, []

    def __iter__(self):
        for b in self.inner:
            self.batches.append(list(b))
            yield b

    def __len__(self):
        return len(self.inner)


FORMATS = [(1, 1), (2, 1), (3, 1), (4, 1), (1, 3), (2, 3), (3, 3), (4, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("prefetch,slow", [(1, False), (3, True)])
@pytest.mark.parametrize("width,channels", FORMATS)
def test_device_batches_equal_the_stacked_items(cpc, tmp_path, width, channels, prefetch, slow):
    lengths, item, unique = LAYOUTS["overlap"]
    root = make_folder(tmp_path / "d", lengths, channels, width, seed=width + 7 * channels)
    datasets = [AudioDataset(root, item_length=item, unique_length=unique),
                AudioTestingDataset(root, item_length=200, unique_length=150)]
    for ds in datasets:
        random.seed(11)
        sampler = RecordingSampler(FileBatchSampler(ds.get_example_count_per_file(), batch_size=4, drop_last=True))
        loader = DL.DeviceBatchLoader(ds, sampler, DEV, prefetch=prefetch)
        seen = 0
        for epoch in range(3):
            for got in loader:
                batch = sampler.batches[seen]
                seen += 1
                if isinstance(ds, AudioTestingDataset):
                    got, labels = got
                    assert torch.equal(labels.cpu(), torch.stack([ds[i][1] for i in batch]))
                if slow:
                    torch.cuda._sleep(2_000_000)                 # the GPU lags: staging slots wait for their kernels
                    time.sleep(0.002)
                want = torch.stack([stock_item(ds, i) for i in batch])
                assert got.is_cuda and got.shape == want.shape
                assert torch.equal(got.cpu(), want), (epoch, batch)
        assert seen == len(sampler.batches) and seen >= 6         # (FileBatchSampler's __len__ is the reference's quirk)
        assert not _loader_threads()


@pytest.mark.gpu
def test_strided_rows_leave_the_padding_untouched(cpc, tmp_path):
    ds = AudioDataset(make_folder(tmp_path / "d", [700, 150, 90, 60, 1200], 3, 3), item_length=256, unique_length=200)
    planner = DL.SegmentPlanner(ds)
    idx = [3, 0, 5, 1]
    buf = {}
    table, header, total = planner.stage(idx, lambda n: buf.setdefault("b", np.zeros(n, dtype=np.uint8)))
    staged = torch.from_numpy(buf["b"]).to(DEV)
    wide = torch.full((len(idx), 300), float("nan"), device=DEV)
    wide[:, 256:] = 7.0
    cpc.ops.pcm_assemble(table, staged[:table.nbytes], staged[header:total], wide[:, :256])
    assert torch.equal(wide[:, :256].cpu(), torch.stack([ds[i] for i in idx]))
    assert bool((wide[:, 256:] == 7.0).all())
    # a table of one frame per segment as a grid check: more segments than one block row
    assert len(table) >= len(idx)


def _raw_wave_setup(cpc, tmp_path, seed=0):
    torch.manual_seed(seed)
    enc = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                            'channel_count': [16, 24, 24, 24, 32], 'bias': True})
    model = cpc.AudioPredictiveCodingModel(enc, cpc.AudioGRUModel(32, 16), enc_size=32, ar_size=16, visible_steps=9,
                                           prediction_steps=4).to(DEV)
    n = model.item_length
    lengths = [3 * n + 17, n // 2, n // 3 + 5, 4 * n, 2 * n + 1, n + 3]
    train_set = AudioDataset(make_folder(tmp_path / "train", lengths, 1, 2, seed=40), item_length=n,
                             unique_length=n * 3 // 4)
    val_set = AudioDataset(make_folder(tmp_path / "val", lengths[::-1], 2, 3, seed=60), item_length=n,
                           unique_length=n // 2)
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=train_set, validation_set=val_set, device=DEV,
                                               score_function=cpc.softplus_score_function, prediction_steps=4,
                                               verbose=False)
    return trainer


@pytest.mark.gpu
def test_train_with_device_loading_sees_the_dataloader_batches(cpc, tmp_path):
    runs = []
    for device_loading in (False, True):
        trainer = _raw_wave_setup(cpc, tmp_path / str(device_loading))
        batches, losses = [], []
        plain = trainer.loss_on_batch

        def recording(batch, plain=plain, batches=batches, losses=losses):
            batches.append(batch.detach().cpu().clone())
            loss, mx = plain(batch)
            losses.append(float(loss.detach()))
            return loss, mx
        trainer.loss_on_batch = recording
        random.seed(123)
        trainer.train(batch_size=4, epochs=2, lr=1e-3, num_workers=0, device_loading=device_loading)
        runs.append((batches, losses))
        assert not _loader_threads()
    (b0, l0), (b1, l1) = runs
    assert len(b0) == len(b1) >= 6
    for x, y in zip(b0, b1):
        assert torch.equal(x, y)
    assert max(abs(x - y) for x, y in zip(l0, l1)) <= 1e-6 * max(1.0, max(abs(x) for x in l0)), (l0, l1)


@pytest.mark.gpu
def test_validate_with_device_loading_equals_validate(cpc, tmp_path):
    trainer = _raw_wave_setup(cpc, tmp_path)
    plain = trainer.validate(batch_size=4, num_workers=0)
    dev = trainer.validate(batch_size=4, device_loading=True)
    assert torch.equal(plain[1], dev[1])                           # accuracies exactly
    assert float((plain[0] - dev[0]).abs().max()) <= 1e-6 * max(1.0, float(plain[0].abs().max()))
    assert abs(plain[2] - dev[2]) <= 1e-6 * max(1.0, abs(plain[2]))
    assert not _loader_threads()
    short = trainer.validate(batch_size=4, device_loading=True, max_steps=1)   # leaves the loop early
    assert torch.equal(short[1], trainer.validate(batch_size=4, num_workers=0, max_steps=1)[1])
    assert not _loader_threads()


@pytest.mark.gpu
def test_two_rank_device_loading(cpc):
    """Two GPUs (skips on one): tests/device_loader_worker.py."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29757", WORKER],
                         capture_output=True, text=True, timeout=400)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RANK_OK 0" in out.stdout and "RANK_OK 1" in out.stdout
