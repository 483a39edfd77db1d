"""Teacher-embedding dump (SURVEY.md §8 row A21) and its on-disk store.

Reference behaviour being replaced:
  * `save_embeddings_one_epoch` (stage1/save_embedding_image_stage1.py:69-126): per batch, teacher forward ->
    `outputs.to(float16, cpu)` -> one record per image `int32 seed || fp16[C*E*E]` handed to a writer process.
  * the store (stage1/data/augmentation/manager.py:7-162): per rank a pair `rank{r}-keys.txt` (one key per line, first
    occurrence wins) + `rank{r}-values.bin` (fixed-size records in key order); written into a temporary directory next to
    the target and moved into place when the writer closes; readers visit packages starting from their own rank.
  * the student side decodes a record as seed = int32 at offset 0, embedding = fp16[topk * num_embedding] after it
    (stage1/data/augmentation/dataset_wrapper.py:50-62).

B200 design: the fp32 -> fp16 cast runs on the device (es3_cast_f32_to_f16) so the D2H copy moves 2 B/element; device and
pinned host staging are double-buffered; the copy is issued on a side stream behind an event, and a host thread turns
finished buffers into records -- so batch i's D2H and file writes overlap batch i+1's teacher forward (the reference
synchronises the device and copies synchronously every batch).
"""
from __future__ import annotations

import os
import queue
import shutil
import tempfile
import threading

import numpy as np
import torch

from .. import ops

SEED_BYTES = 4


def item_size(embed_dim: int, num_embedding: int) -> int:
    """Record size in bytes (dataset_wrapper.py:84-86): 4-byte seed + fp16 embedding."""
    return embed_dim * 2 * num_embedding + SEED_BYTES


def encode_record(seed, embedding_f16: np.ndarray) -> bytes:
    assert embedding_f16.dtype == np.float16
    return np.int32(seed).tobytes() + embedding_f16.tobytes()


def decode_record(record: bytes, shape=None):
    """-> (seed:int, fp16 ndarray).  Mirrors DatasetWrapper._get_saved_embeddings."""
    seed = int(np.frombuffer(record[:SEED_BYTES], dtype=np.int32)[0])
    emb = np.frombuffer(record[SEED_BYTES:], dtype=np.float16).copy()
    return seed, (emb.reshape(shape) if shape is not None else emb)


class EmbeddingStoreWriter:
    """Append-only writer of one rank's package.  `write` is thread-safe; `close` publishes the files."""

    def __init__(self, path: str, rank: int = 0):
        self.path, self.rank = path, rank
        parent = os.path.dirname(os.path.abspath(path))
        os.makedirs(parent, exist_ok=True)
        self._tmp = tempfile.mkdtemp(prefix=f"es3_{os.path.basename(path)}_rank{rank}_", dir=parent)
        stem = os.path.join(self._tmp, f"rank{rank}")
        self._keys_f = open(stem + "-keys.txt", "w")
        self._vals_f = open(stem + "-values.bin", "wb")
        self._seen = set()
        self._lock = threading.Lock()
        self._closed = False

    def write(self, key: str, value: bytes) -> bool:
        with self._lock:
            if self._closed:
                raise RuntimeError("EmbeddingStoreWriter.write after close")
            if key in self._seen:     # first occurrence wins (manager.py:47-48)
                return False
            self._seen.add(key)
            self._keys_f.write(key + "\n")
            self._vals_f.write(value)
            return True

    def close(self):
        with self._lock:
            if self._closed:
                return
            self._closed = True
            self._keys_f.close()
            self._vals_f.close()
        os.makedirs(self.path, exist_ok=True)
        for entry in os.listdir(self._tmp):
            dst = os.path.join(self.path, entry)
            if os.path.isdir(dst):
                shutil.rmtree(dst)
            elif os.path.exists(dst):
                os.remove(dst)
            shutil.move(os.path.join(self._tmp, entry), dst)
        shutil.rmtree(self._tmp, ignore_errors=True)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class EmbeddingStoreReader:
    """Random access by key over every rank's package under `path` (own rank's package searched first)."""

    def __init__(self, path: str, item_size: int, rank: int = 0):
        if not os.path.isdir(path):
            raise FileNotFoundError(f"teacher embeddings not found at {path}")
        self.item_size = item_size
        names = [n[: -len("-values.bin")] for n in os.listdir(path) if n.endswith("-values.bin")]
        names.sort(key=lambda n: (int(n[4:]) - rank) % max(len(names), 1))
        self._stems = [os.path.join(path, n) for n in names]
        self._files = [None] * len(names)
        self._index = {}
        self._loaded = 0      # packages whose key list has been read (lazily, in search order)

    def _load_next(self):
        stem = self._stems[self._loaded]
        with open(stem + "-keys.txt") as f:
            for i, line in enumerate(f):
                # plain assignment, as the reference's _Reader does (manager.py:92-99): a key that the sampler's padding put into
                # several ranks' packages resolves to the LAST package loaded so far, and to the last line inside a package
                self._index[line.strip()] = (self._loaded, i)
        self._loaded += 1

    def read(self, key: str) -> bytes:
        while key not in self._index and self._loaded < len(self._stems):
            self._load_next()
        pkg, idx = self._index[key]          # KeyError when absent, like the reference
        if self._files[pkg] is None:
            self._files[pkg] = open(self._stems[pkg] + "-values.bin", "rb")
        f = self._files[pkg]
        f.seek(self.item_size * idx)
        rec = f.read(self.item_size)
        if len(rec) != self.item_size:
            raise IOError(f"short record for {key!r}: {len(rec)} of {self.item_size} bytes")
        return rec

    def read_embedding(self, key: str, shape=None):
        return decode_record(self.read(key), shape)

    def close(self):
        for f in self._files:
            if f is not None:
                f.close()
        self._files = [None] * len(self._files)


class _Slot:
    def __init__(self, numel, device):
        self.dev = torch.empty(numel, device=device, dtype=torch.float16)
        self.host = torch.empty(numel, dtype=torch.float16, pin_memory=True)
        self.done = torch.cuda.Event()
        self.free = threading.Event()
        self.free.set()


class EmbeddingDumper:
    """Double-buffered device->host->file pipeline for teacher outputs."""

    def __init__(self, writer: EmbeddingStoreWriter, device, max_batch_numel: int, slots: int = 2):
        self.writer = writer
        self.copy_stream = torch.cuda.Stream(device=device)
        self._slots = [_Slot(max_batch_numel, device) for _ in range(slots)]
        self._next = 0
        self._q: "queue.Queue" = queue.Queue()
        self._err = None
        self._thread = threading.Thread(target=self._drain, name="es3-embedding-writer", daemon=True)
        self._thread.start()
        self.d2h_bytes = 0

    def _drain(self):
        while True:
            item = self._q.get()
            if item is None:
                return
            slot, keys, seeds, per = item
            try:
                slot.done.synchronize()
                host = slot.host.numpy()
                for i, (k, s) in enumerate(zip(keys, seeds)):
                    self.writer.write(k, encode_record(s, host[i * per:(i + 1) * per]))
            except BaseException as e:  # surfaced by submit()/close()
                self._err = e
            finally:
                slot.free.set()

    def submit(self, outputs: torch.Tensor, keys, seeds):
        """outputs: [B, C, E, E] fp32 CUDA (teacher forward result on the current stream)."""
        if self._err is not None:
            raise self._err
        B = outputs.shape[0]
        per = outputs[0].numel()
        assert len(keys) == B and len(seeds) == B
        slot = self._slots[self._next]
        self._next = (self._next + 1) % len(self._slots)
        slot.free.wait()           # the host thread has finished writing this slot's previous contents
        slot.free.clear()
        n = B * per
        if n > slot.dev.numel():   # a batch larger than the one the slots were sized from: grow this slot (it is idle here)
            torch.cuda.current_stream().synchronize()
            grown = _Slot(n, slot.dev.device)
            grown.free.clear()
            self._slots[(self._next - 1) % len(self._slots)] = slot = grown
        ops.cast_f32_to_f16(outputs.contiguous(), out=slot.dev[:n])
        ready = torch.cuda.Event()
        ready.record()
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(ready)
            slot.host[:n].copy_(slot.dev[:n], non_blocking=True)
            slot.done.record(self.copy_stream)
        self.d2h_bytes += n * 2
        self._q.put((slot, list(keys), [int(s) for s in seeds], per))

    def close(self):
        self._q.put(None)
        self._thread.join()
        if self._err is not None:
            raise self._err


@torch.no_grad()
def save_embeddings_one_epoch(model, data_loader, path: str, rank: int = 0, max_batch: int | None = None, preprocess=None):
    """Native counterpart of save_embeddings_one_epoch (save_embedding_image_stage1.py:69-126).
    `data_loader` yields ((samples, _), (keys, seeds)) with `samples` a list/tensor of [3,S,S] fp32 images, exactly what the
    reference's write-mode DatasetWrapper + pseudo_collate produce.  With `preprocess` (a stage1.transforms.ImagePreprocessor)
    `samples` are decoded images of any size, resized, normalised and padded on the device.  Returns the number of records
    written."""
    model.eval()
    dev = next(model.parameters()).device
    dumper = None
    n = 0
    with EmbeddingStoreWriter(path, rank) as writer:
        try:
            for (samples, _), (keys, seeds) in data_loader:
                if preprocess is not None:
                    x, _ = preprocess(list(samples))
                else:
                    x = samples if torch.is_tensor(samples) else torch.stack(list(samples), dim=0)
                    x = x.to(dev, non_blocking=True)
                out = model(x)
                if dumper is None:
                    cap = (max_batch or getattr(data_loader, "batch_size", None) or x.shape[0]) * out[0].numel()
                    dumper = EmbeddingDumper(writer, dev, max(cap, out.numel()))
                dumper.submit(out, keys, np.asarray(seeds).astype(np.int32))
                n += x.shape[0]
        finally:
            if dumper is not None:
                dumper.close()
    return n
