"""DataLoader. Parity: python/paddle/io/dataloader/dataloader_iter.py, reader.py:DataLoader.

Pipeline (B200 design): worker threads/processes fetch samples -> native GIL-free collation into a pinned ring
(csrc/runtime/loader.cpp) -> async H2D on a side stream, one batch ahead of compute.
"""
from __future__ import annotations

import itertools
import multiprocessing as mp
import queue
import threading

import numpy as np
import torch

from ..framework.place import _default_device
from ..tensor import Tensor
from .dataset import IterableDataset
from .sampler import BatchSampler

_worker_info = threading.local()


class WorkerInfo:
    def __init__(self, id, num_workers, seed, dataset):  # noqa: A002
        self.id, self.num_workers, self.seed, self.dataset = id, num_workers, seed, dataset


def get_worker_info():
    return getattr(_worker_info, "info", None)


def _to_torch(x):
    if isinstance(x, torch.Tensor):
        return x.as_subclass(torch.Tensor)
    if isinstance(x, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(x))
    if isinstance(x, (int, np.integer)):
        return torch.tensor(int(x), dtype=torch.int64)
    if isinstance(x, (float, np.floating)):
        return torch.tensor(float(x), dtype=torch.float32)
    return None


def default_collate_fn(batch, ring=None, slot=None):
    sample = batch[0]
    if isinstance(sample, (torch.Tensor, np.ndarray, int, float, np.integer, np.floating)):
        ts = [_to_torch(b) for b in batch]
        if ring is not None and ts[0].dim() > 0 and ts[0].device.type == "cpu":
            nbytes = ts[0].numel() * ts[0].element_size() * len(ts)
            off = slot["cursor"]
            if off + nbytes <= ring.slot_bytes():
                slot["cursor"] = (off + nbytes + 255) // 256 * 256
                return ring.collate(slot["index"], off, ts).as_subclass(Tensor)
        return torch.stack(ts, 0).as_subclass(Tensor)
    if isinstance(sample, (str, bytes)):
        return list(batch)
    if isinstance(sample, dict):
        return {k: default_collate_fn([b[k] for b in batch], ring, slot) for k in sample}
    if isinstance(sample, (list, tuple)):
        return [default_collate_fn(list(f), ring, slot) for f in zip(*batch)]
    raise TypeError(f"batch data can only contains: tensor, numpy.ndarray, dict, list, number, but got {type(sample)}")


def default_convert_fn(batch):
    if isinstance(batch, (torch.Tensor, np.ndarray)):
        return _to_torch(batch).as_subclass(Tensor)
    if isinstance(batch, dict):
        return {k: default_convert_fn(v) for k, v in batch.items()}
    if isinstance(batch, (list, tuple)):
        return [default_convert_fn(b) for b in batch]
    return batch


def _mp_worker(dataset, index_q, out_q, wid, nw, seed, init_fn):
    _worker_info.info = WorkerInfo(wid, nw, seed + wid, dataset)
    np.random.seed((seed + wid) % (2 ** 32))
    torch.manual_seed(seed + wid)
    if init_fn is not None:
        init_fn(wid)
    while True:
        job = index_q.get()
        if job is None:
            break
        bi, idxs = job
        try:
            out_q.put((bi, [dataset[i] for i in idxs], None))
        except Exception as e:  # noqa: BLE001
            out_q.put((bi, None, repr(e)))


class DataLoader:
    def __init__(self, dataset, feed_list=None, places=None, return_list=True, batch_sampler=None, batch_size=1, shuffle=False,
                 drop_last=False, collate_fn=None, num_workers=0, use_buffer_reader=True, prefetch_factor=2, use_shared_memory=True,
                 timeout=0, worker_init_fn=None, persistent_workers=False, pin_memory=None, device_prefetch=None):
        self.dataset, self.return_list = dataset, return_list
        # static-graph feeding: with return_list=False every batch is a {variable name: tensor} dict for Executor.run(feed=...)
        self._feed_names = [getattr(v, "name", None) or f"feed_{i}" for i, v in enumerate(feed_list)] if feed_list else None
        self.collate_fn, self.num_workers = collate_fn, int(num_workers)
        self.prefetch_factor, self.timeout, self.worker_init_fn = max(1, prefetch_factor), timeout, worker_init_fn
        self.use_buffer_reader = use_buffer_reader
        self._iterable = isinstance(dataset, IterableDataset)
        self.batch_size, self.drop_last = batch_size, drop_last
        if self._iterable:
            self.batch_sampler = None
        elif batch_sampler is not None:
            self.batch_sampler = batch_sampler
        elif batch_size is None:
            self.batch_sampler = None
        else:
            self.batch_sampler = BatchSampler(dataset, shuffle=shuffle, batch_size=batch_size, drop_last=drop_last)
        self._device = None
        on_gpu = _default_device().type == "cuda"     # the current device (paddle.set_device), not merely a visible GPU
        if device_prefetch is None:
            device_prefetch = on_gpu and use_buffer_reader
        if device_prefetch and torch.cuda.is_available():
            self._device = torch.device("cuda", torch.cuda.current_device())
        self._ring = None
        self._pin = pin_memory if pin_memory is not None else on_gpu

    def __len__(self):
        if self._iterable:
            raise RuntimeError("length of IterableDataset not supported")
        if self.batch_sampler is None:
            return len(self.dataset)
        return len(self.batch_sampler)

    # ---- batch production ---------------------------------------------------
    def _index_batches(self):
        if self.batch_sampler is None:
            for i in range(len(self.dataset)):
                yield [i]
        else:
            yield from self.batch_sampler

    def _sample_batches(self):
        """Yields lists of raw samples."""
        if self._iterable:
            it = iter(self.dataset)
            if self.batch_size is None:
                for s in it:
                    yield [s]
                return
            while True:
                b = list(itertools.islice(it, self.batch_size))
                if not b or (len(b) < self.batch_size and self.drop_last):
                    return
                yield b
        elif self.num_workers == 0:
            for idxs in self._index_batches():
                yield [self.dataset[i] for i in idxs]
        else:
            yield from self._mp_batches()

    def _mp_batches(self):
        ctx = mp.get_context("fork")
        nw = self.num_workers
        index_qs = [ctx.Queue() for _ in range(nw)]
        out_q = ctx.Queue()
        seed = int(torch.initial_seed() % (2 ** 31))
        procs = [ctx.Process(target=_mp_worker, args=(self.dataset, index_qs[w], out_q, w, nw, seed, self.worker_init_fn), daemon=True)
                 for w in range(nw)]
        for p in procs:
            p.start()
        try:
            batches = enumerate(self._index_batches())
            inflight, next_out, done, buf = 0, 0, False, {}
            for _ in range(nw * self.prefetch_factor):
                try:
                    bi, idxs = next(batches)
                    index_qs[bi % nw].put((bi, idxs))
                    inflight += 1
                except StopIteration:
                    done = True
                    break
            while inflight > 0:
                bi, samples, err = out_q.get(timeout=self.timeout or None)
                if err is not None:
                    raise RuntimeError(f"DataLoader worker failed: {err}")
                buf[bi] = samples
                inflight -= 1
                if not done:
                    try:
                        nbi, idxs = next(batches)
                        index_qs[nbi % nw].put((nbi, idxs))
                        inflight += 1
                    except StopIteration:
                        done = True
                while next_out in buf:
                    yield buf.pop(next_out)
                    next_out += 1
        finally:
            for q_ in index_qs:
                q_.put(None)
            for p in procs:
                p.join(timeout=1)
                if p.is_alive():
                    p.terminate()

    def _get_ring(self):
        if self._ring is None and self._pin:
            from .._build import load

            m = load()
            if m is not None:
                try:
                    self._ring = m.PinnedRing(self.prefetch_factor + 2, 256 << 20, 4)
                except Exception:  # noqa: BLE001
                    self._ring = False
            else:
                self._ring = False
        return self._ring or None

    def _collate(self, samples, slot_index):
        if self.batch_sampler is None and not self._iterable and self.batch_size is None:
            return default_convert_fn(samples[0])
        if self.collate_fn is not None:
            return self.collate_fn(samples)
        ring = self._get_ring()
        if ring is not None:
            ring.wait_slot(slot_index)
            return default_collate_fn(samples, ring, {"index": slot_index, "cursor": 0})
        return default_collate_fn(samples)

    def _to_device(self, batch, slot_index, stream):
        if self._device is None:
            return batch
        ring = self._get_ring()

        def mv(x):
            if isinstance(x, torch.Tensor):
                with torch.cuda.stream(stream):
                    dst = torch.empty(x.shape, dtype=x.dtype, device=self._device)
                    src = x.as_subclass(torch.Tensor)
                    if ring is not None and src.device.type == "cpu":
                        ring.h2d(slot_index, src, dst)
                    else:
                        dst.copy_(src, non_blocking=True)
                return dst.as_subclass(Tensor)
            if isinstance(x, dict):
                return {k: mv(v) for k, v in x.items()}
            if isinstance(x, (list, tuple)):
                return [mv(v) for v in x]
            return x

        return mv(batch)

    def __iter__(self):
        if not self.return_list and self._feed_names:
            for batch in self._iter_batches():
                items = list(batch) if isinstance(batch, (list, tuple)) else [batch]
                if len(items) != len(self._feed_names):
                    raise ValueError(f"DataLoader(feed_list=...): the dataset yields {len(items)} fields, feed_list names {len(self._feed_names)}")
                yield dict(zip(self._feed_names, items))
            return
        yield from self._iter_batches()

    def _iter_batches(self):
        nslots = self.prefetch_factor + 2
        if self._device is None or not self.use_buffer_reader:
            for i, samples in enumerate(self._sample_batches()):
                yield self._collate(samples, i % nslots)
            return
        from ..device import side_stream

        stream = side_stream(self._device)
        q = queue.Queue(maxsize=self.prefetch_factor)
        stop = object()

        def producer():
            try:
                for i, samples in enumerate(self._sample_batches()):
                    b = self._collate(samples, i % nslots)
                    b = self._to_device(b, i % nslots, stream)
                    ev = torch.cuda.Event()
                    ev.record(stream)
                    q.put((b, ev))
                q.put((stop, None))
            except Exception as e:  # noqa: BLE001
                q.put((e, None))

        t = threading.Thread(target=producer, daemon=True)
        t.start()
        while True:
            b, ev = q.get()
            if b is stop:
                break
            if isinstance(b, Exception):
                raise b
            torch.cuda.current_stream(self._device).wait_event(ev)
            yield b

    def __call__(self):
        return self.__iter__()
