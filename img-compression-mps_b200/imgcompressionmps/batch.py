"""Concurrent processing of independent tensors on ONE GPU.

The reference's benchmark walks a list of tensors one after the other
(``evaluation/benchmark.py:73-76,117-118``).  On the device a single tensor cannot fill the
machine: the bond-sized eigenproblems of the sweep (``core/ndmps.py:74``) are latency-bound
cooperative kernels on a fraction of the SMs, and the host waits for each truncation decision.
Items are independent, so ``VolumePipeline`` keeps several of them in flight: ``workers`` host
threads, each with its own CUDA stream and its own native context (workspace arena, pinned
scratch -- ``_native.context()`` is per thread), pull items from a queue.  ctypes releases the
GIL for the duration of every native call, so the threads really overlap; on the GPU the
latency-bound kernels of one item run beside the bandwidth-bound kernels of another.

Nothing here changes results: every item goes through exactly the calls a single-threaded
caller would make.
"""
from __future__ import annotations

import os
import queue
import threading
from concurrent.futures import Future
from typing import Callable, Iterable, List, Optional, Sequence


def _walk_tensors(obj, seen=None):
    """Every CUDA torch tensor reachable from ``obj`` through tuples / lists / dicts and the MPS
    containers of this package (``NDMPS.mps.cores``)."""
    import torch
    if seen is None:
        seen = set()
    if id(obj) in seen:
        return
    seen.add(id(obj))
    if isinstance(obj, torch.Tensor):
        if obj.is_cuda:
            yield obj
        return
    if isinstance(obj, (list, tuple)):
        for x in obj:
            yield from _walk_tensors(x, seen)
        return
    if isinstance(obj, dict):
        for x in obj.values():
            yield from _walk_tensors(x, seen)
        return
    mps = getattr(obj, "mps", None)
    cores = getattr(mps if mps is not None else obj, "cores", None)
    if cores is not None and not isinstance(obj, (str, bytes)):
        yield from _walk_tensors(list(cores), seen)


class VolumePipeline:
    """``workers`` host threads x (CUDA stream + native context) on one device.

    Stream safety (torch's caching allocator recycles a block as soon as the stream that ALLOCATED it
    is past its last use, and knows nothing of other streams):

    * item ``i`` of every ``map`` call goes to worker ``i % workers``, so an object that is built in one
      call and transformed in a later one (the cutoff sweep of ``run_benchmark``) stays on ONE stream;
    * every device tensor reachable from an item is ``record_stream``-ed on the worker's stream (inputs
      were allocated on the caller's stream), every device tensor reachable from a result on the
      caller's stream (results were allocated on the worker's);
    * a worker synchronises its stream before its future resolves.
    """

    def __init__(self, workers: int = 3, device: Optional[int] = None, blocking_sync: Optional[bool] = None,
                 wait_mode: Optional[int] = None):
        import torch
        if workers < 1:
            raise ValueError("workers must be >= 1")
        if not torch.cuda.is_available():
            from . import _native
            raise _native.NativeError("VolumePipeline needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.workers = int(workers)
        # host threads that wait for the GPU spin by default; with more waiting threads (all ranks of this
        # node) than cores they would starve each other, so they sleep on blocking events instead
        if blocking_sync is None:
            ranks_here = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
            try:                                        # the cores this process may actually run on (cgroup / taskset aware)
                usable = len(os.sched_getaffinity(0))
            except (AttributeError, OSError):
                usable = os.cpu_count() or 1
            # a spinning waiter per worker of every rank of the node, plus the ranks' main threads, must each find a core
            blocking_sync = (self.workers + 1) * ranks_here > max(1, usable - 1)
        self.blocking_sync = bool(blocking_sync)
        # how a worker's native context waits inside the sweep (ndmps option blocking_sync): 0 spin, 3 watch a pinned word the
        # stream writes + yield (no driver calls while waiting).  Oversubscribed nodes watch and yield: the sweep's waits are
        # short, and a sleep in the driver costs a wake-up per wait
        env_mode = os.environ.get("NDMPS_WAIT_MODE")
        if wait_mode is None and env_mode is not None:
            wait_mode = int(env_mode)
        self.wait_mode = int(wait_mode) if wait_mode is not None else (3 if self.blocking_sync else 0)
        if self.wait_mode not in (0, 3):                # checked here: a worker thread that failed to start would hang the barrier
            raise ValueError(f"wait_mode must be 0 (spin) or 3 (pinned word), got {self.wait_mode}")
        self._ctx_lock = threading.Lock()
        self._contexts = []                             # the workers' native contexts (for launch counts / options)
        self._queues = [queue.SimpleQueue() for _ in range(self.workers)]
        self._threads = [threading.Thread(target=self._worker, args=(w,), name=f"ndmps-worker-{w}", daemon=True)
                         for w in range(self.workers)]
        self._ready = threading.Barrier(self.workers + 1)
        for t in self._threads:
            t.start()
        self._ready.wait()
        self._closed = False

    # -- worker side ---------------------------------------------------------------------------
    def _worker(self, index: int):
        import torch
        from . import _native
        torch.cuda.set_device(self.device)
        stream = torch.cuda.Stream(device=self.device)
        done = torch.cuda.Event(blocking=self.blocking_sync)
        ctx = _native.context()
        if self.wait_mode:
            ctx.set_option("blocking_sync", self.wait_mode)
        with self._ctx_lock:
            self._contexts.append(ctx)
        self._ready.wait()
        q = self._queues[index]
        while True:
            job = q.get()
            if job is None:
                return
            fn, item, ready_event, caller_stream, fut = job
            if not fut.set_running_or_notify_cancel():
                continue
            try:
                with torch.cuda.stream(stream):
                    if ready_event is not None:
                        stream.wait_event(ready_event)  # inputs produced on the submitting stream
                    for t in _walk_tensors(item):
                        t.record_stream(stream)
                    out = fn(item)
                    for t in _walk_tensors(out):
                        t.record_stream(caller_stream)
                    done.record(stream)
                    done.synchronize()                  # the result is complete when the future resolves
                fut.set_result(out)
            except BaseException as exc:                # noqa: BLE001 - handed to the caller
                try:
                    stream.synchronize()
                except Exception:
                    pass
                fut.set_exception(exc)

    # -- caller side ---------------------------------------------------------------------------
    def map(self, fn: Callable, items: Iterable) -> List:
        """``[fn(item) for item in items]`` with up to ``workers`` items in flight, in item order.
        ``fn`` runs with the worker's stream current, so everything it launches (native calls
        included) lands there; device inputs must already be materialised on the calling
        stream, which the workers wait for.  Item ``i`` always runs on worker ``i % workers``."""
        import torch
        if self._closed:
            raise RuntimeError("VolumePipeline is closed")
        caller_stream = torch.cuda.current_stream(self.device)
        ready = torch.cuda.Event()
        ready.record(caller_stream)
        futures = []
        for i, item in enumerate(items):
            fut = Future()
            self._queues[i % self.workers].put((fn, item, ready, caller_stream, fut))
            futures.append(fut)
        results, first_error = [], None
        for f in futures:                               # wait for ALL items, then raise the first failure
            try:
                results.append(f.result())
            except BaseException as exc:                # noqa: BLE001
                results.append(None)
                first_error = first_error or exc
        if first_error is not None:
            raise first_error
        return results

    def roundtrip(self, volumes: Sequence, max_bond: Optional[int] = None, cutoff: float = 1e-10, mode: str = "Std",
                  keep: bool = True) -> List:
        """``NDMPS.from_tensor(v, ...).to_tensor_device()`` for every device tensor in ``volumes``."""
        from .core.ndmps import NDMPS

        def one(v):
            obj = NDMPS.from_tensor(v, mode=mode, cutoff=cutoff, max_bond=max_bond)
            rec = obj.to_tensor_device()
            return (obj, rec) if keep else None

        return self.map(one, volumes)

    def roundtrip_host(self, sources: Sequence, outs: Sequence, max_bond: Optional[int] = None,
                       cutoff: float = 1e-10) -> List:
        """Host-buffer round trips (``_ops.roundtrip_host``): host -> device copy, encode, sweep,
        reconstruct, decode, device -> host copy, several items in flight so the copies of one
        overlap the sweep of another.  ``sources`` / ``outs``: numpy arrays (pinned for overlap)."""
        from . import _ops

        def one(pair):
            src, dst = pair
            return _ops.roundtrip_host(src, max_bond=max_bond, cutoff=cutoff, out=dst)

        return self.map(one, list(zip(sources, outs)))

    def launch_count(self) -> int:
        """Kernels launched so far by all workers of this pipeline."""
        with self._ctx_lock:
            return sum(c.launch_count() for c in self._contexts)

    def close(self):
        if self._closed:
            return
        self._closed = True
        for q in self._queues:
            q.put(None)
        for t in self._threads:
            t.join()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
