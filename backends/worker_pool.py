"""Worker pool — one worker per GPU, shared FIFO, request micro-batching.

Public API identical to the reference's (`backends/worker_pool.py:147-181, 343-485`):
`WorkerPool(queue_max, worker_factory, mode_config, registry)`, `submit_job(job) -> Future`
(raises `queue.Full`), `switch_mode(name) -> Future` (raises `KeyError` for unknown modes),
`get_current_mode()`, `get_queue_size()`, `shutdown()`, module-level `get_worker_pool(...)` /
`reset_worker_pool()`, and the job classes `Job / GenerationJob / ModeSwitchJob / CustomJob /
JobType`.  `server/lcm_sr_server.py` and `server/model_routes.py` use it unchanged.

What is new (the reference runs ONE worker and ONE job at a time, `worker_pool.py:140,228,328`):
  * N workers, worker k pinned to GPU k, each driven by its own thread pulling from the one
    FIFO — independent images shard across GPUs with no collective (SURVEY.md §8e);
  * a worker that exposes `run_batch(jobs)` gets up to `B200_MAX_BATCH` queued generation jobs
    of the same geometry in one call (B200 needs batch >= 16 to approach its roofline);
  * a mode switch is a barrier: it waits for in-flight jobs, recreates every worker, and
    later jobs see the new mode (same FIFO semantics as the reference's single thread).

N comes from the ctor (`num_workers`), else `B200_NUM_WORKERS`, else the number of visible
CUDA devices (1 when that is not a positive integer, e.g. under mocked torch).

Dequeueing is done by ONE worker thread at a time (the collector role, `_collect_lock`): it pops the
next job, tops its batch up from the FIFO prefix — waiting up to `B200_BATCH_WINDOW_MS` (default 2 ms,
0 = never wait) for more compatible requests while the batch is short — registers it as in flight and
only then hands the role to the next idle thread.  Without that, N idle threads race for every arriving
request and batches degrade to 1 below saturation.  A mode switch is executed by the thread that pops it
while it still holds the role, so no later job can be popped before the switch is done (strict FIFO).
"""
from __future__ import annotations

import logging
import os
import queue
import threading
from abc import ABC, abstractmethod
from concurrent.futures import Future
from dataclasses import dataclass, field
from enum import Enum
from typing import Any, Callable, List, Optional

import torch

logger = logging.getLogger(__name__)


class JobType(Enum):
    GENERATION = "generation"
    MODE_SWITCH = "mode_switch"
    MODEL_LOAD = "model_load"
    MODEL_UNLOAD = "model_unload"
    CUSTOM = "custom"


@dataclass
class Job(ABC):
    """Base of everything that travels through the queue; subclass to add job kinds."""
    job_type: JobType = field(init=False)
    fut: Future = field(init=False, default=None)

    def __post_init__(self):
        if self.fut is None:
            self.fut = Future()

    @abstractmethod
    def execute(self, worker) -> Any:
        ...


@dataclass
class GenerationJob(Job):
    req: Any

    def __post_init__(self):
        super().__post_init__()
        self.job_type = JobType.GENERATION

    def execute(self, worker) -> Any:
        if worker is None:
            raise RuntimeError("No worker available for generation")
        return worker.run_job(self)


@dataclass
class ModeSwitchJob(Job):
    target_mode: str
    on_complete: Optional[Callable] = None

    def __post_init__(self):
        super().__post_init__()
        self.job_type = JobType.MODE_SWITCH

    def execute(self, worker) -> Any:
        if self.on_complete:
            self.on_complete(self.target_mode)
        return {"mode": self.target_mode, "status": "switched"}


@dataclass
class CustomJob(Job):
    handler: Callable
    args: tuple = ()
    kwargs: dict = None

    def __post_init__(self):
        super().__post_init__()
        self.job_type = JobType.CUSTOM
        if self.kwargs is None:
            self.kwargs = {}

    def execute(self, worker) -> Any:
        return self.handler(*self.args, **self.kwargs)


def _auto_num_workers() -> int:
    env = os.environ.get("B200_NUM_WORKERS", "").strip()
    if env:
        return max(1, int(env))
    try:
        n = torch.cuda.device_count()
    except Exception:
        return 1
    return n if isinstance(n, int) and n > 0 else 1


def _batch_key(job, same_guidance: bool = False):
    """Generation jobs that may share one batched pass: same size, step count and style (and,
    for workers that run classifier-free guidance on a doubled batch, the same guidance scale).
    Image-to-image requests (an `init_image`) also share their strength: ("img2img", strength) is appended;
    inpainting requests (a `mask_image`) append ("inpaint", strength) instead (default strength 1.0).  A request
    with a non-LCM `sampler` appends ("sampler", name); the LCM sampler (the default) appends nothing."""
    req = getattr(job, "req", None)
    try:
        if same_guidance:
            return _batch_key(job) + (float(req.guidance_scale),)
        sl = getattr(req, "style_lora", None)
        style = (getattr(sl, "style", None), int(getattr(sl, "level", 0) or 0)) if sl else (None, 0)
        if not style[0] or style[1] <= 0:
            style = (None, 0)
        key = (str(req.size).lower(), int(req.num_inference_steps), style)
        if getattr(req, "mask_image", None) is not None:
            st = getattr(req, "strength", None)
            key += (("inpaint", 1.0 if st is None else float(st)),)
        elif getattr(req, "init_image", None) is not None:
            st = getattr(req, "strength", None)
            key += (("img2img", 0.8 if st is None else float(st)),)
        sampler = getattr(req, "sampler", None)
        if sampler is not None and sampler != "lcm":
            key += (("sampler", str(sampler)),)
        return key
    except Exception:
        return None


class WorkerPool:
    def __init__(self, queue_max: int = 64, worker_factory=None, mode_config=None, registry=None,
                 num_workers: Optional[int] = None, max_batch: Optional[int] = None):
        self.queue_max = queue_max
        self.q: "queue.Queue[Job]" = queue.Queue(maxsize=queue_max)
        self._stop = threading.Event()
        self._workers: List[Any] = []
        self._worker_threads: List[threading.Thread] = []
        self._current_mode: Optional[str] = None
        self._lock = threading.Lock()
        # gate: generation jobs hold a share, a mode switch needs it exclusively
        self._gate = threading.Condition()
        self._active = 0
        self._switching = False
        self.num_workers = num_workers if num_workers else _auto_num_workers()
        self.max_batch = max_batch if max_batch else int(os.environ.get("B200_MAX_BATCH", "16"))
        self.batch_window = float(os.environ.get("B200_BATCH_WINDOW_MS", "2")) / 1e3
        self._collect_lock = threading.Lock()

        self._worker_factory = worker_factory or self._default_worker_factory
        if mode_config is None:
            from server.mode_config import get_mode_config
            mode_config = get_mode_config()
        if registry is None:
            from backends.model_registry import get_model_registry
            registry = get_model_registry()
        self._mode_config = mode_config
        self._registry = registry
        self._load_mode(self._mode_config.get_default_mode())

    # reference-compatible single-worker views
    @property
    def _worker(self):
        return self._workers[0] if self._workers else None

    @property
    def _worker_thread(self):
        return self._worker_threads[0] if self._worker_threads else None

    @staticmethod
    def _default_worker_factory(worker_id: int):
        from backends.worker_factory import create_cuda_worker
        return create_cuda_worker(worker_id)

    # ------------------------------------------------------------------ lifecycle
    def _create_workers(self) -> List[Any]:
        """One worker per GPU, built concurrently (each constructor loads and packs its own copy of the
        weights on its own device: 8 serial loads would make a mode switch 8x longer)."""
        if self.num_workers == 1:
            return [self._worker_factory(worker_id=0)]
        out: List[Any] = [None] * self.num_workers
        errs: List[BaseException] = []

        def make(k):
            try:
                out[k] = self._worker_factory(worker_id=k)
            except BaseException as e:                      # noqa: BLE001 - re-raised below
                errs.append(e)
        ts = [threading.Thread(target=make, args=(k,), name=f"WorkerInit-{k}") for k in range(self.num_workers)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        if errs:
            raise errs[0]
        return out

    def _load_mode(self, mode_name: str):
        mode = self._mode_config.get_mode(mode_name)
        old_env = (os.environ.get("MODEL_ROOT"), os.environ.get("MODEL"))
        # the workers read the model location from the environment (reference contract)
        os.environ["MODEL_ROOT"] = self._mode_config.config.model_root
        os.environ["MODEL"] = mode.model
        vram_before = self._registry.get_used_vram()
        try:
            # new workers first (180 GB of HBM hold both generations): a model that fails to load
            # leaves the pool serving the old mode instead of with no workers at all
            new_workers = self._create_workers()
        except BaseException:
            for key, val in zip(("MODEL_ROOT", "MODEL"), old_env):
                if val is None:
                    os.environ.pop(key, None)
                else:
                    os.environ[key] = val
            raise
        vram_used = self._registry.get_used_vram() - vram_before
        if self._workers:
            self._unload_current_worker()
        self._workers = new_workers
        self._registry.register_model(
            name=mode_name, model_path=mode.model_path, vram_bytes=vram_used, worker_id=0,
            loras=[lora.path for lora in mode.loras])
        self._current_mode = mode_name
        self._start_worker_threads()
        logger.info("[WorkerPool] mode '%s' loaded on %d worker(s)", mode_name, len(self._workers))

    def _unload_current_worker(self):
        if not self._workers:
            return
        if self._current_mode:
            self._registry.unregister_model(self._current_mode)
        for w in self._workers:
            # a worker that returns from run_batch(deferred=True) before its GPU work is done finishes it first
            drain = getattr(type(w), "drain", None)
            if callable(drain):
                try:
                    drain(w)
                except Exception as e:                       # noqa: BLE001 - unloading must go on
                    logger.warning("[WorkerPool] drain failed: %s", e)
        self._workers = []
        import gc
        gc.collect()
        torch.cuda.empty_cache()

    def _start_worker_threads(self):
        alive = [t for t in self._worker_threads if t.is_alive()]
        self._worker_threads = alive
        for k in range(len(alive), self.num_workers):
            t = threading.Thread(target=self._worker_loop, args=(k,), daemon=True,
                                 name="WorkerThread" if k == 0 else f"WorkerThread-{k}")
            self._worker_threads.append(t)
            t.start()

    # ------------------------------------------------------------------ worker threads
    def _take_batch(self, first: Job, worker) -> List[Job]:
        """Pull queued generation jobs compatible with `first` (FIFO prefix only); while the batch is
        short, wait up to `batch_window` for more to arrive.  Called by the collector thread only."""
        batch = [first]
        if not (worker is not None and type(first) is GenerationJob and _is_real_batcher(worker)):
            return batch
        same_gs = _same_guidance(worker)
        key = _batch_key(first, same_gs)
        if key is None or self.max_batch <= 1:
            return batch
        import time
        deadline = time.monotonic() + self.batch_window
        with self.q.mutex:                      # peek under the queue's own lock
            while len(batch) < self.max_batch:
                if self.q.queue:
                    nxt = self.q.queue[0]
                    if isinstance(nxt, GenerationJob) and type(nxt) is type(first) and _batch_key(nxt, same_gs) == key:
                        batch.append(self.q.queue.popleft())
                        self.q.not_full.notify()
                        continue
                    break                       # an incompatible job (or a mode switch) ends the prefix
                left = deadline - time.monotonic()
                if left <= 0 or self._stop.is_set():
                    break
                self.q.not_empty.wait(left)     # releases the mutex while waiting
        return batch

    def _run_generation(self, k: int, job: Job, batch: List[Job], worker):
        """`batch` is already registered as in flight (`_active`) by the collector."""
        try:
            if (worker is not None and type(job) is GenerationJob and _is_real_batcher(worker)
                    and getattr(type(worker), "supports_deferred", False) is True):
                # GPU pass here, PNG encoding on the encoder threads: this thread moves on to the
                # next batch while the images of this one are still being compressed
                thunks = worker.run_batch(batch, deferred=True)
                if callable(getattr(thunks[0], "wait", None)):
                    # the batch is only enqueued on the GPU: one waiter thread sleeps on it, this thread goes on
                    # to the next batch (whose host work then overlaps this one's kernels)
                    _waiters().submit(_resolve_batch, batch, thunks)
                else:
                    _resolve_batch(batch, thunks)
            elif len(batch) > 1:
                results = worker.run_batch(batch)
                for j, r in zip(batch, results):
                    if not j.fut.done():
                        j.fut.set_result(r)
            else:
                result = job.execute(worker)
                if not job.fut.done():
                    job.fut.set_result(result)
        except Exception as e:
            logger.error("[WorkerPool] Job failed: %s", e, exc_info=True)
            for j in batch:
                if not j.fut.done():
                    j.fut.set_exception(e)
        finally:
            for _ in batch:
                self.q.task_done()
            with self._gate:
                self._active -= 1
                self._gate.notify_all()

    def _run_mode_switch(self, job: ModeSwitchJob):
        """Runs on the collector thread (no other job can be popped meanwhile): waits for the batches
        in flight, then recreates every worker."""
        with self._gate:
            self._switching = True
            while self._active > 0:
                self._gate.wait()
        try:
            if self._current_mode == job.target_mode:
                result = {"mode": job.target_mode, "status": "already_loaded"}
            else:
                result = job.execute(self._worker)
                self._load_mode(job.target_mode)
            if not job.fut.done():
                job.fut.set_result(result)
        except Exception as e:
            logger.error("[WorkerPool] Mode switch failed: %s", e, exc_info=True)
            if not job.fut.done():
                job.fut.set_exception(e)
        finally:
            self.q.task_done()
            with self._gate:
                self._switching = False
                self._gate.notify_all()

    def _worker_loop(self, k: int = 0):
        while not self._stop.is_set():
            with self._collect_lock:                 # the collector role: one dequeuer at a time
                try:
                    job = self.q.get(timeout=0.25)
                except queue.Empty:
                    continue
                if isinstance(job, ModeSwitchJob):
                    self._run_mode_switch(job)
                    continue
                with self._gate:
                    self._active += 1
                worker = self._workers[k] if k < len(self._workers) else None
                batch = self._take_batch(job, worker)
            self._run_generation(k, job, batch, worker)

    # ------------------------------------------------------------------ public API
    def submit_job(self, job: Job) -> Future:
        try:
            self.q.put_nowait(job)
            return job.fut
        except queue.Full:
            raise queue.Full(f"Job queue full (max: {self.queue_max}). "
                             "Try again later or increase QUEUE_MAX.")

    def switch_mode(self, mode_name: str) -> Future:
        self._mode_config.get_mode(mode_name)          # raises KeyError for unknown modes
        return self.submit_job(ModeSwitchJob(target_mode=mode_name))

    def get_current_mode(self) -> Optional[str]:
        return self._current_mode

    def get_queue_size(self) -> int:
        return self.q.qsize()

    def shutdown(self):
        self.q.join()
        self._stop.set()
        for t in self._worker_threads:
            if t.is_alive():
                t.join(timeout=5.0)
        self._unload_current_worker()


_WAITERS = None
_WAITERS_LOCK = threading.Lock()


def _waiters():
    """Threads that sleep until a batch's GPU work is done (one per batch in flight; they hold no GIL while waiting)."""
    global _WAITERS
    with _WAITERS_LOCK:
        if _WAITERS is None:
            from concurrent.futures import ThreadPoolExecutor
            _WAITERS = ThreadPoolExecutor(max_workers=int(os.environ.get("B200_WAITER_THREADS", "32")),
                                          thread_name_prefix="batch-wait")
        return _WAITERS


def _resolve_batch(batch, thunks):
    """Waits for the batch (when its results are deferred past the GPU work), then hands one task per request to
    the encoder threads."""
    from backends.b200_worker import _encoders
    try:
        wait = getattr(thunks[0], "wait", None)
        if callable(wait):
            wait()
    except Exception as e:                                  # noqa: BLE001 - forwarded to the callers
        logger.error("[WorkerPool] Batch failed on the device: %s", e, exc_info=True)
        for j in batch:
            if not j.fut.done():
                j.fut.set_exception(e)
        return
    for j, th in zip(batch, thunks):
        _encoders().submit(_resolve, j, th)


def _resolve(job, thunk):
    """Encoder-thread side of a deferred result."""
    try:
        r = thunk()
        if not job.fut.done():
            job.fut.set_result(r)
    except Exception as e:                                  # noqa: BLE001 - forwarded to the caller
        logger.error("[WorkerPool] Job failed while encoding: %s", e, exc_info=True)
        if not job.fut.done():
            job.fut.set_exception(e)


def _same_guidance(worker) -> bool:
    """Does this worker need one guidance scale per batch (classifier-free guidance on a doubled batch)?
    Read through the class so that a Mock's auto-attributes do not count; a property is evaluated."""
    v = getattr(type(worker), "batch_same_guidance", False)
    if isinstance(v, property):
        v = v.fget(worker)
    return v is True


def _is_real_batcher(worker) -> bool:
    """`run_batch` must be a real method, not an auto-attribute of a Mock."""
    fn = getattr(type(worker), "run_batch", None)
    return callable(fn)


_worker_pool: Optional[WorkerPool] = None


def get_worker_pool(worker_factory=None, mode_config=None, registry=None) -> WorkerPool:
    """Process-wide pool; the first call wins (dependency injection honoured on that call)."""
    global _worker_pool
    if _worker_pool is None:
        _worker_pool = WorkerPool(queue_max=int(os.environ.get("QUEUE_MAX", "64")),
                                  worker_factory=worker_factory, mode_config=mode_config,
                                  registry=registry)
    return _worker_pool


def reset_worker_pool():
    global _worker_pool
    if _worker_pool is not None:
        try:
            _worker_pool.shutdown()
        except Exception:
            pass
    _worker_pool = None
