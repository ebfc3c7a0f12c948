"""Multi-GPU front of the upscaler service: one object with the reference service's interface, N GPUs behind it.

Reference: the orchestrator (src/sharkshark/pipeline.py:39-50,61-138) owns ONE ``FsrcnnUpscalerService`` -- one process,
one GPU -- and talks to it through ``start() / push_job() / push_job_nowait() / get_result() / stop()`` and the
``on_queue`` callback (src/upscale/base_service.py:13-110), reading ``lr_shape`` and writing ``output_shape``.  This
class keeps exactly that surface, so the unchanged orchestrator can drive a whole box:

  * one worker process per GPU, each running the single-GPU service (``service.FsrcnnUpscalerService`` by default);
  * jobs (``UpscalerQueueEntry``: a small batch of uint8 frames) are dealt round-robin in arrival order; the frames
    travel as CUDA tensors through torch.multiprocessing queues (CUDA IPC handles, as in the reference) and the
    worker's ``upscale()`` moves them to its own device (a peer copy over NVLink);
  * results are re-assembled IN ORDER in the parent (reorder buffer keyed by the arrival sequence number) before
    ``on_queue`` / ``get_result`` sees them -- the reference's single process produced them in order for free;
  * the reference's drop policy is kept: ``push_job_nowait`` raises ``queue.Full`` when the chosen worker's queue is
    full, and the dropped sequence number is skipped by the reorder buffer instead of stalling it;
  * a worker that fails reports the exception; it is re-raised in the parent by the next call;
  * every other keyword goes to the workers' services unchanged: ``out_fmt=FMT_NV12`` makes them return packed NV12
    frames ``uint8 [N, H*3/2, W]`` for an encoder.  The reorder buffer moves whole entries and never looks at the
    frames' shape.

The convnets need no collective (frames are independent, weights replicated); the temporal BSVD path shards as
contiguous chunks with a 16-frame halo instead (``sharding.bsvd_chunks`` / ``sharding.StreamChunker``).
"""
import queue
import threading
import time
import traceback

import torch
import torch.multiprocessing as mp


def _default_factory(device, **kw):
    from . import service
    return service.FsrcnnUpscalerService(device=device, **kw)


def _worker_main(factory, device, kwargs, output_shape, job_q, result_q, cmd_q):
    try:
        if isinstance(device, int) and torch.cuda.is_available():
            torch.cuda.set_device(device)   # allocations and kernel launches of this process go to its own GPU
        svc = factory(device, **kwargs)
        if output_shape is not None:
            svc.output_shape = output_shape
        svc.proc_init()
        result_q.put(("ready", device, None))
        while True:
            try:
                if cmd_q.get_nowait() == "exit":
                    break
            except queue.Empty:
                pass
            try:
                seq, job = job_q.get(timeout=0.01)
            except queue.Empty:
                continue
            try:
                result_q.put(("ok", seq, svc.proc_job_recieved(job)))
            except Exception:
                result_q.put(("error", seq, traceback.format_exc()))
        svc.proc_cleanup()
    except Exception:
        result_q.put(("fatal", device, traceback.format_exc()))


class WorkerError(RuntimeError):
    pass


class MultiGpuUpscalerService:
    def __init__(self, devices, on_queue=None, worker_factory=None, queue_size=32, start_method="spawn", **service_kwargs):
        self.devices = list(devices)
        assert self.devices, "at least one device"
        self.on_queue = on_queue
        self.factory = worker_factory or _default_factory
        self.kwargs = dict(service_kwargs)
        self.queue_size = queue_size
        self.output_shape = None
        self._ctx = mp.get_context(start_method)
        self._lock = threading.Lock()
        self._seq = 0             # arrival order of the jobs
        self._next = 0            # next sequence number to hand out
        self._pending = {}        # seq -> entry, waiting for its predecessors
        self._dropped = set()     # sequence numbers whose job never reached a worker (queue.Full)
        self._results = queue.Queue(maxsize=queue_size)
        self._error = None
        self._procs, self._job_qs, self._cmd_qs = [], [], []
        self._result_q = None
        self._collector = None
        self._stop = threading.Event()

    # the orchestrator reads lr_shape right after construction (pipeline.py:45)
    @property
    def lr_shape(self):
        from . import service
        return service.FsrcnnUpscalerService.LR_SHAPES[self.kwargs.get("lr_level", 3)]

    # ------------------------------------------------------------------ life cycle (base_service.py:27-31,104-110)
    def start(self, ready_timeout=600):
        self._result_q = self._ctx.Queue(maxsize=4 * self.queue_size)
        for dev in self.devices:
            jq, cq = self._ctx.Queue(maxsize=self.queue_size), self._ctx.Queue(maxsize=64)
            p = self._ctx.Process(target=_worker_main, daemon=True,
                                  args=(self.factory, dev, self.kwargs, self.output_shape, jq, self._result_q, cq))
            p.start()
            self._procs.append(p)
            self._job_qs.append(jq)
            self._cmd_qs.append(cq)
        ready, t0 = 0, time.time()
        while ready < len(self.devices):
            try:
                kind, a, b = self._result_q.get(timeout=1.0)
            except queue.Empty:
                if time.time() - t0 > ready_timeout:
                    raise WorkerError("workers did not come up")
                continue
            if kind == "ready":
                ready += 1
            elif kind == "fatal":
                self.stop()
                raise WorkerError(f"worker on device {a} failed to start:\n{b}")
        self._collector = threading.Thread(target=self._collect, daemon=True)
        self._collector.start()

    def stop(self):
        self._stop.set()
        for cq in self._cmd_qs:
            try:
                cq.put_nowait("exit")
            except Exception:
                pass
        for p in self._procs:
            p.join(timeout=15)
            if p.is_alive():
                p.terminate()
        if self._collector is not None:
            self._collector.join(timeout=5)

    # ------------------------------------------------------------------ jobs in (base_service.py:88-94)
    def _check(self):
        if self._error is not None:
            err, self._error = self._error, None
            raise WorkerError(err)

    def _put(self, entry, block, timeout):
        self._check()
        with self._lock:
            seq = self._seq
            self._seq += 1
        w = seq % len(self.devices)
        try:
            if block:
                self._job_qs[w].put((seq, entry), timeout=timeout)
            else:
                self._job_qs[w].put_nowait((seq, entry))
        except queue.Full:
            with self._lock:
                self._dropped.add(seq)      # the reorder buffer must not wait for it
            self._flush()
            raise
        return seq

    def push_job(self, entry, timeout=10):
        return self._put(entry, True, timeout)

    def push_job_nowait(self, entry):
        return self._put(entry, False, None)

    # ------------------------------------------------------------------ results out, in arrival order
    def _emit(self, entry):
        if self.on_queue is not None:
            self.on_queue(entry)
        else:
            try:
                self._results.put_nowait(entry)
            except queue.Full:
                print("MultiGpuUpscalerService: result queue is full. Is the consumer not fast enough?")

    def _flush(self):
        out = []
        with self._lock:
            while True:
                if self._next in self._dropped:
                    self._dropped.discard(self._next)
                    self._next += 1
                elif self._next in self._pending:
                    out.append(self._pending.pop(self._next))
                    self._next += 1
                else:
                    break
        for e in out:
            if e is not None:
                self._emit(e)

    def _collect(self):
        while not self._stop.is_set():
            try:
                kind, seq, payload = self._result_q.get(timeout=0.05)
            except queue.Empty:
                continue
            if kind == "ok":
                with self._lock:
                    self._pending[seq] = payload
            elif kind == "error":
                self._error = payload
                with self._lock:
                    self._pending[seq] = None   # the failed job produces no frames; later jobs still flow
            elif kind == "fatal":
                self._error = payload
            self._flush()

    def get_result(self, timeout=10):
        self._check()
        return self._results.get(timeout=timeout)

    def wait_for_job_clear(self):
        while any(not q.empty() for q in self._job_qs):
            time.sleep(0.001)
