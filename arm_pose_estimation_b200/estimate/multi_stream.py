"""Many sensor streams behind ONE batched estimator (SURVEY.md §8f.3).

The reference runs one ``Estimator`` thread per socket: ``ImuListener.listen_in_thread() -> sensor_q`` feeds
``Estimator.processing_loop`` (``estimate/estimator.py:145-178``), which takes one row per iteration, sheds the backlog
while more than five rows wait (``:159-161``), estimates, and puts the message on ``msg_q`` for
``PoseEstPublisherUDP.publish_in_thread`` (``stream/publisher/pose_est_udp.py:26-51``).  Here B such sensor queues feed one
``BatchedEstimator``: every tick takes at most one row per stream - with the same freshness policy, per stream - and
runs ONE batched step over the streams that had a row.  Streams advance independently: each has its own frame counter
(the kernels take it as ``stream_frames[b]``; a stream without a new row is skipped and its window / smoothing history
stays where it was), so every stream sees exactly the estimates a dedicated single-stream estimator would have produced
from the rows it kept (bit-for-bit: the Philox dropout keys are (stream id, the stream's own frame number, ...)).

The listeners and publishers stay the reference's own classes, one per stream::

    sensor_qs = [ImuListener(ip, port=p).listen_in_thread() for p in ports]          # stream/listener/imu.py:31-39
    ms = MultiStreamEstimator(engine)                                                # engine: BatchedEstimator, B = len(ports)
    msg_qs = ms.process_in_thread(sensor_qs)
    for q, p in zip(msg_qs, out_ports):
        PoseEstPublisherUDP(ip, p).publish_in_thread(q)                              # stream/publisher/pose_est_udp.py:26-31
"""
import logging
import queue
import threading
import time
from datetime import datetime

import numpy as np


class MultiStreamEstimator:
    def __init__(self, engine, add_mc_samples=True, max_backlog=5, idle_sleep_s=0.0005, no_data_after_s=2.0, tag="MULTI STREAM"):
        """``engine``: a ``BatchedEstimator`` built with ``frames_per_call=1`` and ``n_streams`` = number of sensor queues
        (anything with ``B``, ``ncols``, ``S`` and ``step(rows, stream_frames=...)`` works - the host logic is tested with a
        stand-in).  ``max_backlog`` is the reference's freshness bound (rows beyond it are shed, ``estimator.py:160``)."""
        self._engine = engine
        self._B = int(engine.B)
        self._add_mc_samples = bool(add_mc_samples)
        self._max_backlog = int(max_backlog)
        self._idle_sleep_s = float(idle_sleep_s)
        self._no_data_after_s = float(no_data_after_s)
        self._tag = tag
        self._active = False
        self._frames = np.zeros(self._B, dtype=np.int64)      # rows estimated so far, per stream = its next frame number
        self._dropped = np.zeros(self._B, dtype=np.int64)     # rows shed by the freshness policy, per stream
        self._rows = np.zeros((self._B, 1, int(engine.ncols)), dtype=np.float32)
        self._last_msg = [None] * self._B
        self._last_std = [None] * self._B
        self._thread = None

    # ---- the reference's estimator controls, per front-end (estimator.py:72-91) ---------------------------------------
    def is_active(self):
        return self._active

    def terminate(self):
        self._active = False

    def reset(self):
        """Forget every stream's history: the next row of each stream is its frame 0 again (estimator.py:88-91)."""
        self._frames[:] = 0
        self._dropped[:] = 0

    def reset_stream(self, b):
        """One stream reconnected: its next row starts a fresh window; the others are not disturbed."""
        self._frames[b] = 0

    def set_bonemap(self, b, bonemap):
        """Stream ``b`` gets its own skeleton (the reference's per-socket ``bonemap``, estimator.py:57-68): the engine's
        ``set_bonemap``, which applies from the next tick on.  A new user on a stream is ``reset_stream(b); set_bonemap(b, bm)``:
        from then on the stream sees exactly what a single-stream estimator built with ``bonemap=bm`` would produce."""
        self._engine.set_bonemap(b, bonemap)

    def get_last_msg(self, b):
        return self._last_msg[b]

    def get_last_std(self, b):
        return self._last_std[b]

    @property
    def frames(self):
        return self._frames.copy()

    @property
    def dropped(self):
        return self._dropped.copy()

    # ---- one tick -----------------------------------------------------------------------------------------------------
    def collect(self, sensor_qs):
        """At most one row per stream, newest-first under backlog (estimator.py:159-161).  Returns the bool mask of streams
        that had a row; their rows are in the staging array."""
        active = np.zeros(self._B, dtype=bool)
        for b, q in enumerate(sensor_qs):
            row = None
            try:
                row = q.get_nowait()
                while q.qsize() > self._max_backlog:
                    row = q.get_nowait()
                    self._dropped[b] += 1
            except queue.Empty:
                pass                                           # ran dry while shedding: keep the newest row taken so far
            if row is not None:
                self._rows[b, 0, :] = np.asarray(row, dtype=np.float32)
                active[b] = True
        return active

    def tick(self, active):
        """One batched step over the active streams (rows already staged by ``collect``).  Returns {stream: message}."""
        if not active.any():
            return {}
        stream_frames = np.where(active, self._frames, -1).astype(np.int32)
        out = self._engine.step_graph(self._rows, stream_frames=stream_frames)     # one CUDA-graph launch per tick
        msgs = {}
        for b in np.flatnonzero(active):
            if int(out.status[b, 0]) != 0:
                # the reference's estimator thread dies on this (LinAlgError from eigh, SURVEY.md §5); one bad stream must not
                # take the others down: log, skip the message, keep the stream's history
                logging.warning(f"[{self._tag}] stream {b}: degenerate 6D rotation, frame {int(self._frames[b])} dropped")
                self._frames[b] += 1
                continue
            msg = out.msg[b, 0].astype(np.float64)
            self._last_msg[b] = msg.copy()
            self._last_std[b] = out.std[b, 0].astype(np.float64)
            if self._add_mc_samples:                           # estimator.py:131-136
                msg = list(msg)
                if self._engine.S > 1:
                    msg += out.samples[b, 0].astype(np.float64).ravel().tolist()
            msgs[int(b)] = msg
            self._frames[b] += 1
        return msgs

    # ---- threads ------------------------------------------------------------------------------------------------------
    def process_in_thread(self, sensor_qs):
        """``sensor_qs``: one ``queue.Queue`` per stream (what ``ImuListener.listen_in_thread`` returns).  Returns one message
        queue per stream for the reference's publishers / recorders (estimator.py:139-143)."""
        if len(sensor_qs) != self._B:
            raise UserWarning(f"the engine serves {self._B} streams, got {len(sensor_qs)} sensor queues")
        msg_qs = [queue.Queue() for _ in range(self._B)]
        self._thread = threading.Thread(target=self.processing_loop, args=(sensor_qs, msg_qs))
        self._thread.start()
        return msg_qs

    def processing_loop(self, sensor_qs, msg_qs):
        logging.info(f"[{self._tag}] wearable streaming loop, {self._B} streams")
        self.reset()
        self._active = True
        start, last_data, n_est = datetime.now(), time.monotonic(), 0
        while self._active:
            active = self.collect(sensor_qs)
            if not active.any():
                if time.monotonic() - last_data >= self._no_data_after_s:
                    logging.info(f"[{self._tag}] no data")         # estimator.py:162-164
                    last_data = time.monotonic()
                time.sleep(self._idle_sleep_s)
                continue
            last_data = time.monotonic()
            for b, msg in self.tick(active).items():
                msg_qs[b].put(msg)
                n_est += 1
            now = datetime.now()
            if (now - start).seconds >= 5:                          # estimator.py:166-171
                logging.info(f"[{self._tag}] {n_est / 5} estimates/s over {self._B} streams")
                start, n_est = now, 0
