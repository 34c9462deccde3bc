"""TensorBoard event files, written without TensorFlow: what ``tf.summary.FileWriter`` writes for the reference's merged
summary (sequential_base_model.py:268-274) - loss scalars and one histogram per variable - minus the graph def.

Format: ``events.out.tfevents.<unix time>.<hostname>`` holds TFRecord records (uint64 length, masked CRC-32C of the length,
the bytes, masked CRC-32C of the bytes); each record is an ``Event`` protobuf (tensorflow/core/util/event.proto), the first one
``file_version: "brain.Event:2"``.  Histograms arrive already binned and compacted by the device (Engine.histograms)."""
import os
import queue
import socket
import struct
import threading
import time

import numpy as np

from .checkpoint import _mask, _varint, crc32c

__all__ = ["histogram_proto", "summary_proto", "event_proto", "record", "EventFileWriter"]


def _key(field, wire):
    return _varint(field << 3 | wire)


def _bytes(field, data):
    return _key(field, 2) + _varint(len(data)) + data


def _double(field, v):
    return _key(field, 1) + struct.pack("<d", float(v))


def histogram_proto(h):
    """HistogramProto (summary.proto): min 1, max 2, num 3, sum 4, sum_squares 5, packed bucket_limit 6 and bucket 7 (doubles).
    h: a dict with those keys, the two repeated fields as arrays."""
    out = b"".join(_double(i + 1, h[k]) for i, k in enumerate(("min", "max", "num", "sum", "sum_squares")))
    for field, k in ((6, "bucket_limit"), (7, "bucket")):
        out += _bytes(field, np.ascontiguousarray(h[k], dtype="<f8").tobytes())
    return out


def summary_proto(scalars=(), histograms=()):
    """Summary: one Value (tag 1, simple_value 2 as float32, histo 5) per scalar (tag, value) and histogram (tag, dict)."""
    out = b""
    for tag, v in scalars:
        out += _bytes(1, _bytes(1, tag.encode()) + _key(2, 5) + struct.pack("<f", v))
    for tag, h in histograms:
        out += _bytes(1, _bytes(1, tag.encode()) + _bytes(5, histogram_proto(h)))
    return out


def event_proto(wall_time, step=0, summary=None, file_version=None):
    """Event: wall_time 1 (double), step 2 (int64), file_version 3, summary 5."""
    out = _double(1, wall_time)
    if step:
        out += _key(2, 0) + _varint(int(step))
    if file_version is not None:
        out += _bytes(3, file_version.encode())
    if summary is not None:
        out += _bytes(5, summary)
    return out


def record(data):
    """TFRecord framing of one serialized record."""
    n = struct.pack("<Q", len(data))
    return n + struct.pack("<I", _mask(crc32c(n))) + data + struct.pack("<I", _mask(crc32c(data)))


class EventFileWriter:
    """A new event file in ``logdir``.  ``add_summary`` hands the event to a background thread that frames and appends it; ``flush`` waits
    until everything handed over is written and flushed to the operating system; ``close`` flushes and ends the thread."""

    def __init__(self, logdir):
        os.makedirs(logdir, exist_ok=True)
        self.path = os.path.join(logdir, "events.out.tfevents.{:010d}.{}".format(int(time.time()), socket.gethostname()))
        self._f = open(self.path, "wb")
        self._q = queue.Queue()
        self._error = None
        self._thread = threading.Thread(target=self._run, name="pamrec-event-writer", daemon=True)
        self._thread.start()
        self._q.put(event_proto(time.time(), file_version="brain.Event:2"))

    def _run(self):
        while True:
            item = self._q.get()
            if item is None:
                return
            try:
                if isinstance(item, threading.Event):
                    if self._error is None:
                        self._f.flush()
                elif self._error is None:
                    self._f.write(record(item))
            except Exception as e:                           # reported by the next flush / close
                self._error = e
            finally:
                if isinstance(item, threading.Event):
                    item.set()

    def add_summary(self, summary, step, wall_time=None):
        """Queue one Event carrying a serialized Summary at global step ``step``."""
        if self._f is None:
            raise ValueError("add_summary on a closed EventFileWriter")
        self._q.put(event_proto(time.time() if wall_time is None else wall_time, step, summary=summary))

    def flush(self):
        if self._f is None:
            return
        done = threading.Event()
        self._q.put(done)
        done.wait()
        if self._error is not None:
            raise IOError("writing {} failed: {}".format(self.path, self._error))

    def close(self):
        if self._f is None:
            return
        try:
            self.flush()
        finally:
            self._q.put(None)
            self._thread.join()
            self._f.close()
            self._f = None
