"""Many cameras over several ``DAVO`` handles, usually one per GPU of a box (include/davo_b200.h: davo_odometry_*).

Each camera is an odometry session on one handle.  ``push`` advances any set of cameras by one batched push per handle
(``DAVO.odometry_push_many_host`` / ``odometry_push_many``), ``rebalance`` evens out the handles with
``Odometry.move_to``, and ``save`` / ``load`` carry every camera across a restart of the process.  The pool holds no
numerics of its own: every result is that of the batched push on one handle, and a camera's results do not depend on
which handle it is on, on whether it moved, or on whether it was saved and loaded.
"""
from __future__ import annotations

import numpy as np

from .davo import DAVO

_INPUTS = ("img", "flow_fwd", "flow_bwd", "seg", "depth")


class OdometryPool(object):
    """Cameras spread over ``systems`` (set-up ``DAVO`` handles with weights loaded, of one version and frame size).

    ``pairs``, ``max_push`` and ``host`` are those of ``DAVO.odometry`` for every camera.  A host pool takes numpy
    arrays; a device pool (``host=False``) takes each camera's CUDA tensors on its handle's device (``device_of``)."""

    def __init__(self, systems, pairs='trajectory', max_push=1, host=True):
        systems = list(systems)
        if not systems:
            raise ValueError("OdometryPool: no handle")
        for i, s in enumerate(systems):
            if not isinstance(s, DAVO) or getattr(s, "_h", None) is None or not s._weights_loaded:
                raise ValueError("OdometryPool: handle %d is not set up with weights loaded" % i)
            if (s.version, s.img_height, s.img_width) != (systems[0].version, systems[0].img_height, systems[0].img_width):
                raise ValueError("OdometryPool: handle %d runs another version or frame size than handle 0" % i)
            if any(s is t for t in systems[:i]):
                raise ValueError("OdometryPool: handle %d is given twice" % i)
        self._systems, self._pairs, self._max_push, self._host = systems, pairs, int(max_push), bool(host)
        self._cams = {}                                  # camera id -> Odometry
        self._next = 0

    def counts(self):
        """Sessions per handle, in the order of ``systems``."""
        n = [0] * len(self._systems)
        for od in self._cams.values():
            n[self._index(od)] += 1
        return n

    def _index(self, od):
        return next(i for i, s in enumerate(self._systems) if s is od._system)

    def open(self):
        """A new camera on the handle with the fewest sessions (the first such handle); returns its id."""
        n = self.counts()
        s = self._systems[n.index(min(n))]
        od = s.odometry(self._pairs, self._max_push, self._host)
        cam = self._next
        self._next += 1
        self._cams[cam] = od
        return cam

    def close(self, cam):
        """Destroys camera ``cam``'s session."""
        self._cams.pop(cam).close()

    def close_all(self):
        for cam in list(self._cams):
            self.close(cam)

    def device_of(self, cam):
        """The CUDA device index that camera ``cam``'s frames go to in a device pool."""
        return self._cams[cam]._system.device

    def session(self, cam):
        """Camera ``cam``'s ``Odometry`` session."""
        return self._cams[cam]

    def push(self, ids, img, flow_fwd, flow_bwd, seg=None, depth=None, attention=False):
        """One push on each camera of ``ids``: the inputs are lists aligned with ``ids``, entry j holding what
        ``Odometry.push`` takes for camera ``ids[j]`` (None, or a list of None, where no camera has one).  One batched
        push per handle, all queued before any is waited for; returns the dicts ``Odometry.push`` returns, in ``ids``
        order (with each posed frame's ``'attention'`` and ``'att_weights'`` when ``attention`` is true)."""
        ids = list(ids)
        n = len(ids)
        lists = {}
        for name, x in zip(_INPUTS, (img, flow_fwd, flow_bwd, seg, depth)):
            lists[name] = [None] * n if x is None else list(x)
            if len(lists[name]) != n:
                raise ValueError("OdometryPool.push: %s has %d entries for %d cameras" % (name, len(lists[name]), n))
        if len(set(ids)) != n:
            raise ValueError("OdometryPool.push: a camera is given twice")
        for cam in ids:
            if cam not in self._cams:
                raise ValueError("OdometryPool.push: camera %r is not open" % (cam,))
        groups = {}                                      # handle index -> positions in ids
        for j, cam in enumerate(ids):
            groups.setdefault(self._index(self._cams[cam]), []).append(j)
        import torch
        out, pending = [None] * n, []
        for i, pos in sorted(groups.items()):
            s = self._systems[i]
            args = [[self._cams[ids[j]] for j in pos]] + [[lists[name][j] for j in pos] for name in _INPUTS]
            with torch.cuda.device(s.device):            # the library switches devices; torch's current one is restored
                if self._host:
                    pending.append((pos, s.odometry_push_many_host_async(*args, attention=attention)))
                else:
                    for j, r in zip(pos, s.odometry_push_many(*args, attention=attention)):
                        out[j] = r
        for pos, p in pending:
            for j, r in zip(pos, p.result()):
                out[j] = r
        return out

    def save(self):
        """``{camera id: blob}`` of every camera (``Odometry.save``'s bytes, as buffer-protocol objects): one
        ``DAVO.odometry_save_many`` per handle.  The cameras do not change."""
        out = {}
        for s in self._systems:
            cams = sorted(c for c, od in self._cams.items() if od._system is s)
            if cams:
                out.update(zip(cams, s.odometry_save_many([self._cams[c] for c in cams])))
        return out

    def load(self, blobs):
        """Restores the cameras of ``blobs`` (``{camera id: blob}`` from ``save``, of this pool or another, in this
        process or another) under the same ids: each goes to the handle with the fewest sessions, in id order, and
        each handle takes its cameras in one ``DAVO.odometry_load_many``.  Every blob is checked before any is loaded;
        ids that ``open`` gives afterwards are above the restored ones.  Returns the restored ids."""
        items = sorted(dict(blobs).items())
        n = self.counts()
        groups = {}                                      # handle index -> [(camera, blob)]
        for cam, blob in items:
            if cam in self._cams:
                raise ValueError("OdometryPool.load: camera %r is open" % (cam,))
            i = n.index(min(n))
            hdr = self._systems[i]._blob_header(blob, "odometry_load_many: camera %r" % (cam,))
            if (hdr["host"], hdr["pairs"], hdr["max_push"]) != (self._host, self._pairs, self._max_push):
                raise ValueError("OdometryPool.load: camera %r was saved as a %s session, pairs=%r, max_push=%d; this pool "
                                 "holds %s sessions, pairs=%r, max_push=%d" % (
                                     cam, "host" if hdr["host"] else "device", hdr["pairs"], hdr["max_push"],
                                     "host" if self._host else "device", self._pairs, self._max_push))
            n[i] += 1
            groups.setdefault(i, []).append((cam, blob))
        import torch
        loaded = []
        try:
            for i, group in sorted(groups.items()):
                s = self._systems[i]
                with torch.cuda.device(s.device):
                    loaded += zip([c for c, _ in group], s.odometry_load_many([b for _, b in group]))
        except Exception:
            for _, od in loaded:                         # all or nothing
                od.close()
            raise
        self._cams.update(loaded)
        if items:
            self._next = max(self._next, max(c for c, _ in items) + 1)
        return [c for c, _ in items]

    def rebalance(self):
        """Moves sessions from the fullest handle to the emptiest (``Odometry.move_to``, the most recently opened
        first) until the session counts differ by at most one.  Returns the number of moves."""
        moved = 0
        while True:
            n = self.counts()
            hi, lo = int(np.argmax(n)), int(np.argmin(n))
            if n[hi] - n[lo] <= 1:
                return moved
            cam = max(c for c, od in self._cams.items() if self._index(od) == hi)
            self._cams[cam].move_to(self._systems[lo])
            moved += 1
