"""``DAVO`` -- the reference's model wrapper for the pose path, over libdavo_b200.so.

Keeps the calling surface of the reference class (reference ``davo.py:30-33``
constructor, ``:1533-1551`` ``setup_inference``, ``:1553-1569`` ``inference``)
and of its use in ``test_kitti_pose.py:126-135``:

    system = DAVO(version=FLAGS.version)
    system.setup_inference(H, W, "davo", seq_length, batch_size, input_batch,
                           input_flow=..., input_depth=..., input_seglabel=...)
    system.load_weights(ckpt)            # stands in for saver.restore(sess, ckpt)
    pred = system.inference(sess, mode='pose')     # {'pose': ndarray [B,2,6]}

The TensorFlow graph/session is replaced by one C call per ``inference``.
Inputs bound at ``setup_inference`` may be torch CUDA tensors (used in place),
numpy arrays (copied host->device inside the call) or callables returning the
next batch, which plays the role of the reference's ``tf.data`` iterator
outputs.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import struct

import numpy as np

from . import _capi
from . import tf_checkpoint
from . import version as V


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


# include/davo_b200.h: the header of a saved odometry session, format version 1
_BLOB_HEADER = struct.Struct("<8sIIQ20iQ6i2q4i6Q6QQ")
_BLOB_CONFIG = [n for n, _ in _capi.DavoConfigC._fields_ if n != "max_batch"]


def odometry_blob_header(blob):
    """The header of a saved odometry session (include/davo_b200.h: davo_odometry_save) of any buffer-protocol object,
    as a dict.  Raises ValueError for what is not a version-1 blob: too short, a bad magic, another version."""
    mv = memoryview(blob).cast("B")
    if mv.nbytes < _BLOB_HEADER.size:
        raise ValueError("a saved odometry session is at least %d bytes; this is %d (truncated?)" % (_BLOB_HEADER.size, mv.nbytes))
    f = _BLOB_HEADER.unpack_from(mv, 0)
    if f[0] != b"DAVOSESS":
        raise ValueError("not a saved odometry session (bad magic)")
    if f[1] != 1 or f[2] != _BLOB_HEADER.size:
        raise ValueError("saved odometry session of format version %d; this library reads version 1" % f[1])
    cfg, rest = f[4:24], f[24:]
    return {"bytes": mv.nbytes, "total_bytes": f[3], "config": dict(zip(_BLOB_CONFIG, cfg)), "weights_digest": rest[0],
            "weight_rounding": rest[1], "conv_impl": rest[2], "host": bool(rest[3]), "label_form": rest[4],
            "pairs": {v: k for k, v in _capi.PAIRS.items()}.get(rest[5], rest[5]), "max_push": rest[6],
            "pushed": rest[7], "posed": rest[8], "carried_frames": rest[9], "carried_fwd": bool(rest[10]),
            "carried_pose": bool(rest[11]), "section_off": list(rest[13:19]), "section_bytes": list(rest[19:25]),
            "checksum": rest[25]}


class DAVO(object):
    def __init__(self, version=None):
        self.version = version                       # reference davo.py:31-33
        self._h = None
        self._lib = None
        self._weights_loaded = False

    # ------------------------------------------------------------------ setup
    def setup_inference(self, img_height, img_width, mode, seq_length=3, batch_size=1,
                        input_img_uint8=None, input_pose=None, input_flow=None,
                        input_depth=None, input_seglabel=None, device=None, micro_batch=0, flow_f16=None):
        """Reference ``davo.py:1533-1551``; only ``mode == 'davo'`` builds anything there.

        ``flow_f16`` (extension; default False, or the environment's ``DAVO_B200_FLOW16=1``): define the optical
        flow input as rounded to IEEE binary16 on both entry points, which lets the host entry point move it
        over PCIe at half the bytes (include/davo_b200.h: davo_config.flow_f16).  Off, the flow is read as the
        float32 it is given in, like the reference's graph."""
        self.img_height = img_height
        self.img_width = img_width
        self.mode = mode
        self.batch_size = batch_size
        if self.mode != 'davo':
            return
        assert self.version is not None              # reference davo.py:959
        if seq_length != 3:
            raise NotImplementedError("davo_b200: only seq_length=3 (two source frames) is built")
        self.seq_length = seq_length
        self.num_source = seq_length - 1
        self.config = V.parse_version(self.version)  # raises NameError like the reference
        self._inputs = (input_img_uint8, input_flow, input_depth, input_seglabel)
        self._lib = _capi.load()
        if device is None:
            for t in self._inputs:
                if _is_torch(t) and t.is_cuda:
                    device = t.device.index
                    break
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = int(device)
        cfg = _capi.DavoConfigC(
            H=img_height, W=img_width, max_batch=batch_size, posenn=self.config.posenn,
            cnv6_out=self.config.cnv6_out, in_mode=self.config.in_mode,
            att_src=self.config.att_src, att_tgt_ones=self.config.att_tgt_ones,
            mask_mode=self.config.mask_mode, se_act=self.config.se_act,
            flow_abs=self.config.flow_abs, flow_norm=self.config.flow_norm,
            posenn_se=self.config.posenn_se, micro_batch=micro_batch, depth_norm=self.config.depth_norm,
            se_pool=self.config.se_pool, se_hidden=self.config.se_hidden, pixel_map=self.config.pixel_map,
            depth_split=self.config.depth_split, batch_norm=self.config.batch_norm,
            flow_f16=int(os.environ.get("DAVO_B200_FLOW16", "0") == "1") if flow_f16 is None else int(bool(flow_f16)))
        self.flow_f16 = bool(cfg.flow_f16)
        self._cfg = cfg
        h = C.c_void_p()
        rc = self._lib.davo_create(C.byref(cfg), self.device, C.byref(h))
        if rc != 0:
            raise RuntimeError("davo_create failed (%d): %s" % (rc, _capi.last_error(self._lib, None)))
        self._h = h
        self._pose_dev = None
        self._graph, self._graph_key, self._graph_hits = None, None, 0
        self._graph_ok = os.environ.get("DAVO_B200_GRAPH", "1") != "0"

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, _capi.last_error(self._lib, self._h)))

    # ---------------------------------------------------------------- weights
    def load_weights(self, weights):
        """``{tf variable name: ndarray}``, a ``.npz`` of that, or the prefix of a TensorFlow checkpoint
        (``model-<step>``: ``.index`` + ``.data-*``, read by ``tf_checkpoint.py``); stands in for
        ``tf.train.Saver(trainable_variables).restore`` (reference test_kitti_pose.py:129-131)."""
        if self._h is None:
            raise RuntimeError("DAVO.load_weights: call setup_inference(mode='davo') first")
        if isinstance(weights, (str, os.PathLike)):
            path = os.fspath(weights)
            if tf_checkpoint.is_checkpoint_prefix(path):      # a TF checkpoint prefix, as given to saver.restore
                weights = tf_checkpoint.read_checkpoint(path, tf_checkpoint.pose_variables)
            else:
                with np.load(path) as z:
                    weights = {k: z[k] for k in z.files}
        for name, arr in weights.items():
            a = np.ascontiguousarray(np.asarray(arr), dtype=np.float32)
            shape = (C.c_int64 * a.ndim)(*a.shape)
            self._check(self._lib.davo_set_weight(self._h, name.encode(), a.ctypes.data_as(C.c_void_p),
                                                  shape, a.ndim), "davo_set_weight(%s)" % name)
        self._check(self._lib.davo_finalize_weights(self._h), "davo_finalize_weights")
        self._weights_loaded = True

    restore = load_weights

    # -------------------------------------------------------------- inference
    def _resolve(self, x):
        return x() if callable(x) and not _is_torch(x) and not isinstance(x, np.ndarray) else x

    def inference(self, sess=None, mode='pose', inputs=None, as_torch=False, pairs='all'):
        """Reference ``davo.py:1553-1569``: one run of the pose graph -> ``{'pose': [B,2,6]}``.

        ``sess`` is accepted for signature compatibility and ignored.  ``inputs``
        may override the bound tensors as ``(img_u8, flow, seg)`` or a dict with
        keys ``img``, ``flow``, ``seg``.  ``pairs``: ``'all'`` (the graph's output),
        ``'trajectory'`` (only ``pose[:,1]``, what reference test_kitti_pose.py:143-145
        composes) or ``'trajectory_first'`` (plus ``pose[0,0]``, for the batch that opens a
        sequence); rows that are not computed are zero.
        """
        if pairs not in _capi.PAIRS:
            raise ValueError("DAVO.inference: pairs must be one of %s" % sorted(_capi.PAIRS))
        sel = _capi.PAIRS[pairs]
        if mode not in ('pose', 'feature'):
            raise NotImplementedError("davo_b200: inference mode %r is not built ('pose', 'feature')" % (mode,))
        if mode == 'feature' and sel != 0:
            raise ValueError("DAVO.inference: mode='feature' computes every pair (pairs='all')")
        if not self._weights_loaded:
            raise RuntimeError("DAVO.inference: weights not loaded")
        depth = None
        if inputs is None:
            img, flow, depth, seg = (self._resolve(t) for t in self._inputs)
        elif isinstance(inputs, dict):
            img, flow, seg, depth = inputs.get("img"), inputs.get("flow"), inputs.get("seg"), inputs.get("depth")
        elif len(inputs) == 4:
            img, flow, seg, depth = inputs
        else:
            img, flow, seg = inputs
        if self.config.att_src != V.ATT_SE_DEPTH_SEG and not self.config.depth_split:
            depth = None                                  # only the depth sources read it
        elif depth is None:
            raise ValueError("DAVO.inference: version %r reads input_depth [B,3,H,W,1]" % (self.version,))
        B = int(img.shape[0])
        H, W = self.img_height, self.img_width
        if (isinstance(img, np.ndarray) and mode == 'pose' and flow is not None and seg is not None
                and getattr(flow, "dtype", None) == np.float16 and getattr(seg, "dtype", None) == np.uint8):
            return self._run_host_compact(B, img, flow, seg, sel, depth)       # the caller holds the compact forms
        want = {"img": (B, H, 3 * W, 3), "flow": (B, 4, H, W, 2), "seg": (B, 3, H, W, 1), "depth": (B, 3, H, W, 1)}
        for name, t in (("img", img), ("flow", flow), ("seg", seg), ("depth", depth)):
            if t is not None and tuple(t.shape) != want[name]:
                raise ValueError("DAVO.inference: %s has shape %s, expected %s" % (name, tuple(t.shape), want[name]))
        if mode == 'feature':
            return self._run_features(B, img, flow, seg, depth, as_torch)
        if _is_torch(img):
            return self._run_device(B, img, flow, seg, as_torch, sel, depth)
        if self.config.batch_norm:
            # batch statistics need the whole batch in one pass: no chunked streaming; upload and take the device path
            import torch
            dev = "cuda:%d" % self.device
            up = lambda t, dt: None if t is None else torch.as_tensor(np.ascontiguousarray(t)).to(device=dev, dtype=dt)
            return self._run_device(B, up(img, torch.uint8), up(flow, torch.float32), up(seg, torch.float32), as_torch, sel,
                                    up(depth, torch.float32))
        return self._run_host(B, img, flow, seg, sel, depth)

    def _run_device(self, B, img, flow, seg, as_torch, sel=0, depth=None):
        import torch
        for name, t, dt in (("img", img, torch.uint8), ("flow", flow, torch.float32), ("seg", seg, torch.float32),
                            ("depth", depth, torch.float32)):
            if t is None:
                continue
            if not (t.is_cuda and t.device.index == self.device and t.dtype == dt and t.is_contiguous()):
                raise ValueError("DAVO.inference: %s must be a contiguous %s tensor on cuda:%d" % (name, dt, self.device))
        if self._pose_dev is None or self._pose_dev.shape[0] < B:
            self._pose_dev = torch.empty((max(B, self.batch_size), 2, 6), dtype=torch.float32,
                                         device="cuda:%d" % self.device)
        out = self._pose_dev[:B]
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None

        def launch():
            stream = torch.cuda.current_stream(self.device).cuda_stream
            self._check(self._lib.davo_forward_pairs(self._h, B, sel, ptr(img), ptr(flow), ptr(seg), ptr(depth),
                                                     C.c_void_p(out.data_ptr()), C.c_void_p(stream)), "davo_forward")

        # The same buffers called again and again (the bound-inputs form of the reference's
        # sess.run loop): davo_forward only enqueues work, so the third identical call is captured
        # into a CUDA graph and later ones replay it (launch gaps: -13 % latency at B=1, -1.4 % at
        # B=128).  DAVO_B200_GRAPH=0 switches this off; any capture failure does too.  Side effects to know
        # about: torch's capture synchronises the device once (at the third identical call) and frees its
        # cached blocks; nothing else in the process is touched.
        key = (B, sel, out.data_ptr()) + tuple(t.data_ptr() if t is not None else 0 for t in (img, flow, seg, depth))
        if torch.cuda.is_current_stream_capturing():     # the caller is building a graph of their own
            launch()
            return {'pose': out}
        if self._graph_ok and key == self._graph_key:
            self._graph_hits += 1
        else:
            self._graph_key, self._graph_hits, self._graph = key, 1, None
        if self._graph is not None:
            self._graph.replay()
        elif self._graph_ok and self._graph_hits == 3:
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):            # ends (and discards) the capture itself if launch() raises
                    launch()
                g.replay()
                self._graph = g
            except Exception:
                self._graph_ok, self._graph = False, None
                torch.cuda.synchronize(self.device)
                if torch.cuda.is_current_stream_capturing():
                    raise                            # the stream is still in an invalidated capture: do not launch into it
                launch()
        else:
            launch()
        if as_torch:
            # ``out`` is the handle's reusable output buffer (a fixed address is what lets the call be replayed as a
            # graph): the caller gets a tensor of its own, which the next inference() does not overwrite
            return {'pose': out.clone()}
        return {'pose': out.cpu().numpy()}

    def _run_features(self, B, img, flow, seg, depth, as_torch):
        """mode='feature' (reference davo.py:1553-1564): poses plus the visualisation tensors, as the
        same nested dict ``sess.run`` returns.  Lists are ordered [tgt, src0, src1] (davo.py:967-971,
        1467-1474); 'flows' holds the two source flows (davo.py:989).  One C call, all on the GPU."""
        import torch
        if flow is None or seg is None:
            raise ValueError("DAVO.inference: mode='feature' reads input_flow and input_seglabel")
        img, flow, seg, depth = self._upload(img, torch.uint8), self._upload(flow), self._upload(seg), self._upload(depth)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        return self._features(B, as_torch, "davo_forward_features", lambda pose, table, stream: self._lib.davo_forward_features(
            self._h, B, ptr(img), ptr(flow), ptr(seg), ptr(depth), ptr(pose), table, stream))

    def _upload(self, t, dt=None):
        """A numpy array or tensor as a contiguous tensor of dtype ``dt`` (float32 by default) on this handle's GPU."""
        import torch
        if t is None:
            return None
        return (t if _is_torch(t) else torch.as_tensor(np.ascontiguousarray(t))).to(
            device="cuda:%d" % self.device, dtype=torch.float32 if dt is None else dt).contiguous()

    def _features(self, B, as_torch, what, call):
        """The output tensors of mode='feature' for B samples, ``call(pose, table, stream)`` on them, and the dict."""
        import torch
        dev = "cuda:%d" % self.device
        H, W, c6 = self.img_height, self.img_width, self.config.cnv6_out
        if self.config.posenn_se == V.PSE_REPLACE:
            c6 = 256                                     # "cnv6" is se_block(cnv5) there (reference posenn.py:234-236)
        f32 = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
        u8 = lambda *shape: torch.empty(shape, dtype=torch.uint8, device=dev)
        pose = f32(B, 2, 6)
        image, att, masked = f32(3, B, H, W, 3), f32(3, B, H, W, 1), f32(3, B, H, W, 3)
        seg19, segc, flowc = f32(3, B, H, W, 19), u8(3, B, H, W, 3), u8(2, B, H, W, 3)
        rot, trans = f32(B, H, W, c6), f32(B, H, W, c6)
        table = _capi.DavoFeaturesC(*(C.c_void_p(t.data_ptr()) for t in (image, att, masked, seg19, segc, flowc, rot, trans)))
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(call(pose, C.byref(table), C.c_void_p(stream)), what)
        conv = (lambda t: t) if as_torch else (lambda t: t.cpu().numpy())
        squeeze = (lambda t: t.squeeze()) if as_torch else np.squeeze        # tf.squeeze drops every unit axis (davo.py:1115)
        return {
            'pose': conv(pose),
            'masks': {'image': [conv(masked[f]) for f in range(3)], 'attention': [conv(att[f]) for f in range(3)]},
            'features': {'rot': conv(rot), 'trans': conv(trans)},
            'images': [conv(image[f]) for f in range(3)],
            'flows': [conv(flowc[k]) for k in range(2)],
            'segs': [conv(segc[f]) for f in range(3)],
            'seg_19': [squeeze(conv(seg19[f])) for f in range(3)],
        }

    def _run_host(self, B, img, flow, seg, sel=0, depth=None):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        flow = None if flow is None else np.ascontiguousarray(flow, dtype=np.float32)
        seg = None if seg is None else np.ascontiguousarray(seg, dtype=np.float32)
        depth = None if depth is None else np.ascontiguousarray(depth, dtype=np.float32)
        out = np.empty((B, 2, 6), np.float32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        self._check(self._lib.davo_forward_host_pairs(self._h, B, sel, ptr(img), ptr(flow), ptr(seg), ptr(depth),
                                                      ptr(out), None), "davo_forward_host")
        return {'pose': out}

    def _run_host_compact(self, B, img, flow16, seg8, sel=0, depth=None):
        """Extension (include/davo_b200.h: davo_forward_host_compact): ``flow16`` float16 [B,2,H,W,2] = the two flow
        planes the graph reads, ``seg8`` uint8 [B,3,H,W(,1)] = the labels as bytes (255 = no class).  No CPU pass."""
        H, W = self.img_height, self.img_width
        if tuple(img.shape) != (B, H, 3 * W, 3) or tuple(flow16.shape) != (B, 2, H, W, 2) or seg8.size != B * 3 * H * W:
            raise ValueError("DAVO.inference (compact inputs): img [B,H,3W,3] uint8, flow [B,2,H,W,2] float16, seg [B,3,H,W] uint8")
        img, flow16, seg8 = np.ascontiguousarray(img), np.ascontiguousarray(flow16), np.ascontiguousarray(seg8)
        depth = None if depth is None else np.ascontiguousarray(depth, dtype=np.float32)
        out = np.empty((B, 2, 6), np.float32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        self._check(self._lib.davo_forward_host_compact(self._h, B, sel, ptr(img), ptr(flow16), ptr(seg8), ptr(depth),
                                                        ptr(out), None), "davo_forward_host_compact")
        return {'pose': out}

    # ------------------------------------------------------------ asynchronous host calls
    class _Pending(object):
        """A queued host-input inference; ``result()`` waits for it and returns ``{'pose': ndarray [B,2,6]}``."""

        def __init__(self, system, ticket, out, keep):
            self._system, self._ticket, self._out, self._keep = system, ticket, out, keep

        def result(self):
            if self._ticket is not None:
                s = self._system
                s._check(s._lib.davo_host_wait(s._h, self._ticket), "davo_host_wait")
                self._ticket, self._keep = None, None
                self._out = np.array(self._out)      # the caller's own copy: the pinned ring slot is reused 8 calls later
            return {'pose': self._out}

    def inference_async(self, inputs, pairs='all'):
        """``inference(sess, 'pose', inputs=<host arrays>)`` without waiting: the copies and launches are queued and the
        call returns, so the NEXT call's host->device copies run under this one's compute (what ``tf.data``'s prefetch
        gives the reference's ``sess.run`` loop).  ``inputs`` as in ``inference`` (float32 arrays, or the compact
        ``float16`` / ``uint8`` forms); they must not be modified before ``.result()``.  Returns a handle whose
        ``.result()`` gives the same dict as ``inference``.  Up to 8 calls may be in flight."""
        import torch
        if self.config.batch_norm:
            raise NotImplementedError("DAVO.inference_async: -batch_norm takes the device path (one pass per batch)")
        sel = _capi.PAIRS[pairs]
        depth = None
        if len(inputs) == 4:
            img, flow, seg, depth = inputs
        else:
            img, flow, seg = inputs
        if self.config.att_src != V.ATT_SE_DEPTH_SEG and not self.config.depth_split:
            depth = None
        B = int(img.shape[0])
        ring = getattr(self, "_async_out", None)
        if ring is None or ring[0].shape[0] < B:
            ring = self._async_out = [torch.empty((max(B, self.batch_size), 2, 6), dtype=torch.float32).pin_memory() for _ in range(8)]
            self._async_n = 0
        out = ring[self._async_n % 8][:B].numpy()
        self._async_n += 1
        compact = getattr(flow, "dtype", None) == np.float16 and getattr(seg, "dtype", None) == np.uint8
        img = np.ascontiguousarray(img, dtype=np.uint8)
        if compact:
            flow, seg = np.ascontiguousarray(flow), np.ascontiguousarray(seg)
        else:
            flow = None if flow is None else np.ascontiguousarray(flow, dtype=np.float32)
            seg = None if seg is None else np.ascontiguousarray(seg, dtype=np.float32)
        depth = None if depth is None else np.ascontiguousarray(depth, dtype=np.float32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        ticket = C.c_longlong(0)
        fn = self._lib.davo_forward_host_compact_async if compact else self._lib.davo_forward_host_pairs_async
        self._check(fn(self._h, B, sel, ptr(img), ptr(flow), ptr(seg), ptr(depth), ptr(out), None, C.byref(ticket)),
                    "davo_forward_host_async")
        return DAVO._Pending(self, ticket.value, out, (img, flow, seg, depth))

    # ------------------------------------------------------------ frame-sequence inputs
    def _sequence_args(self, img, flow_fwd, flow_bwd, seg, depth, pairs, who):
        if pairs not in _capi.PAIRS:
            raise ValueError("DAVO.%s: pairs must be one of %s" % (who, sorted(_capi.PAIRS)))
        if not self._weights_loaded:
            raise RuntimeError("DAVO.%s: weights not loaded" % who)
        if self.config.att_src != V.ATT_SE_DEPTH_SEG and not self.config.depth_split:
            depth = None                                  # only the depth sources read it
        elif depth is None:
            raise ValueError("DAVO.%s: version %r reads depth [N,H,W,1]" % (who, self.version))
        N, H, W = int(img.shape[0]), self.img_height, self.img_width
        want = {"img": (N, H, W, 3), "flow_fwd": (N - 1, H, W, 2), "flow_bwd": (N - 1, H, W, 2), "seg": (N, H, W, 1),
                "depth": (N, H, W, 1)}
        for name, t in (("img", img), ("flow_fwd", flow_fwd), ("flow_bwd", flow_bwd), ("seg", seg), ("depth", depth)):
            if t is not None and tuple(t.shape) != want[name]:
                raise ValueError("DAVO.%s: %s has shape %s, expected %s" % (who, name, tuple(t.shape), want[name]))
        return N, _capi.PAIRS[pairs], depth

    def inference_sequence(self, img, flow_fwd, flow_bwd, seg, depth=None, pairs='all', as_torch=False, mode='pose'):
        """Poses of a frame sequence -> ``{'pose': [N-2,2,6]}`` (include/davo_b200.h: davo_forward_sequence).

        ``img`` uint8 [N,H,W,3]; ``flow_fwd`` / ``flow_bwd`` float32 [N-1,H,W,2], entry i the flow from frame i to i+1 /
        from i+1 to i; ``seg`` float32 [N,H,W,1]; ``depth`` float32 [N,H,W,1] (depth sources only).  Sample s is frames
        (s, s+1, s+2); the poses equal ``inference`` on ``sequence_to_triplets`` of the same frames, bit for bit.
        ``flow_fwd`` may be None under ``pairs='trajectory'`` for the shared nets.  numpy arrays take the host path
        (each frame crosses PCIe once), CUDA tensors the device path; ``-batch_norm`` uploads and takes the device
        path.  A long sequence continues with a call that starts two frames before the previous one ended.

        ``mode='feature'`` (include/davo_b200.h: davo_forward_sequence_features) returns the nested dict of
        ``inference(mode='feature')`` for the N-2 samples, the same bits as that call on ``sequence_to_triplets`` of the
        frames; it computes every pair (``pairs='all'``), reads both flows and the labels, and takes one pass (2(N-2),
        or N-2 for the non-shared nets, <= micro_batch).  numpy inputs are uploaded."""
        if mode not in ('pose', 'feature'):
            raise NotImplementedError("davo_b200: inference_sequence mode %r is not built ('pose', 'feature')" % (mode,))
        if mode == 'feature' and pairs != 'all':
            raise ValueError("DAVO.inference_sequence: mode='feature' computes every pair (pairs='all')")
        N, sel, depth = self._sequence_args(img, flow_fwd, flow_bwd, seg, depth, pairs, "inference_sequence")
        if mode == 'feature':
            if flow_fwd is None or flow_bwd is None or seg is None:
                raise ValueError("DAVO.inference_sequence: mode='feature' reads flow_fwd, flow_bwd and seg")
            import torch
            img, seg, depth = self._upload(img, torch.uint8), self._upload(seg), self._upload(depth)
            flow_fwd, flow_bwd = self._upload(flow_fwd), self._upload(flow_bwd)
            ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
            return self._features(N - 2, as_torch, "davo_forward_sequence_features",
                                  lambda pose, table, stream: self._lib.davo_forward_sequence_features(
                                      self._h, N, ptr(img), ptr(flow_fwd), ptr(flow_bwd), ptr(seg), ptr(depth), ptr(pose),
                                      table, stream))
        if not _is_torch(img) and not self.config.batch_norm:
            return self.inference_sequence_async(img, flow_fwd, flow_bwd, seg, depth, pairs, _block=True).result()
        import torch
        dev = "cuda:%d" % self.device
        up = lambda t, dt: None if t is None else (t if _is_torch(t) else torch.as_tensor(np.ascontiguousarray(t))).to(
            device=dev, dtype=dt)
        img, flow_fwd, flow_bwd = up(img, torch.uint8), up(flow_fwd, torch.float32), up(flow_bwd, torch.float32)
        seg, depth = up(seg, torch.float32), up(depth, torch.float32)
        for name, t in (("img", img), ("flow_fwd", flow_fwd), ("flow_bwd", flow_bwd), ("seg", seg), ("depth", depth)):
            if t is not None and not (t.device.index == self.device and t.is_contiguous()):
                raise ValueError("DAVO.inference_sequence: %s must be a contiguous tensor on %s" % (name, dev))
        out = torch.empty((N - 2, 2, 6), dtype=torch.float32, device=dev)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.davo_forward_sequence(self._h, N, sel, ptr(img), ptr(flow_fwd), ptr(flow_bwd), ptr(seg),
                                                    ptr(depth), ptr(out), C.c_void_p(stream)), "davo_forward_sequence")
        return {'pose': out if as_torch else out.cpu().numpy()}

    def inference_sequence_async(self, img, flow_fwd, flow_bwd, seg, depth=None, pairs='all', _block=False):
        """``inference_sequence`` on host arrays without waiting (davo_forward_sequence_host with a ticket): returns
        the handle of ``inference_async``, whose ``.result()`` gives ``{'pose': [N-2,2,6]}``.  The arrays must not be
        modified before ``.result()``; up to 8 calls may be in flight."""
        N, sel, depth = self._sequence_args(img, flow_fwd, flow_bwd, seg, depth, pairs, "inference_sequence_async")
        if self.config.batch_norm:
            raise NotImplementedError("DAVO.inference_sequence_async: -batch_norm takes the device path (one pass per batch)")
        arr = lambda a, dt: None if a is None else np.ascontiguousarray(a, dtype=dt)
        img, flow_fwd, flow_bwd = arr(img, np.uint8), arr(flow_fwd, np.float32), arr(flow_bwd, np.float32)
        seg, depth = arr(seg, np.float32), arr(depth, np.float32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        if _block:
            out = np.empty((N - 2, 2, 6), np.float32)
            self._check(self._lib.davo_forward_sequence_host(self._h, N, sel, ptr(img), ptr(flow_fwd), ptr(flow_bwd),
                                                             ptr(seg), ptr(depth), ptr(out), None, None),
                        "davo_forward_sequence_host")
            return DAVO._Pending(self, None, out, None)
        import torch
        ring = getattr(self, "_async_out", None)
        if ring is None or ring[0].shape[0] < N - 2:
            ring = self._async_out = [torch.empty((max(N - 2, self.batch_size), 2, 6), dtype=torch.float32).pin_memory()
                                      for _ in range(8)]
            self._async_n = 0
        out = ring[self._async_n % 8][:N - 2].numpy()
        self._async_n += 1
        ticket = C.c_longlong(0)
        self._check(self._lib.davo_forward_sequence_host(self._h, N, sel, ptr(img), ptr(flow_fwd), ptr(flow_bwd), ptr(seg),
                                                         ptr(depth), ptr(out), None, C.byref(ticket)),
                    "davo_forward_sequence_host")
        return DAVO._Pending(self, ticket.value, out, (img, flow_fwd, flow_bwd, seg, depth))

    def odometry(self, pairs='trajectory', max_push=None, host=True):
        """An online odometry session on this handle (include/davo_b200.h: davo_odometry_*): push frames as they
        arrive, get every frame's absolute pose.  ``pairs``: ``'trajectory'`` (what the trajectory reads) or ``'all'``;
        ``max_push``: most frames per push (default: the handle's batch size); ``host``: pushes take numpy arrays and
        return numpy arrays, else CUDA tensors in and out."""
        return Odometry(self, pairs, self.batch_size if max_push is None else max_push, host)

    def _blob_header(self, blob, who):
        """The header of a blob this handle is to load, checked before any device work: the handle set up with weights
        loaded, a version-1 blob, saved by a handle of the same version, frame size and configuration."""
        if getattr(self, "_h", None) is None:
            raise ValueError("DAVO.%s: the handle is not set up (DAVO.setup_inference(mode='davo'))" % who)
        if not self._weights_loaded:
            raise ValueError("DAVO.%s: the handle has no weights loaded" % who)
        try:
            hdr = odometry_blob_header(blob)
        except ValueError as e:
            raise ValueError("DAVO.%s: %s" % (who, e))
        cfg = hdr["config"]
        if (cfg["H"], cfg["W"]) != (self.img_height, self.img_width):
            raise ValueError("DAVO.%s: the session's frames are %dx%d, this handle's %dx%d"
                             % (who, cfg["H"], cfg["W"], self.img_height, self.img_width))
        for name in _BLOB_CONFIG:
            if cfg[name] != getattr(self._cfg, name):
                raise ValueError("DAVO.%s: the session was saved by a handle of another version or configuration "
                                 "(davo_config.%s: %d in the blob, %d here)" % (who, name, cfg[name], getattr(self._cfg, name)))
        return hdr

    def odometry_load(self, blob):
        """A session saved by ``Odometry.save`` -- on this handle or another, in this process or another -- as a new
        session of this handle (include/davo_b200.h: davo_odometry_load).  Every later push gives the bits the saved
        session would have given; loading a blob twice forks the stream.  ``blob``: a buffer-protocol object."""
        hdr = self._blob_header(blob, "odometry_load")
        a = np.frombuffer(blob, np.uint8)
        out = C.c_void_p()
        import torch
        with torch.cuda.device(self.device):             # the call switches devices; torch's current one is restored
            self._check(self._lib.davo_odometry_load(self._h, C.c_void_p(a.ctypes.data), a.size, C.byref(out)),
                        "davo_odometry_load")
        return Odometry._adopt(self, out, hdr)

    def odometry_save_many(self, sessions):
        """The blobs of several sessions of this handle (include/davo_b200.h: davo_odometry_save_many), each what
        ``Odometry.save`` gives, as slices of one page-locked buffer (buffer-protocol objects), in list order.  The
        launches do not depend on the number of sessions; the sessions do not change."""
        sessions = list(sessions)
        if not sessions:
            raise ValueError("DAVO.odometry_save_many: no session")
        for i, od in enumerate(sessions):
            if not isinstance(od, Odometry) or od._system is not self:
                raise ValueError("DAVO.odometry_save_many: session %d is not a session of this handle" % i)
            if od._o is None:
                raise RuntimeError("DAVO.odometry_save_many: session %d is closed" % i)
        n = len(sessions)
        size = C.c_int64(0)
        total = 0
        for od in sessions:
            self._check(self._lib.davo_odometry_state_bytes(od._o, C.byref(size)), "davo_odometry_state_bytes")
            total += size.value
        import torch
        buf = torch.empty((total,), dtype=torch.uint8).pin_memory().numpy()
        offsets = (C.c_int64 * (n + 1))()
        with torch.cuda.device(self.device):
            self._check(self._lib.davo_odometry_save_many(n, (C.c_void_p * n)(*[od._o.value for od in sessions]),
                                                          C.c_void_p(buf.ctypes.data), total, offsets),
                        "davo_odometry_save_many")
        mv = memoryview(buf)
        return [mv[offsets[i]:offsets[i + 1]] for i in range(n)]

    def odometry_load_many(self, blobs):
        """New sessions of this handle from several blobs (include/davo_b200.h: davo_odometry_load_many), each as
        ``odometry_load`` would load it, in list order; all are checked before any is loaded, and a refused call loads
        none.  The blobs are gathered into one page-locked buffer, sent in one copy."""
        blobs = list(blobs)
        if not blobs:
            raise ValueError("DAVO.odometry_load_many: no blob")
        hdrs = [self._blob_header(b, "odometry_load_many: blob %d" % i) for i, b in enumerate(blobs)]
        n = len(blobs)
        offsets = (C.c_int64 * (n + 1))()
        for i, h in enumerate(hdrs):
            offsets[i + 1] = offsets[i] + h["bytes"]
        import torch
        buf = torch.empty((offsets[n],), dtype=torch.uint8).pin_memory().numpy()
        for i, b in enumerate(blobs):
            buf[offsets[i]:offsets[i + 1]] = np.frombuffer(b, np.uint8)
        out = (C.c_void_p * n)()
        with torch.cuda.device(self.device):
            self._check(self._lib.davo_odometry_load_many(self._h, n, C.c_void_p(buf.ctypes.data), offsets, out),
                        "davo_odometry_load_many")
        return [Odometry._adopt(self, C.c_void_p(out[i]), h) for i, h in enumerate(hdrs)]

    def _att_shape(self):
        """(slots, width) of a frame's attention weights: the far table is slot 1 under -se_flow_on_depthseg_seplayers;
        the width is that of get_intermediate('att_weights:<k>')."""
        c = self.config
        width = 19 if not c.pixel_map else 3 if c.pixel_map == 2 else 3 if c.att_src == 4 else 1 if c.att_src == 5 else 21
        return (2 if c.depth_split else 1), width

    def _att_host(self, n_t):
        return (np.empty((n_t, self.img_height, self.img_width), np.float32), np.empty((n_t, 2, 24), np.float32))

    def _result(self, pose, traj, frames, amap=None, aw=None):
        """A push's dict; with attention, the maps and the weight rows trimmed to the variant's slots and width."""
        out = {'pose': pose, 'trajectory': traj, 'frames': frames}
        if amap is not None:
            slots, width = self._att_shape()
            out['attention'], out['att_weights'] = amap, aw[:, :slots, :width]
        return out

    def _many_args(self, sessions, img, flow_fwd, flow_bwd, seg, depth, host, who):
        """The list and session checks of the batched pushes; returns the sessions, each entry's inputs and its
        (k, n_samples, n_traj)."""
        sessions = list(sessions)
        n = len(sessions)
        per = lambda x: [None] * n if x is None else list(x)
        lists = {"img": per(img), "flow_fwd": per(flow_fwd), "flow_bwd": per(flow_bwd), "seg": per(seg), "depth": per(depth)}
        for name, x in lists.items():
            if len(x) != n:
                raise ValueError("DAVO.%s: %s has %d entries for %d sessions" % (who, name, len(x), n))
        if n == 0:
            raise ValueError("DAVO.%s: no session" % who)
        for i, od in enumerate(sessions):
            if not isinstance(od, Odometry) or od._system is not self:
                raise ValueError("DAVO.%s: session %d is not a session of this handle" % (who, i))
            if od._host and not host:
                raise ValueError("DAVO.%s: session %d is a host session; a batched push takes device sessions "
                                 "(DAVO.odometry(host=False)); DAVO.odometry_push_many_host takes host sessions" % (who, i))
            if host and not od._host:
                raise ValueError("DAVO.%s: session %d is a device session; DAVO.odometry_push_many takes it" % (who, i))
            if any(od is o for o in sessions[:i]):
                raise ValueError("DAVO.%s: session %d is given twice" % (who, i))
        ins, counts = [], []
        for i, od in enumerate(sessions):                    # shapes of every entry
            x = [lists[name][i] for name in ("img", "flow_fwd", "flow_bwd", "seg", "depth")]
            k, x[4] = od._args(*x, who="DAVO.%s: session %d" % (who, i))
            ins.append(x)
            counts.append((k,) + od._counts(k))
        return sessions, ins, counts

    def odometry_push_many(self, sessions, img, flow_fwd, flow_bwd, seg=None, depth=None, attention=False):
        """One push on each of several device sessions of this handle, in one forward pass (include/davo_b200.h:
        davo_odometry_push_many).  ``img``, ``flow_fwd``, ``flow_bwd``, ``seg`` and ``depth`` are lists aligned with
        ``sessions``, entry i holding the CUDA tensors ``sessions[i].push`` takes (None, or a list of None, where no
        entry has one).  Returns the list of the dicts ``push`` returns; the results are the bits of pushing each
        session alone, in list order.  Enqueued on the current stream.  ``attention=True`` adds each session's
        ``'attention'`` and ``'att_weights'`` (``Odometry.push``), with one extra launch per micro-batch in all."""
        sessions, ins, counts = self._many_args(sessions, img, flow_fwd, flow_bwd, seg, depth, False, "odometry_push_many")
        n = len(sessions)
        for i, (od, x) in enumerate(zip(sessions, ins)):     # where the tensors live
            od._check_device(*x, who="DAVO.odometry_push_many: session %d" % i)
        import torch
        dev = "cuda:%d" % self.device
        outs = [(torch.zeros((ns, 2, 6), dtype=torch.float32, device=dev),
                 torch.empty((nt, 4, 4), dtype=torch.float64, device=dev)) for _, ns, nt in counts]
        vp = C.c_void_p
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None
        arr = lambda vals: (vp * n)(*vals)
        cols = [arr([ptr(x[j]) for x in ins]) for j in range(5)]
        ns, nt = (C.c_int * n)(), (C.c_int * n)()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        head = (n, arr([od._o.value for od in sessions]), (C.c_int * n)(*[c[0] for c in counts]), *cols,
                arr([ptr(o[0]) for o in outs]), arr([ptr(o[1]) for o in outs]))
        atts = [(None, None)] * n
        if attention:
            atts = [(torch.empty((c[2], self.img_height, self.img_width), dtype=torch.float32, device=dev),
                     torch.empty((c[2], 2, 24), dtype=torch.float32, device=dev)) for c in counts]
            table = (_capi.DavoOdometryAttentionC * n)(*[_capi.DavoOdometryAttentionC(ptr(a), ptr(w)) for a, w in atts])
            self._check(self._lib.davo_odometry_push_many_attention(*head, table, ns, nt, vp(stream)),
                        "davo_odometry_push_many_attention")
        else:
            self._check(self._lib.davo_odometry_push_many(*head, ns, nt, vp(stream)), "davo_odometry_push_many")
        res = []
        for od, (k, _, _), (pose, traj), m, (a, w) in zip(sessions, counts, outs, nt, atts):
            res.append(self._result(pose, traj, range(od._posed, od._posed + m), a, w))
            od._pushed += k
            od._posed += m
        return res

    def odometry_push_many_host(self, sessions, img, flow_fwd, flow_bwd, seg=None, depth=None, attention=False):
        """One push on each of several host sessions of this handle, in one forward pass (include/davo_b200.h:
        davo_odometry_push_many_host): many cameras whose frames arrive in host memory.  The lists are those of
        ``odometry_push_many``, holding the numpy arrays ``sessions[i].push`` takes.  Returns the list of the dicts
        ``push`` returns; the results are the bits of pushing each session alone, in list order.  ``attention`` as
        for ``odometry_push_many``, as numpy arrays."""
        return self.odometry_push_many_host_async(sessions, img, flow_fwd, flow_bwd, seg, depth, _block=True,
                                                  attention=attention).result()

    def odometry_push_many_host_async(self, sessions, img, flow_fwd, flow_bwd, seg=None, depth=None, _block=False,
                                      attention=False):
        """``odometry_push_many_host`` without waiting: returns a handle whose ``.result()`` gives the list of dicts.
        The results land in each session's page-locked ring slot (as ``Odometry.push_async``); the inputs must stay
        unmodified until ``.result()``.  Up to 8 calls may be in flight."""
        who = "odometry_push_many_host"
        sessions, ins, counts = self._many_args(sessions, img, flow_fwd, flow_bwd, seg, depth, True, who)
        n = len(sessions)
        conv = lambda a, dt: None if a is None else np.ascontiguousarray(a, dtype=dt)
        dts = (np.uint8, np.float32, np.float32, np.float32, np.float32)
        ins = [tuple(conv(a, dt) for a, dt in zip(x, dts)) for x in ins]
        if _block:
            outs = [(np.zeros((ns, 2, 6), np.float32), np.empty((nt, 4, 4), np.float64))
                    + (self._att_host(nt) if attention else (None, None)) for _, ns, nt in counts]
        else:
            outs = [od._ring_slot(ns, nt, attention) for od, (_, ns, nt) in zip(sessions, counts)]
        vp = C.c_void_p
        hp = lambda a: a.ctypes.data if a is not None and a.size else None
        arr = lambda vals: (vp * n)(*vals)
        cols = [arr([hp(x[j]) for x in ins]) for j in range(5)]
        ns, nt = (C.c_int * n)(), (C.c_int * n)()
        ticket = C.c_longlong(0)
        head = (n, arr([od._o.value for od in sessions]), (C.c_int * n)(*[c[0] for c in counts]), *cols,
                arr([hp(o[0]) for o in outs]), arr([hp(o[1]) for o in outs]))
        tail = (ns, nt, None, None if _block else C.byref(ticket))
        if attention:
            table = (_capi.DavoOdometryAttentionC * n)(*[_capi.DavoOdometryAttentionC(hp(o[2]), hp(o[3])) for o in outs])
            self._check(self._lib.davo_odometry_push_many_host_attention(*head, table, *tail),
                        "davo_odometry_push_many_host_attention")
        else:
            self._check(self._lib.davo_odometry_push_many_host(*head, *tail), "davo_odometry_push_many_host")
        res = []
        for od, (k, _, _), o, m in zip(sessions, counts, outs, nt):
            res.append(Odometry._Pending(None, self._result(o[0], o[1], range(od._posed, od._posed + m), o[2], o[3])))
            od._pushed += k
            od._posed += m
        return DAVO._PendingMany(self, None if _block else ticket.value, res, None if _block else ins)

    class _PendingMany(object):
        """A queued batched host push; ``result()`` waits for it and returns the list of the dicts ``push`` returns."""

        def __init__(self, system, ticket, pending, keep):
            self._system, self._ticket, self._pending, self._keep = system, ticket, pending, keep

        def result(self):
            if self._ticket is not None:
                s = self._system
                s._check(s._lib.davo_host_wait(s._h, self._ticket), "davo_host_wait")
                self._ticket, self._keep = None, None
                for p in self._pending:                      # own copies: the pinned ring slots are reused
                    p._out = {k: (v if k == 'frames' else np.array(v)) for k, v in p._out.items()}
            return [p.result() for p in self._pending]

    def bind_host_numa(self):
        """Bind this thread (and threads created after it) to the CPUs next to this handle's GPU
        (``davo_bind_host_numa``); call it before allocating pinned inputs.  Returns the NUMA node or -1."""
        return int(self._lib.davo_bind_host_numa(self._h))

    # ------------------------------------------------------ test / debug taps
    def get_intermediate(self, name: str, pair: int) -> np.ndarray:
        """What the last forward left for ``pair`` under ``name`` (include/davo_b200.h: davo_get_intermediate), flat."""
        buf = np.empty((self.img_height * self.img_width * 16,), np.float32)
        n = C.c_int64(0)
        rc = self._lib.davo_get_intermediate(self._h, name.encode(), pair, buf.ctypes.data_as(C.c_void_p), buf.size,
                                             C.byref(n))
        if rc != 0 and n.value > buf.size:                   # the library names the size it needs
            buf = np.empty((n.value,), np.float32)
            rc = self._lib.davo_get_intermediate(self._h, name.encode(), pair, buf.ctypes.data_as(C.c_void_p), buf.size,
                                                 C.byref(n))
        self._check(rc, "davo_get_intermediate(%s)" % name)
        return buf[:n.value].copy()

    def last_host_copy_bytes(self):
        """(host->device, device->host) bytes moved by the last numpy-input inference."""
        a, b = C.c_longlong(0), C.c_longlong(0)
        self._check(self._lib.davo_last_host_copy_bytes(self._h, C.byref(a), C.byref(b)),
                    "davo_last_host_copy_bytes")
        return int(a.value), int(b.value)

    def last_launch_count(self) -> int:
        return int(self._lib.davo_last_launch_count(self._h))

    def profile_layers(self, iters: int = 10):
        """Mean ms per kernel of one micro-batch: front, cnv1..cnv7, head; and pairs per launch."""
        import torch
        ms = (C.c_float * 9)()
        n = C.c_int(0)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.davo_profile_layers(self._h, iters, ms, C.byref(n), C.c_void_p(stream)),
                    "davo_profile_layers")
        names = ["front", "cnv1", "cnv2", "cnv3", "cnv4", "cnv5", "cnv6", "cnv7", "head"]
        return dict(zip(names, [float(v) for v in ms])), int(n.value)

    def _debug_set_conv_impl(self, impl: int):
        self._graph, self._graph_key, self._graph_hits = None, None, 0      # a captured graph holds the old path
        self._check(self._lib.davo_debug_set_conv_impl(self._h, impl), "davo_debug_set_conv_impl")

    # ------------------------------------------------------------------ multi-GPU
    def init_comm(self, rank=None, world=None):
        """Build the handle's NCCL communicator (``davo_comm_create``).  Collective: every rank
        calls it.  The 128-byte id made on rank 0 travels over the already initialised
        ``torch.distributed`` group (plumbing only; the gather itself is the library's)."""
        import torch
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            if world in (None, 1):
                return 1
            raise RuntimeError("DAVO.init_comm: torch.distributed is not initialised")
        rank = dist.get_rank() if rank is None else rank
        world = dist.get_world_size() if world is None else world
        if world == 1:
            return 1
        ident = (C.c_ubyte * 128)()
        if rank == 0:
            rc = self._lib.davo_comm_unique_id(ident)
            if rc != 0:
                raise RuntimeError("davo_comm_unique_id failed (%d): %s" % (rc, _capi.last_error(self._lib, None)))
        box = [bytes(ident)]
        dist.broadcast_object_list(box, src=0)
        ident = (C.c_ubyte * 128).from_buffer_copy(box[0])
        self._check(self._lib.davo_comm_create(self._h, ident, rank, world), "davo_comm_create")
        self._comm_world = world
        return world

    def comm_world(self) -> int:
        return getattr(self, "_comm_world", 1)

    def allgather_poses(self, local_poses):
        """``[n_local,2,6]`` CUDA tensor of this rank -> ``[world*n_local,2,6]`` in rank order,
        enqueued on the current stream (``davo_allgather_poses``)."""
        import torch
        assert local_poses.is_cuda and local_poses.dtype == torch.float32 and tuple(local_poses.shape[1:]) == (2, 6)
        local_poses = local_poses.contiguous()
        n_local = int(local_poses.shape[0])
        out = torch.empty((self.comm_world() * n_local, 2, 6), dtype=torch.float32, device=local_poses.device)
        stream = torch.cuda.current_stream(local_poses.device).cuda_stream
        self._check(self._lib.davo_allgather_poses(self._h, None, C.c_void_p(local_poses.data_ptr()), n_local,
                                                   C.c_void_p(out.data_ptr()), C.c_void_p(stream)),
                    "davo_allgather_poses")
        return out

    def close(self):
        self._graph = None
        if self._h is not None and self._lib is not None:
            self._lib.davo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Odometry(object):
    """An online odometry session (``DAVO.odometry``).  ``push(img, flow_fwd, flow_bwd, seg, depth=None)`` takes the next
    k frames of the sequence: ``img`` uint8 [k,H,W,3], ``seg`` / ``depth`` float32 [k,H,W,1], ``flow_fwd`` / ``flow_bwd``
    float32 [k',H,W,2] with k' = k, or k-1 on the first push (entry j: the flow between the frame before frame j of the
    push and frame j; on the first push between frames j and j+1).  It returns ``{'pose': [n_s,2,6], 'trajectory':
    [n_t,4,4] float64, 'frames': range of the frame indices of the trajectory rows}``: the poses of the samples whose
    last frame is new and the absolute poses that became known.  ``push_async`` queues a host push and returns a handle
    whose ``.result()`` gives that dict (the inputs must stay unmodified until then; up to 8 in flight)."""

    def __init__(self, system, pairs, max_push, host):
        if pairs not in ('trajectory', 'all'):
            raise ValueError("DAVO.odometry: pairs must be 'trajectory' or 'all'")
        if not system._weights_loaded:
            raise RuntimeError("DAVO.odometry: weights not loaded")
        self._system, self._host, self._pushed, self._posed = system, bool(host), 0, 0
        self._ring, self._ring_n = None, 0
        self.pairs = pairs
        h = C.c_void_p()
        system._check(system._lib.davo_odometry_create(system._h, int(max_push), _capi.PAIRS[pairs], int(self._host),
                                                       C.byref(h)), "davo_odometry_create")
        self._o, self.max_push = h, int(max_push)

    def _counts(self, k):
        f0 = self._pushed
        ns = max(0, f0 + k - 2) - max(0, f0 - 2)
        return ns, ns + 2 if (f0 <= 2 and ns > 0) else ns

    def _args(self, img, flow_fwd, flow_bwd, seg, depth, who="Odometry.push"):
        s = self._system
        if self._o is None:
            raise RuntimeError("%s: the session is closed" % who)
        if s.config.att_src != V.ATT_SE_DEPTH_SEG and not s.config.depth_split:
            depth = None
        elif depth is None:
            raise ValueError("%s: version %r reads depth [k,H,W,1]" % (who, s.version))
        k, H, W = int(img.shape[0]), s.img_height, s.img_width
        kf = k if self._pushed > 0 else k - 1
        want = {"img": (k, H, W, 3), "flow_fwd": (kf, H, W, 2), "flow_bwd": (kf, H, W, 2), "seg": (k, H, W, 1),
                "depth": (k, H, W, 1)}
        for name, t in (("img", img), ("flow_fwd", flow_fwd), ("flow_bwd", flow_bwd), ("seg", seg), ("depth", depth)):
            if t is not None and tuple(t.shape) != want[name]:
                raise ValueError("%s: %s has shape %s, expected %s" % (who, name, tuple(t.shape), want[name]))
        return k, depth

    def _check_device(self, img, flow_fwd, flow_bwd, seg, depth, who="Odometry.push"):
        import torch
        dev = "cuda:%d" % self._system.device
        for name, t, dt in (("img", img, torch.uint8), ("flow_fwd", flow_fwd, torch.float32),
                            ("flow_bwd", flow_bwd, torch.float32), ("seg", seg, torch.float32),
                            ("depth", depth, torch.float32)):
            if t is not None and not (_is_torch(t) and t.is_cuda and t.device.index == self._system.device
                                      and t.dtype == dt and t.is_contiguous()):
                raise ValueError("%s: %s must be a contiguous %s tensor on %s" % (who, name, dt, dev))

    def _call(self, k, ins, pose, traj, stream, ticket, att=None):
        s = self._system
        ns, nt = C.c_int(0), C.c_int(0)
        if att is None:
            s._check(s._lib.davo_odometry_push(self._o, k, *ins, pose, traj, C.byref(ns), C.byref(nt), stream, ticket),
                     "davo_odometry_push")
        else:
            s._check(s._lib.davo_odometry_push_attention(self._o, k, *ins, pose, traj, C.byref(att), C.byref(ns),
                                                         C.byref(nt), stream, ticket), "davo_odometry_push_attention")
        frames = range(self._posed, self._posed + nt.value)
        self._pushed += k
        self._posed += nt.value
        return frames

    def push_async(self, img, flow_fwd, flow_bwd, seg=None, depth=None, _block=False, attention=False):
        k, depth = self._args(img, flow_fwd, flow_bwd, seg, depth)
        n_s, n_t = self._counts(k)
        s = self._system
        if not self._host:
            import torch
            dev = "cuda:%d" % s.device
            self._check_device(img, flow_fwd, flow_bwd, seg, depth)
            pose = torch.zeros((n_s, 2, 6), dtype=torch.float32, device=dev)
            traj = torch.empty((n_t, 4, 4), dtype=torch.float64, device=dev)
            ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None and t.numel() else None
            amap = aw = att = None
            if attention:
                amap = torch.empty((n_t, s.img_height, s.img_width), dtype=torch.float32, device=dev)
                aw = torch.empty((n_t, 2, 24), dtype=torch.float32, device=dev)
                att = _capi.DavoOdometryAttentionC(ptr(amap), ptr(aw))
            stream = torch.cuda.current_stream(s.device).cuda_stream
            frames = self._call(k, [ptr(t) for t in (img, flow_fwd, flow_bwd, seg, depth)], ptr(pose), ptr(traj),
                                C.c_void_p(stream), None, att)
            return Odometry._Pending(None, s._result(pose, traj, frames, amap, aw), None)
        arr = lambda a, dt: None if a is None else np.ascontiguousarray(a, dtype=dt)
        ins = (arr(img, np.uint8), arr(flow_fwd, np.float32), arr(flow_bwd, np.float32), arr(seg, np.float32),
               arr(depth, np.float32))
        hp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None
        if _block:
            pose, traj = np.zeros((n_s, 2, 6), np.float32), np.empty((n_t, 4, 4), np.float64)
            amap, aw = s._att_host(n_t) if attention else (None, None)
        else:
            pose, traj, amap, aw = self._ring_slot(n_s, n_t, attention)
        att = _capi.DavoOdometryAttentionC(hp(amap), hp(aw)) if attention else None
        ticket = C.c_longlong(0)
        frames = self._call(k, [hp(a) for a in ins], hp(pose), hp(traj), None, None if _block else C.byref(ticket), att)
        out = s._result(pose, traj, frames, amap, aw)
        if _block:
            return Odometry._Pending(None, out, None)
        return Odometry._Pending(s, out, ticket.value, ins)

    def _ring_slot(self, n_s, n_t, attention=False):
        """The next page-locked (pose, trajectory, map, weights) outputs of an asynchronous host push, single or batched;
        map and weights are None unless asked for.  The attention slots are allocated by the first push that asks
        (a 128x416 map is 213 KB: a ring of them for every session would pin far more than the poses need)."""
        import torch
        if self._ring is None:                      # page-locked results, one slot per call that can be in flight
            self._ring = [(torch.empty((self.max_push, 2, 6), dtype=torch.float32).pin_memory(),
                           torch.empty((self.max_push + 2, 4, 4), dtype=torch.float64).pin_memory()) for _ in range(8)]
        i = self._ring_n % 8
        self._ring_n += 1
        slot = self._ring[i]
        amap = aw = None
        if attention:
            s = self._system
            if getattr(self, "_att_ring", None) is None:
                self._att_ring = [(torch.empty((self.max_push + 2, s.img_height, s.img_width), dtype=torch.float32).pin_memory(),
                                   torch.empty((self.max_push + 2, 2, 24), dtype=torch.float32).pin_memory())
                                  for _ in range(8)]
            amap, aw = self._att_ring[i][0][:n_t].numpy(), self._att_ring[i][1][:n_t].numpy()
        return slot[0][:n_s].numpy(), slot[1][:n_t].numpy(), amap, aw

    def push(self, img, flow_fwd, flow_bwd, seg=None, depth=None, attention=False):
        """See the class.  ``attention=True`` adds each posed frame's attention (include/davo_b200.h:
        davo_odometry_push_attention): ``'attention'`` [n_t,H,W], the map of the frame of ``trajectory[i]`` as the pair
        that placed it masks it, and ``'att_weights'`` [n_t,slots,width], the table(s) it was computed from (slots 2
        under -se_flow_on_depthseg_seplayers, else 1; width that of ``get_intermediate('att_weights:<k>')``; zeros for
        a map of ones).  CUDA tensors for device sessions, numpy for host sessions."""
        return self.push_async(img, flow_fwd, flow_bwd, seg, depth, _block=True, attention=attention).result()

    class _Pending(object):
        def __init__(self, system, out, ticket=None, keep=None):
            self._system, self._out, self._ticket, self._keep = system, out, ticket, keep

        def result(self):
            if self._ticket is not None:
                s = self._system
                s._check(s._lib.davo_host_wait(s._h, self._ticket), "davo_host_wait")
                self._ticket, self._keep = None, None
                # own copies: the pinned ring slot is reused
                self._out = {k: (v if k == 'frames' else np.array(v)) for k, v in self._out.items()}
            return self._out

    def move_to(self, system):
        """Re-home this session onto the handle ``system``, which may be on another GPU (include/davo_b200.h:
        davo_odometry_move): every later push gives the bits it would have given without the move, and the session now
        belongs to ``system`` (its ``close`` destroys the session; a batched push on ``system`` takes it).  The target
        is checked before any device work: set up, weights loaded, the same version and frame size.  Waits for the
        session's device and returns once the carried state has been copied.  Returns ``self``."""
        s = self._system
        if self._o is None:
            raise RuntimeError("Odometry.move_to: the session is closed")
        if s._h is None:
            raise RuntimeError("Odometry.move_to: the session was destroyed with its handle")
        if system is s:
            return self
        if not isinstance(system, DAVO) or getattr(system, "_h", None) is None:
            raise ValueError("Odometry.move_to: the target is not set up (DAVO.setup_inference(mode='davo'))")
        if not system._weights_loaded:
            raise ValueError("Odometry.move_to: the target has no weights loaded")
        if system.version != s.version:
            raise ValueError("Odometry.move_to: the target runs version %r, the session %r" % (system.version, s.version))
        if (system.img_height, system.img_width) != (s.img_height, s.img_width):
            raise ValueError("Odometry.move_to: the target's frames are %dx%d, the session's %dx%d"
                             % (system.img_height, system.img_width, s.img_height, s.img_width))
        import torch
        with torch.cuda.device(s.device):                 # the call switches devices; torch's current one is restored
            s._check(s._lib.davo_odometry_move(self._o, system._h), "davo_odometry_move")
        self._system = system
        return self

    @classmethod
    def _adopt(cls, system, h, hdr):
        """The Python side of a session the library loaded onto ``system`` (DAVO.odometry_load): its kind from the
        blob's header, its counts from the library."""
        od = cls.__new__(cls)
        od._system, od._host, od._o, od.max_push, od.pairs = system, hdr["host"], h, hdr["max_push"], hdr["pairs"]
        od._ring, od._ring_n = None, 0
        pushed, posed = C.c_longlong(0), C.c_longlong(0)
        system._check(system._lib.davo_odometry_frames(h, C.byref(pushed), C.byref(posed)), "davo_odometry_frames")
        od._pushed, od._posed = int(pushed.value), int(posed.value)
        return od

    def save(self):
        """This session's carried state as bytes (include/davo_b200.h: davo_odometry_save): ``DAVO.odometry_load`` on a
        handle of the same version, frame size and weights -- in this process or another -- continues the stream with
        the bits this session would give.  Does not change the session; waits for the work queued on its device,
        host pushes in flight included."""
        s = self._system
        if self._o is None:
            raise RuntimeError("Odometry.save: the session is closed")
        if s._h is None:
            raise RuntimeError("Odometry.save: the session was destroyed with its handle")
        size = C.c_int64(0)
        s._check(s._lib.davo_odometry_state_bytes(self._o, C.byref(size)), "davo_odometry_state_bytes")
        buf = np.empty((size.value,), np.uint8)
        import torch
        with torch.cuda.device(s.device):
            s._check(s._lib.davo_odometry_save(self._o, C.c_void_p(buf.ctypes.data), buf.size, C.byref(size)),
                     "davo_odometry_save")
        return buf.tobytes()

    def frames(self):
        """(frames pushed, frames whose absolute pose has been returned)."""
        return self._pushed, self._posed

    def reset(self):
        """The next push is frame 0 of a new sequence."""
        if self._o is not None:
            self._system._check(self._system._lib.davo_odometry_reset(self._o), "davo_odometry_reset")
        self._pushed, self._posed = 0, 0

    def close(self):
        if self._o is not None and self._system._h is not None:
            self._system._lib.davo_odometry_destroy(self._o)
        self._o = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
