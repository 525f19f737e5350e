"""Batched device-resident engine: rtpose VGG19 forward + fused post-processing behind the C ABI.

This is the new batched entry point SURVEY.md 8(b) asks for (`infer_batch`); the reference-shaped per-image calls
(get_model().forward, get_outputs, paf_to_pose_cpp) are thin wrappers over the same native objects.
"""
import ctypes

import numpy as np

from . import _native as nat


class NativeNet:
    """Owns a b200pose_net handle on one CUDA device."""

    def __init__(self, device_index):
        self._h = ctypes.c_void_p()
        nat.check(nat.lib().b200pose_net_create(ctypes.byref(self._h), int(device_index)), "b200pose_net_create")
        self.device_index = int(device_index)

    def load_state_dict_arrays(self, arrays):
        """arrays: 184 float32 numpy arrays in the reference state_dict order."""
        L = nat.lib()
        if len(arrays) != nat.NUM_TENSORS:
            raise nat.B200PoseError("expected %d tensors, got %d" % (nat.NUM_TENSORS, len(arrays)))
        for i, a in enumerate(arrays):
            a = np.ascontiguousarray(a, dtype=np.float32)
            nat.check(L.b200pose_net_set_tensor(self._h, i, a.ctypes.data, a.size), "set_tensor(%d)" % i)
        nat.check(L.b200pose_net_finalize(self._h), "b200pose_net_finalize")

    def set_preprocess(self, name):
        """Normalisation fused into the uint8 entry points: 'rtpose' (default), 'vgg', 'inception' or 'ssd'
        (lib/datasets/preprocessing.py; get_outputs' `preprocess` argument)."""
        if name not in nat.PREPROCESS:
            raise nat.B200PoseError("unknown preprocess %r (expected one of %s)" % (name, sorted(nat.PREPROCESS)))
        nat.check(nat.lib().b200pose_net_set_preprocess(self._h, nat.PREPROCESS[name]), "b200pose_net_set_preprocess")

    def forward_ptr(self, in_ptr, in_on_device, n, H, W, mode, out_ptrs, out_on_device, stream):
        arr = (ctypes.c_void_p * 12)(*[ctypes.c_void_p(p) if p else None for p in out_ptrs])
        nat.check(nat.lib().b200pose_net_forward(self._h, ctypes.c_void_p(in_ptr), int(in_on_device), n, H, W, mode,
                                                 arr, int(out_on_device), ctypes.c_void_p(stream)), "b200pose_net_forward")

    def forward_u8_ptr(self, in_ptr, in_on_device, n, H, W, mode, out_ptrs, out_on_device, stream):
        """uint8 HWC BGR frames [n,H,W,3]; rtpose_preprocess is fused into the first convolution."""
        arr = (ctypes.c_void_p * 12)(*[ctypes.c_void_p(p) if p else None for p in out_ptrs])
        nat.check(nat.lib().b200pose_net_forward_u8(self._h, ctypes.c_void_p(in_ptr), int(in_on_device), n, H, W, mode,
                                                    arr, int(out_on_device), ctypes.c_void_p(stream)),
                  "b200pose_net_forward_u8")

    def forward_u8_ragged_ptr(self, in_ptr, in_on_device, n, H, W, ext_h, ext_w, mode, out_ptrs, out_on_device, stream):
        """Ragged batch: uint8 HWC BGR canvas [n,H,W,3], frame i valid in its top-left ext_h[i] x ext_w[i] (multiples of
        8); outputs canvas-shaped, +0 outside each extent, bit-identical to forward_u8_ptr of each frame alone inside."""
        if len(ext_h) != n or len(ext_w) != n:
            raise nat.B200PoseError("forward_u8_ragged_ptr: %d images but %d / %d extents" % (n, len(ext_h), len(ext_w)))
        arr = (ctypes.c_void_p * 12)(*[ctypes.c_void_p(p) if p else None for p in out_ptrs])
        eh = (ctypes.c_int * n)(*[int(v) for v in ext_h])
        ew = (ctypes.c_int * n)(*[int(v) for v in ext_w])
        nat.check(nat.lib().b200pose_net_forward_u8_ragged(self._h, ctypes.c_void_p(in_ptr), int(in_on_device), n, H, W,
                                                           eh, ew, mode, arr, int(out_on_device), ctypes.c_void_p(stream)),
                  "b200pose_net_forward_u8_ragged")

    def crop_with_factor(self, images, dest_size=368, factor=8):
        """Device-side crop_with_factor (im_transform.py:119-134) of uint8 BGR frames of one size: [n,h,w,3] or [h,w,3]
        -> (padded frames, im_scale, resized shape) like the reference (which returns them for one image)."""
        images = np.ascontiguousarray(images, dtype=np.uint8)
        single = images.ndim == 3
        if single:
            images = images[None]
        n, sh, sw, c = images.shape
        if c != 3:
            raise nat.B200PoseError("crop_with_factor: expected 3-channel BGR frames")
        scale, (rh, rw), (ph, pw) = nat.crop_geometry(sh, sw, dest_size, factor)
        out = np.empty((n, ph, pw, 3), np.uint8)
        nat.check(nat.lib().b200pose_net_crop_with_factor(self._h, ctypes.c_void_p(images.ctypes.data), 0, n, sh, sw,
                                                          int(dest_size), int(factor), ctypes.c_void_p(out.ctypes.data), 0,
                                                          None), "b200pose_net_crop_with_factor")
        return (out[0] if single else out), scale, (rh, rw, 3)

    def __del__(self):
        try:
            if self._h:
                nat.lib().b200pose_net_destroy(self._h)
                self._h = None
        except Exception:
            pass


class NativePost:
    """Owns a b200pose_post handle (fused NMS + PAF scoring + matching + assembly)."""

    def __init__(self, device_index, batch_cap=32, peak_cap=1024, human_cap=1024):
        self._h = ctypes.c_void_p()
        nat.check(nat.lib().b200pose_post_create(ctypes.byref(self._h), int(device_index), batch_cap, peak_cap, human_cap),
                  "b200pose_post_create")
        self.batch_cap, self.peak_cap, self.human_cap = batch_cap, peak_cap, human_cap

    def run(self, heat_ptr, paf_ptr, on_device, layout, n, h, w, thresh, stream=0):
        nat.check(nat.lib().b200pose_post_run(self._h, ctypes.c_void_p(heat_ptr), ctypes.c_void_p(paf_ptr), int(on_device),
                                              layout, n, h, w, ctypes.c_float(thresh), ctypes.c_void_p(stream)),
                  "b200pose_post_run")

    def flip_merge(self, normal_heat, flipped_heat, normal_paf, flipped_paf, layout=1):
        """Device-side handle_paf_and_heat (evaluate/coco_eval.py:197-242) on host float32 arrays.
        layout 1: heat [n,h,w,19] / paf [n,h,w,38] (or a single image [h,w,C]); layout 0: [n,C,h,w].
        Returns (averaged_paf, averaged_heat) like the reference; the inputs are not modified."""
        arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in (normal_heat, flipped_heat, normal_paf, flipped_paf)]
        single = arrs[0].ndim == 3
        if single:
            arrs = [a[None] for a in arrs]
        if layout == 1:
            n, h, w, ch = arrs[0].shape
            cp = arrs[2].shape[3]
        else:
            n, ch, h, w = arrs[0].shape
            cp = arrs[2].shape[1]
        if ch != 19 or cp != 38 or arrs[1].shape != arrs[0].shape or arrs[3].shape != arrs[2].shape:
            raise nat.B200PoseError("flip_merge: expected heat with 19 and paf with 38 channels, equal shapes")
        out_heat, out_paf = np.empty_like(arrs[0]), np.empty_like(arrs[2])
        nat.check(nat.lib().b200pose_flip_merge(self._h, *[ctypes.c_void_p(a.ctypes.data) for a in arrs], 0, int(layout),
                                                n, h, w, ctypes.c_void_p(out_heat.ctypes.data),
                                                ctypes.c_void_p(out_paf.ctypes.data), None), "b200pose_flip_merge")
        return (out_paf[0], out_heat[0]) if single else (out_paf, out_heat)

    def sync(self):
        nat.check(nat.lib().b200pose_post_sync(self._h), "b200pose_post_sync")

    def last_ticket(self):
        return int(nat.lib().b200pose_post_last_ticket(self._h))

    def select(self, ticket):
        """Wait for run `ticket` (one of the last two submitted) and make the getters read its results."""
        nat.check(nat.lib().b200pose_post_select(self._h, int(ticket)), "b200pose_post_select")

    def status(self, img):
        return int(nat.lib().b200pose_post_status(self._h, img))

    def status_accum(self, reset=False):
        """OR of the status bits of every image of every run since the last reset (waits for the second stream)."""
        st = int(nat.lib().b200pose_post_status_accum(self._h, int(bool(reset))))
        if st < 0:
            nat.check(1, "b200pose_post_status_accum")
        return st

    def check_status(self, n):
        for i in range(n):
            st = self.status(i)
            if st < 0 or (st & 0xF):
                raise nat.B200PoseError("post-processing capacity exceeded on image %d (status bits %d: 1=peaks>%d per "
                                        "part, 2=candidate pool, 4=rows, 8=humans>%d); raise the caps"
                                        % (i, st & 0xF, self.peak_cap, self.human_cap))

    def humans(self, img):
        """float32 [k, 73]: score, 18 x (x, y, peak score, peak id | -1)."""
        L = nat.lib()
        k = L.b200pose_post_num_humans(self._h, img)
        if k < 0:
            nat.check(1, "b200pose_post_num_humans")
        out = np.empty((max(k, 1), nat.HUMAN_FLOATS), np.float32)
        got = L.b200pose_post_get_humans(self._h, img, out.ctypes.data, k)
        return out[:got]

    def peaks(self, img):
        """float32 [P, 5]: x, y, score, id, part (the joint_list of paf_to_pose.py:376-378)."""
        cap = 18 * self.peak_cap
        out = np.empty((cap, 5), np.float32)
        got = nat.lib().b200pose_post_get_peaks(self._h, img, out.ctypes.data, cap)
        if got < 0:
            nat.check(1, "b200pose_post_get_peaks")
        return out[:got].copy()

    def __del__(self):
        try:
            if self._h:
                nat.lib().b200pose_post_destroy(self._h)
                self._h = None
        except Exception:
            pass


def humans_to_dicts(rows, width, height):
    """[(score, {part: (x/width, y/height, peak score)})] - the content paf_to_pose_cpp puts into Human objects.
    Conversions are done in bulk (float32 -> Python float, i.e. double, then the divisions in double exactly like the
    reference's `float(x) / W`); the per-person dictionaries are the only Python-level loop left."""
    rows = np.asarray(rows, dtype=np.float32).reshape(-1, nat.HUMAN_FLOATS)
    if rows.shape[0] == 0:
        return []
    body = rows[:, 1:].reshape(-1, 18, 4).astype(np.float64)
    xs = (body[:, :, 0] / width).tolist()
    ys = (body[:, :, 1] / height).tolist()
    ss = body[:, :, 2].tolist()
    present = (body[:, :, 3] >= 0).tolist()
    scores = rows[:, 0].astype(np.float64).tolist()
    out = []
    for k in range(len(scores)):
        pr, x, y, sc = present[k], xs[k], ys[k], ss[k]
        parts = {p: (x[p], y[p], sc[p]) for p in range(18) if pr[p]}
        if parts:
            out.append((scores[k], parts))
    return out


def _of_image(v, i):
    """Padded size of image i of a run: runs of one shape keep an int, ragged runs a tuple per image."""
    return v[i] if isinstance(v, tuple) else v


def ragged_groups(padded_shapes, batch_cap):
    """Frames of different padded sizes [(ph, pw), ...] -> ragged runs: a list of (frame indices, (canvas_h, canvas_w)).
    Landscape (ph <= pw) and portrait frames go to separate runs: the short side is dest_size for both, so a run's canvas
    only wastes pixels along the long side.  Each orientation is sorted by the padded long side (ties in input order) and
    cut into runs of at most batch_cap frames; the canvas of a run is the largest ph x the largest pw of its frames."""
    if batch_cap < 1:
        raise nat.B200PoseError("ragged_groups: batch_cap must be >= 1")
    shapes = [(int(h), int(w)) for h, w in padded_shapes]
    land = sorted((i for i, (h, w) in enumerate(shapes) if h <= w), key=lambda i: (shapes[i][1], i))
    port = sorted((i for i, (h, w) in enumerate(shapes) if h > w), key=lambda i: (shapes[i][0], i))
    runs = []
    for idx in (land, port):
        for k in range(0, len(idx), batch_cap):
            part = idx[k:k + batch_cap]
            runs.append((part, (max(shapes[i][0] for i in part), max(shapes[i][1] for i in part))))
    return runs


class PoseEngine:
    """Fused batched inference on one GPU: images -> humans, maps never leave the device."""

    def __init__(self, state_arrays, device_index=0, mode="bf16", batch_cap=32, peak_cap=1024, human_cap=1024, net=None):
        if net is None:
            net = NativeNet(device_index)
            net.load_state_dict_arrays(state_arrays)
        self.net = net
        self.post = NativePost(device_index, batch_cap, peak_cap, human_cap)
        self.mode = nat.MODES[mode]
        self.device_index = device_index
        self._shapes = {}
        self._last = None

    def _remember(self, n, H, W):
        """Shape of the run just submitted, kept per ticket (two runs may be in flight with different batch sizes or
        frame shapes: fetch(ticket=i) must read run i with run i's n and normalise image k by run i's W[k] / H[k]).
        H, W: one padded size for the whole run, or per-image tuples (ragged runs)."""
        t = self.post.last_ticket()
        if self.__dict__.get("_shapes") is None:
            self._shapes = {}
        self._shapes[t] = (n, H, W)
        for old in [k for k in self._shapes if k < t - 1]:
            del self._shapes[old]
        self._last = (n, H, W)
        return t

    def _shape_of(self, ticket):
        if ticket is None:
            return self._last
        if ticket not in (self.__dict__.get("_shapes") or {}):
            raise nat.B200PoseError("ticket %r is not one of the last two runs" % (ticket,))
        return self._shapes[ticket]

    @classmethod
    def from_net(cls, net, mode="bf16", batch_cap=32, peak_cap=1024, human_cap=1024):
        """An engine around an existing NativeNet (e.g. the one a get_model() module already packed its weights into)."""
        return cls(None, net.device_index, mode, batch_cap, peak_cap, human_cap, net=net)

    def submit_images(self, images, dest_size=368, factor=8, thresh=0.1, flip=False):
        """Asynchronous half of infer_images for frames of ONE shape (a video stream): returns a ticket; the frames must
        stay alive until fetch(ticket=...).  Two submissions may be in flight."""
        batch = np.ascontiguousarray(np.stack(images))
        if batch.dtype != np.uint8 or batch.ndim != 4 or batch.shape[3] != 3:
            raise nat.B200PoseError("submit_images: expected uint8 [h,w,3] frames of one shape")
        if len(batch) > self.post.batch_cap:
            raise nat.B200PoseError("submit_images: %d frames exceed batch_cap %d" % (len(batch), self.post.batch_cap))
        t = self.infer_raw_async_u8(batch.ctypes.data, False, len(batch), batch.shape[1], batch.shape[2], dest_size, factor,
                                    thresh, flip)
        if self.__dict__.get("_alive") is None:
            self._alive = {}
        self._alive[t] = batch                      # host staging is read asynchronously: keep it until the fetch
        for old in [k for k in self._alive if k < t - 1]:
            del self._alive[old]
        return t

    def infer_async(self, in_ptr, in_on_device, n, H, W, thresh=0.1, stream=0):
        nat.check(nat.lib().b200pose_infer(self.net._h, self.post._h, ctypes.c_void_p(in_ptr), int(in_on_device), n, H, W,
                                           self.mode, ctypes.c_float(thresh), ctypes.c_void_p(stream)), "b200pose_infer")
        return self._remember(n, H, W)

    def infer_async_u8(self, in_ptr, in_on_device, n, H, W, thresh=0.1, stream=0):
        """uint8 HWC BGR frames [n,H,W,3] (host pinned or device); preprocessing runs on the device."""
        nat.check(nat.lib().b200pose_infer_u8(self.net._h, self.post._h, ctypes.c_void_p(in_ptr), int(in_on_device), n, H,
                                              W, self.mode, ctypes.c_float(thresh), ctypes.c_void_p(stream)),
                  "b200pose_infer_u8")
        return self._remember(n, H, W)

    def infer_flip_async(self, in_ptr, in_on_device, n, H, W, thresh=0.1, stream=0):
        """Flip test-time averaging (fp32 NCHW input): frames + device-made mirrored copies as one 2n batch, maps merged
        as handle_paf_and_heat does, post-processing on the averaged maps."""
        nat.check(nat.lib().b200pose_infer_flip(self.net._h, self.post._h, ctypes.c_void_p(in_ptr), int(in_on_device), n,
                                                H, W, self.mode, ctypes.c_float(thresh), ctypes.c_void_p(stream)),
                  "b200pose_infer_flip")
        return self._remember(n, H, W)

    def infer_flip_async_u8(self, in_ptr, in_on_device, n, H, W, thresh=0.1, stream=0):
        nat.check(nat.lib().b200pose_infer_u8_flip(self.net._h, self.post._h, ctypes.c_void_p(in_ptr), int(in_on_device),
                                                   n, H, W, self.mode, ctypes.c_float(thresh), ctypes.c_void_p(stream)),
                  "b200pose_infer_u8_flip")
        return self._remember(n, H, W)

    def infer_raw_async_u8(self, in_ptr, in_on_device, n, src_h, src_w, dest_size=368, factor=8, thresh=0.1, flip=False,
                           stream=0):
        """Raw uint8 BGR frames of one size [n,src_h,src_w,3]: crop_with_factor (resize + pad), the network and the
        post-processing all run on the device.  Person coordinates refer to the padded frame."""
        nat.check(nat.lib().b200pose_infer_raw_u8(self.net._h, self.post._h, ctypes.c_void_p(in_ptr), int(in_on_device), n,
                                                  src_h, src_w, int(dest_size), int(factor), self.mode,
                                                  ctypes.c_float(thresh), int(bool(flip)), ctypes.c_void_p(stream)),
                  "b200pose_infer_raw_u8")
        _, _, (ph, pw) = nat.crop_geometry(src_h, src_w, dest_size, factor)
        return self._remember(n, ph, pw)

    def infer_raw_ragged_async_u8(self, frames, dest_size=368, factor=8, thresh=0.1, stream=0):
        """Raw uint8 BGR frames of DIFFERENT sizes (a list of [h,w,3] arrays, at most batch_cap): every frame gets its own
        crop_with_factor, then all of them run through the network and the post-processing as one batch (a canvas of the
        largest padded height x width).  Returns a ticket; per frame the person rows equal infer_raw_async_u8 of that frame
        alone, coordinates in pixels of its own padded frame."""
        frames = [np.ascontiguousarray(f) for f in frames]
        if not frames:
            raise nat.B200PoseError("infer_raw_ragged_async_u8: no frames")
        for f in frames:
            if f.dtype != np.uint8 or f.ndim != 3 or f.shape[2] != 3:
                raise nat.B200PoseError("infer_raw_ragged_async_u8: expected uint8 [h,w,3] frames")
        n = len(frames)
        packed = np.concatenate([f.reshape(-1) for f in frames])
        sh = (ctypes.c_int * n)(*[f.shape[0] for f in frames])
        sw = (ctypes.c_int * n)(*[f.shape[1] for f in frames])
        nat.check(nat.lib().b200pose_infer_raw_u8_ragged(self.net._h, self.post._h, ctypes.c_void_p(packed.ctypes.data), 0,
                                                         n, sh, sw, int(dest_size), int(factor), self.mode,
                                                         ctypes.c_float(thresh), ctypes.c_void_p(stream)),
                  "b200pose_infer_raw_u8_ragged")
        _, pads, _ = nat.ragged_layout([f.shape[:2] for f in frames], dest_size, factor)
        t = self._remember(n, tuple(p[0] for p in pads), tuple(p[1] for p in pads))
        if self.__dict__.get("_alive") is None:
            self._alive = {}
        self._alive[t] = packed                     # host staging is read asynchronously: keep it until the fetch
        for old in [k for k in self._alive if k < t - 1]:
            del self._alive[old]
        return t

    def infer_raw_multiscale_async_u8(self, in_ptr, in_on_device, n, src_h, src_w, scales, base_size=368, factor=8,
                                      thresh=0.1, flip=False, stream=0):
        """Multi-scale (+ flip) test-time averaging of raw uint8 BGR frames of one size (BASELINE.json configs[4]):
        every scale s runs crop_with_factor(int(base_size * s)) + the network on the device, the maps are resized
        (bicubic) to the grid of base_size, averaged, and post-processed.  Coordinates refer to the padded base frame."""
        arr = (ctypes.c_double * len(scales))(*[float(s) for s in scales])
        nat.check(nat.lib().b200pose_infer_raw_u8_multiscale(self.net._h, self.post._h, ctypes.c_void_p(in_ptr),
                                                             int(in_on_device), n, src_h, src_w, int(base_size),
                                                             int(factor), arr, len(scales), self.mode,
                                                             ctypes.c_float(thresh), int(bool(flip)),
                                                             ctypes.c_void_p(stream)),
                  "b200pose_infer_raw_u8_multiscale")
        _, _, (ph, pw) = nat.crop_geometry(src_h, src_w, base_size, factor)
        return self._remember(n, ph, pw)

    def infer_images_arrays(self, images, dest_size=368, factor=8, thresh=0.1, flip=False, scales=None, ragged=False):
        """infer_images, but per image the raw person rows (float32 [k, 73], pixel coordinates of the padded frame)."""
        return self.infer_images(images, dest_size, factor, thresh, flip, scales, ragged, _arrays=True)

    def infer_images(self, images, dest_size=368, factor=8, thresh=0.1, flip=False, scales=None, ragged=False,
                     _arrays=False):
        """images: a list of raw uint8 BGR frames of arbitrary (mixed) sizes, as cv2.imread returns them.  Frames are
        bucketed by shape (one launch sequence per bucket, at most batch_cap frames each); returns per-image human lists
        in input order, coordinates normalised to the padded frame like paf_to_pose_cpp's.
        scales: e.g. (0.5, 1.0, 1.5, 2.0) for multi-scale test-time averaging around dest_size.
        ragged=True: frames of different sizes share runs (ragged_groups: by orientation and padded long side, up to
        batch_cap frames each; the next run is submitted before the previous one is fetched) - same results as the
        bucketed path, fewer and fuller batches on photo collections.  Not combined with flip or scales."""
        if ragged and (flip or scales is not None):
            raise nat.B200PoseError("infer_images: ragged=True does not combine with flip or scales")
        buckets = {}
        for i, im in enumerate(images):
            if im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3:
                raise nat.B200PoseError("infer_images: expected uint8 [h,w,3] frames")
            buckets.setdefault(im.shape[:2], []).append(i)
        out = [None] * len(images)
        if ragged and images:
            _, pads, _ = nat.ragged_layout([im.shape[:2] for im in images], dest_size, factor)
            pending = None
            for part, _ in ragged_groups(pads, self.post.batch_cap) + [(None, None)]:
                t = None if part is None else self.infer_raw_ragged_async_u8([images[i] for i in part], dest_size, factor,
                                                                              thresh)
                if pending is not None:
                    pt, pidx = pending
                    res = self.fetch_arrays(ticket=pt) if _arrays else self.fetch(ticket=pt)
                    for i, humans in zip(pidx, res):
                        out[i] = humans.copy() if _arrays else humans
                pending = None if part is None else (t, part)
            return out
        for (sh, sw), idx in buckets.items():
            for k in range(0, len(idx), self.post.batch_cap):
                part = idx[k:k + self.post.batch_cap]
                batch = np.ascontiguousarray(np.stack([images[i] for i in part]))
                self._keep = batch
                if scales is None:
                    self.infer_raw_async_u8(batch.ctypes.data, False, len(part), sh, sw, dest_size, factor, thresh, flip)
                else:
                    self.infer_raw_multiscale_async_u8(batch.ctypes.data, False, len(part), sh, sw, scales, dest_size,
                                                       factor, thresh, flip)
                for i, humans in zip(part, self.fetch_arrays() if _arrays else self.fetch()):
                    out[i] = humans.copy() if _arrays else humans
        return out

    def fetch(self, check=True, ticket=None):
        """Results of run `ticket` (default: the latest).  Up to two runs may be in flight: submit i+1, then fetch i."""
        n, H, W = self._shape_of(ticket)
        if ticket is None:
            self.post.sync()
        else:
            self.post.select(ticket)
        if check:
            self.post.check_status(n)
        return [humans_to_dicts(self.post.humans(i), _of_image(W, i), _of_image(H, i)) for i in range(n)]

    def fetch_arrays(self, check=True, ticket=None):
        """Like fetch() but without building Python objects: per image a float32 array [k, 73] with rows
        (score, 18 x (x, y, peak score, peak id | -1)), x / y in pixels of the (padded) network input."""
        n, H, W = self._shape_of(ticket)
        if ticket is None:
            self.post.sync()
        else:
            self.post.select(ticket)
        if check:
            self.post.check_status(n)
        return [self.post.humans(i) for i in range(n)]

    def infer_batch(self, images, thresh=0.1, flip=False):
        """images: uint8 numpy [n,H,W,3] (BGR frames, preprocessing fused on the device), float32 numpy [n,3,H,W]
        (already preprocessed, host) or a CUDA float tensor.  Returns per-image human lists.
        flip=True: left/right flip test-time averaging on the device (handle_paf_and_heat semantics)."""
        run_u8 = self.infer_flip_async_u8 if flip else self.infer_async_u8
        run_f32 = self.infer_flip_async if flip else self.infer_async
        if isinstance(images, np.ndarray) and images.dtype == np.uint8:
            images = np.ascontiguousarray(images)
            n, H, W, _ = images.shape          # [n,H,W,3] BGR, already cropped/padded to multiples of 8
            self._keep = images
            run_u8(images.ctypes.data, False, n, H, W, thresh)
        elif isinstance(images, np.ndarray):
            images = np.ascontiguousarray(images, dtype=np.float32)
            n, _, H, W = images.shape
            self._keep = images
            run_f32(images.ctypes.data, False, n, H, W, thresh)
        else:
            import torch
            if not images.is_cuda:
                raise nat.B200PoseError("torch inputs must live on the GPU (no CPU fallback)")
            images = images.contiguous().float()
            n, _, H, W = images.shape
            self._keep = images
            run_f32(images.data_ptr(), True, n, H, W, thresh, torch.cuda.current_stream().cuda_stream)
        return self.fetch()
