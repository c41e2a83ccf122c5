"""Drop-in replacement for the reference package ``diff_gaussian_rasterization``.

Same public surface as ``sugar/gaussian_splatting/submodules/diff-gaussian-rasterization/
diff_gaussian_rasterization/__init__.py`` (reference lines in brackets):

* ``GaussianRasterizationSettings``  NamedTuple, 12 fields                        [:160-172]
* ``GaussianRasterizer(nn.Module)``  ``.forward(...)`` -> (color, depth, alpha, radii), ``.markVisible``  [:174-223]
* ``rasterize_gaussians(...)`` and ``_RasterizeGaussians`` (autograd.Function)     [:21-158]

and, beyond the reference's surface, ``rasterize_gaussians_multi`` (``_RasterizeGaussiansMulti``): the two rasterizer calls of
one training frame (SH colours, then a second colour set on the same geometry) as one autograd call with one forward and one
backward pass.

Host code stays Python/PyTorch; all device work happens in the hand-written sm_100a library behind the C ABI
of ``include/gsr_b200.h`` (loaded through ctypes by ``_lib``).  PyTorch only provides memory (the caching
allocator), the current stream and autograd plumbing.  There is no CPU path.

Differences a caller can observe:
* kernels run on PyTorch's *current* stream and on ``means3D``'s device (the reference uses the legacy default
  stream and the current device, rasterize_points.cu:73);
* the three opaque buffers saved for backward have a different (smaller) layout;
* by default one event synchronisation per forward remains (the reference blocks on a cudaMemcpy,
  rasterizer_impl.cu:281-282); ``set_sync_mode("async")`` removes it (see ``FrameTicket``).
"""
from __future__ import annotations

import collections
import ctypes as C
import weakref
from typing import Dict, NamedTuple, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib
from ._lib import lib as _L

__all__ = ["GaussianRasterizationSettings", "GaussianRasterizer", "rasterize_gaussians", "set_sync_mode", "get_sync_mode",
           "set_tight_tiles", "get_tight_tiles", "set_geometry_reuse", "set_exact_images", "get_exact_images",
           "last_frame_stats", "FrameTicket", "forward_raw", "forward_multi", "PreparedForward", "debug_views",
           "invalidate_geometry_cache", "rasterize_gaussians_multi"]


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


# ----------------------------------------------------------------------------------------------- engine state
_SYNC_MODE = "safe"


def set_sync_mode(mode: str) -> None:
    """"safe": every forward validates the binning capacity before returning (one event sync, automatic
    re-run on overflow).  "async": no host synchronisation at all; each forward returns immediately and its
    ``FrameTicket`` (``last_ticket()``) must be validated by the caller before the images are trusted."""
    global _SYNC_MODE
    if mode not in ("safe", "async"):
        raise ValueError("sync mode must be 'safe' or 'async'")
    _SYNC_MODE = mode


def get_sync_mode() -> str:
    return _SYNC_MODE


_TIGHT_TILES = False
_REUSE_GEOMETRY = True
_EXACT_IMAGES = False


def set_exact_images(on: bool) -> None:
    """Default off.  On: the blend uses the reference's own fp32 instruction sequence (GSR_FLAG_EXACT_IMAGES) and
    color / depth / alpha are bit-identical to the reference's CUDA rasterizer.  Off: alpha = ex2.approx(power*log2e +
    log2(opacity)); every skip / termination decision inside the approximation's error band is re-done exactly, so the
    images differ from the exact ones by ~1e-6 relative (the requirement is 1e-4 max abs) and radii / per-tile lists /
    n_contrib are unchanged."""
    global _EXACT_IMAGES
    _EXACT_IMAGES = bool(on)


def get_exact_images() -> bool:
    return _EXACT_IMAGES



def set_geometry_reuse(on: bool) -> None:
    """The product frame calls the rasterizer twice per camera with identical geometry (SH pass, then
    ``colors_precomp`` = normals; reference gaussian_renderer/__init__.py:151-185).  When enabled (default) a
    ``colors_precomp`` forward under ``torch.no_grad()`` whose geometry tensors, camera and settings are the very same
    (same storage, same version counters) as the previous forward on that stream skips projection, binning and sorting
    and only re-blends (GSR_FLAG_REUSE_GEOMETRY).  Outputs are bit-identical to a full forward."""
    global _REUSE_GEOMETRY
    _REUSE_GEOMETRY = bool(on)


def set_tight_tiles(on: bool) -> None:
    """Opt-in (default off): only emit a (Gaussian, tile) instance if the splat can reach alpha >= 1/255 at a pixel of the
    tile (GSR_FLAG_TIGHT_TILES).  color / depth / alpha / radii and all gradients are bit-for-bit unchanged; the opaque
    per-tile lists become sub-sequences of the reference's, so fewer instances are sorted and staged."""
    global _TIGHT_TILES
    _TIGHT_TILES = bool(on)


def get_tight_tiles() -> bool:
    return _TIGHT_TILES


class FrameTicket:
    """Handle on the device-side counters of one forward call (gsr_counters, include/gsr_b200.h)."""

    __slots__ = ("event", "slot", "capacity", "_state", "_snap", "__weakref__")

    def __init__(self, event, slot, capacity, state):
        self.event, self.slot, self.capacity, self._state = event, slot, capacity, state
        self._snap = None

    def ready(self) -> bool:
        return self.event.query()

    def snapshot(self) -> None:
        """Copy the counters out of the shared pinned ring slot (called on first use, and by the ring before it recycles
        the slot, so a ticket held across more than RING later forwards still reads its own frame)."""
        if self._snap is None:
            self.event.synchronize()
            self._snap = [int(x) for x in self.slot.tolist()]

    def stats(self) -> Dict[str, int]:
        """Blocks until the frame's counters have reached the host."""
        self.snapshot()
        c = self._snap
        return {"num_rendered": int(c[0]), "overflow": int(c[1]), "max_tile": int(c[2]), "trapped": int(c[3]),
                "num_visible": int(c[4]), "foot_total": int(c[5]) & 0xffffffff, "exact_redos": int(c[6]),
                "capacity": int(self.capacity)}

    def ok(self) -> bool:
        s = self.stats()
        if s["overflow"]:
            self._state.grow(needed_capacity(s))
        return not s["overflow"]


def needed_capacity(stats: Dict[str, int]) -> int:
    """Binning capacity (instances) a frame with these counters needs."""
    return int(stats["num_rendered"])


class _DeviceState:
    RING = 64

    def __init__(self, device: torch.device):
        self.device = device
        self.capacity = 1 << 20
        self.pinned = torch.zeros((self.RING, 8), dtype=torch.int32).pin_memory()
        self.events = [None] * self.RING
        self.tickets = [None] * self.RING  # weak references to the ticket reading each slot
        self.cursor = 0
        self.cache: Dict[Tuple, torch.Tensor] = {}
        self.last_ticket: Optional[FrameTicket] = None
        self.side_stream: Optional[torch.cuda.Stream] = None
        # geometry of the last full (non-autograd) forward per stream: (key, tensors kept alive, radii)
        self.geom_cache: Dict[int, Tuple] = {}

    def grow(self, needed: int) -> None:
        self.capacity = max(self.capacity, int(needed * 1.25) + 4096)

    def ensure_capacity(self, P: int, W: int = 0, H: int = 0) -> None:
        # first guess: a few instances per Gaussian; corrected from the counters of real frames
        if self.capacity < 4 * P:
            self.capacity = 4 * P
        # the binning workspace also holds the footprint ballot matrix: capacity / 32 + 131072 rows, one per 32 list entries + one per tile
        tiles = ((W + 15) // 16) * ((H + 15) // 16)
        if tiles > 131072 and self.capacity < 32 * (tiles - 131072) + 64:
            self.capacity = 32 * (tiles - 131072) + 64

    def next_slot(self):
        i = self.cursor
        self.cursor = (i + 1) % self.RING
        ev = self.events[i]
        if ev is not None:
            ev.synchronize()  # the slot is only reused once its previous copy has landed
            old = self.tickets[i]() if self.tickets[i] is not None else None
            if old is not None:
                old.snapshot()  # a ticket still alive keeps its own counters
        ev = torch.cuda.Event()
        self.events[i] = ev
        return self.pinned[i], ev

    def issue_ticket(self, counters: torch.Tensor, stream, capacity: int, early: bool = False) -> "FrameTicket":
        """Async copy of a frame's 32-byte counters into the next pinned ring slot + the event that says it has landed.
        ``early``: the copy runs on a side stream that only waits for what ``stream`` holds right now, so it neither waits for
        nor delays the work enqueued on ``stream`` afterwards (the safe mode's capacity check between the two halves of a frame)."""
        i = self.cursor
        slot, ev = self.next_slot()
        if early:
            if self.side_stream is None:
                self.side_stream = torch.cuda.Stream(self.device)
            mark = torch.cuda.Event()
            mark.record(stream)
            self.side_stream.wait_event(mark)
            with torch.cuda.stream(self.side_stream):
                slot.copy_(counters, non_blocking=True)
            ev.record(self.side_stream)
        else:
            slot.copy_(counters, non_blocking=True)
            ev.record(stream)
        ticket = FrameTicket(ev, slot, capacity, self)
        self.tickets[i] = weakref.ref(ticket)
        self.last_ticket = ticket
        return ticket

    def workspace(self, kind: str, nbytes: int, fresh: bool) -> torch.Tensor:
        if fresh:
            return torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        key = (kind, torch.cuda.current_stream(self.device).cuda_stream)
        t = self.cache.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(int(nbytes * 1.1) + 256, dtype=torch.uint8, device=self.device)
            self.cache[key] = t
        return t


_STATES: Dict[int, _DeviceState] = {}


def _state(device: torch.device) -> _DeviceState:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    st = _STATES.get(idx)
    if st is None:
        st = _DeviceState(torch.device("cuda", idx))
        _STATES[idx] = st
    return st


def invalidate_geometry_cache(device=None) -> None:
    """Forget which geometry the cached workspaces hold.  Called by code that rewrites parameter tensors in place through
    raw pointers (``edit.activate_into``): such writes do not bump the tensors' version counters, which the automatic
    second-pass reuse (``set_geometry_reuse``) relies on."""
    if device is None:
        for st in _STATES.values():
            st.geom_cache.clear()
        return
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx in _STATES:
        _STATES[idx].geom_cache.clear()


def last_ticket(device=None) -> Optional[FrameTicket]:
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    return _state(dev).last_ticket


def last_frame_stats(device=None) -> Dict[str, int]:
    """num_rendered (R), num_visible (P_vis), max_tile ... of the most recent forward on ``device``."""
    t = last_ticket(device)
    if t is None:
        raise RuntimeError("no frame has been rasterized on this device yet")
    return t.stats()


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None or t.numel() == 0:
        return None
    return t.data_ptr()


def _dev_f32(t: torch.Tensor, device: torch.device) -> torch.Tensor:
    if t.device != device:
        t = t.to(device, non_blocking=True)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _opt(t: Optional[torch.Tensor], device: torch.device) -> Optional[torch.Tensor]:
    if t is None or t.numel() == 0:
        return None
    return _dev_f32(t, device)


def _fill_frame(fr: _lib.gsr_frame, P, D, M, W, H, settings, bg, means3D, shs, colors_precomp, opacities, scales, rotations, cov3D,
                view, proj, campos):
    fr.P, fr.D, fr.M, fr.W, fr.H = P, D, M, W, H
    fr.scale_modifier = settings.scale_modifier
    fr.tanfovx, fr.tanfovy = settings.tanfovx, settings.tanfovy
    fr.prefiltered, fr.debug = int(bool(settings.prefiltered)), int(bool(settings.debug))
    fr.bg, fr.means3D, fr.shs, fr.colors_precomp = _ptr(bg), _ptr(means3D), _ptr(shs), _ptr(colors_precomp)
    fr.opacities, fr.scales, fr.rotations, fr.cov3D_precomp = _ptr(opacities), _ptr(scales), _ptr(rotations), _ptr(cov3D)
    fr.viewmatrix, fr.projmatrix, fr.campos = _ptr(view), _ptr(proj), _ptr(campos)


def forward_raw(means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, settings: GaussianRasterizationSettings,
                for_backward: bool = False, sorted_keys: bool = False, sync: Optional[bool] = None, out=None,
                tight: Optional[bool] = None, extra: Optional[torch.Tensor] = None, extra_out: Optional[torch.Tensor] = None,
                exact: Optional[bool] = None):
    """One rasterizer forward through the C ABI.  Returns (color, depth, alpha, radii, workspaces, ticket, keepalive).
    ``workspaces`` = (geom, binning, image) byte tensors; fresh allocations when ``for_backward`` (they must outlive
    the call), otherwise per-(device, stream) cached buffers.  ``out`` optionally supplies preallocated
    (color, depth, alpha, radii) tensors (used by the frame loop to render straight into its ring).  ``extra`` ([P,3]
    colours) + ``extra_out`` ([3,H,W]) blend a second colour set in the same pass (gsr_forward_multi, see ``forward_multi``)."""
    if (extra is None) != (extra_out is None):
        raise ValueError("extra and extra_out go together")
    if means3D.dim() != 2 or means3D.size(1) != 3:
        raise RuntimeError("means3D must have dimensions (num_points, 3)")  # rasterize_points.cu:57-59
    if not means3D.is_cuda:
        raise RuntimeError("autovfx_b200 rasterizer: means3D must be a CUDA tensor (there is no CPU path)")
    device = means3D.device
    st = _state(device)
    P = means3D.size(0)
    H, W = int(settings.image_height), int(settings.image_width)
    with torch.cuda.device(device):
        means3D = _dev_f32(means3D, device)
        shs, colors_precomp = _opt(shs, device), _opt(colors_precomp, device)
        scales, rotations, cov3D_precomp = _opt(scales, device), _opt(rotations, device), _opt(cov3D_precomp, device)
        opacities = _dev_f32(opacities, device)
        if extra is not None:
            extra = _dev_f32(extra, device)
            if extra.shape != (P, 3) or extra_out.shape != (3, H, W) or extra_out.dtype != torch.float32 or not extra_out.is_contiguous():
                raise ValueError("extra must be [P,3] and extra_out a contiguous float32 [3,H,W]")
        bg = _dev_f32(settings.bg, device)
        view = _dev_f32(settings.viewmatrix, device)
        proj = _dev_f32(settings.projmatrix, device)
        campos = _dev_f32(settings.campos, device)
        M = shs.size(1) if shs is not None else 0
        if out is None:
            color = torch.empty((3, H, W), dtype=torch.float32, device=device)
            depth = torch.empty((1, H, W), dtype=torch.float32, device=device)
            alpha = torch.empty((1, H, W), dtype=torch.float32, device=device)
            radii = torch.empty((P,), dtype=torch.int32, device=device)
        else:
            color, depth, alpha, radii = out
        flags = (_lib.GSR_FLAG_FOR_BACKWARD if for_backward else 0) | (_lib.GSR_FLAG_SORTED_KEYS if sorted_keys else 0)
        if _TIGHT_TILES if tight is None else tight:
            flags |= _lib.GSR_FLAG_TIGHT_TILES
        use_exact = _EXACT_IMAGES if exact is None else bool(exact)
        if use_exact:
            flags |= _lib.GSR_FLAG_EXACT_IMAGES
        fr = _lib.gsr_frame()
        _fill_frame(fr, P, int(settings.sh_degree), M, W, H, settings, bg, means3D, shs, colors_precomp, opacities, scales, rotations,
                    cov3D_precomp, view, proj, campos)
        geom_b, img_b = _L.gsr_geom_bytes(P), _L.gsr_image_bytes(W, H)
        geom = st.workspace("geom", geom_b, for_backward)
        image = st.workspace("image", img_b, for_backward)
        st.ensure_capacity(P, W, H)
        do_sync = (_SYNC_MODE == "safe") if sync is None else sync
        stream = torch.cuda.current_stream(device)
        use_tight = _TIGHT_TILES if tight is None else tight

        def tk(t):
            return None if t is None else (t.data_ptr(), t._version, tuple(t.shape))
        gkey = (tk(means3D), tk(opacities), tk(scales), tk(rotations), tk(cov3D_precomp), tk(view), tk(proj), tk(campos), W, H,
                float(settings.tanfovx), float(settings.tanfovy), float(settings.scale_modifier), bool(settings.prefiltered),
                bool(use_tight), bool(use_exact), geom.data_ptr(), image.data_ptr())
        cached = st.geom_cache.get(stream.cuda_stream)
        if (_REUSE_GEOMETRY and not for_backward and not sorted_keys and colors_precomp is not None and P > 0 and cached is not None
                and cached[0] == gkey):
            # second pass over the same geometry: recolour + blend only
            _, _, radii_prev, binning = cached
            ws = _lib.gsr_workspace(geom.data_ptr(), geom.numel(), binning.data_ptr(), binning.numel(), image.data_ptr(), image.numel())
            rc = _L.gsr_forward_multi(C.byref(fr), C.byref(ws), color.data_ptr(), depth.data_ptr(), alpha.data_ptr(), radii_prev.data_ptr(),
                                      _ptr(extra) if P > 0 else None, _ptr(extra_out) if extra is not None and P > 0 else None,
                                      flags | _lib.GSR_FLAG_REUSE_GEOMETRY, C.c_void_p(stream.cuda_stream))
            _lib.check(rc, "gsr_forward(reuse)")
            if out is None:
                radii = radii_prev.clone()
            elif radii.data_ptr() != radii_prev.data_ptr():
                radii.copy_(radii_prev)
            ticket = st.issue_ticket(image[:32].view(torch.int32), stream, _L.gsr_binning_capacity(binning.numel()))
            if do_sync and ticket.stats()["overflow"]:
                raise RuntimeError("autovfx_b200: reused geometry pass found an overflowed first pass")
            keep = (means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, bg, view, proj, campos, extra)
            return color, depth, alpha, radii, (geom, binning, image), ticket, keep
        if not for_backward:
            st.geom_cache.pop(stream.cuda_stream, None)  # the shared workspaces are about to be rewritten (also by a P == 0 call)
        while True:
            cap = st.capacity
            binning = st.workspace("binning", _L.gsr_binning_bytes(cap), for_backward)
            ws = _lib.gsr_workspace(geom.data_ptr(), geom.numel(), binning.data_ptr(), binning.numel(), image.data_ptr(), image.numel())
            if extra is not None and P == 0:
                extra_out.zero_()
            args = (C.byref(fr), C.byref(ws), color.data_ptr(), depth.data_ptr(), alpha.data_ptr(), radii.data_ptr() if P > 0 else None,
                    _ptr(extra) if P > 0 else None, _ptr(extra_out) if extra is not None and P > 0 else None)
            cap_now = _L.gsr_binning_capacity(binning.numel())
            if do_sync and P > 0 and not settings.debug:
                # safe mode: the frame is issued in two halves; the counters are final after the first (projection + tile scan), so
                # the host waits for THAT copy while colour / emission / sort / blend are already queued behind it
                _lib.check(_L.gsr_forward_multi(*args, flags | _lib.GSR_FLAG_BINNING_ONLY, C.c_void_p(stream.cuda_stream)), "gsr_forward")
                check = st.issue_ticket(image[:32].view(torch.int32), stream, cap_now, early=True)
                _lib.check(_L.gsr_forward_multi(*args, flags | _lib.GSR_FLAG_RESUME, C.c_void_p(stream.cuda_stream)), "gsr_forward")
                ticket = st.issue_ticket(image[:32].view(torch.int32), stream, cap_now)  # the frame's final counters (exact_redos)
            else:
                _lib.check(_L.gsr_forward_multi(*args, flags, C.c_void_p(stream.cuda_stream)), "gsr_forward")
                check = ticket = st.issue_ticket(image[:32].view(torch.int32), stream, cap_now)
            if not do_sync:
                break
            s = check.stats()
            if s["trapped"]:
                raise RuntimeError("Point is filtered although prefiltered is set. This shouldn't happen!")  # auxiliary.h:158
            if not s["overflow"]:
                break
            st.grow(needed_capacity(s))  # rare: first frames of a new scene; re-run with a larger binning buffer
        if not for_backward and P > 0:
            # remember which geometry the shared workspaces now hold (tensors kept alive so their storage cannot be recycled)
            st.geom_cache[stream.cuda_stream] = (gkey, (means3D, opacities, scales, rotations, cov3D_precomp, view, proj, campos), radii, binning)
    keep = (means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, bg, view, proj, campos, extra)
    return color, depth, alpha, radii, (geom, binning, image), ticket, keep


def forward_multi(means3D, shs, colors_precomp, extra_colors, opacities, scales, rotations, cov3D_precomp,
                  settings: GaussianRasterizationSettings, sync: Optional[bool] = None, out=None, extra_out=None,
                  tight: Optional[bool] = None, exact: Optional[bool] = None):
    """Both rasterizer passes of one product frame in ONE pass (forward only): ``(color, depth, alpha, extra_image, radii,
    ticket)`` where ``extra_image`` [3,H,W] is bit-identical to the colour image a second
    ``GaussianRasterizer(...)(colors_precomp=extra_colors, ...)`` call would return
    (reference: gaussian_renderer/__init__.py:134-166 runs the whole pipeline twice)."""
    H, W = int(settings.image_height), int(settings.image_width)
    if extra_out is None:
        extra_out = torch.empty((3, H, W), dtype=torch.float32, device=means3D.device)
    color, depth, alpha, radii, _ws, ticket, _keep = forward_raw(means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp,
                                                               settings, sync=sync, out=out, tight=tight, extra=extra_colors,
                                                               extra_out=extra_out, exact=exact)
    return color, depth, alpha, extra_out, radii, ticket


class PreparedForward:
    """A forward call with everything resolved ahead of time — parameter tensors, the device-resident camera row the caller
    overwrites per frame, outputs, workspaces, flags — so that issuing a frame costs one C call, one 32-byte counters copy and
    an event (a few microseconds of host time instead of the ~0.3 ms of argument checking in ``forward_raw``).  Used by
    ``render_loop.FrameLoop``; forward-only (no buffers are kept for a backward pass).

    ``cam`` is a contiguous float32 device tensor holding view(16) | proj(16) | campos(3) at its start."""

    def __init__(self, means3D, shs, opacities, scales, rotations, cam: torch.Tensor, W: int, H: int, bg: torch.Tensor, sh_degree: int,
                 scale_modifier: float, out, extra: Optional[torch.Tensor] = None, extra_out: Optional[torch.Tensor] = None,
                 tight: Optional[bool] = None, exact: Optional[bool] = None):
        device = means3D.device
        self.device, self.st = device, _state(device)
        self.P, self.W, self.H = int(means3D.shape[0]), int(W), int(H)
        chk = [means3D, shs, opacities, scales, rotations, cam, bg] + list(out) + ([extra, extra_out] if extra is not None else [])
        for t in chk:
            if not (t.is_cuda and t.device == device and t.is_contiguous()):
                raise ValueError("PreparedForward: tensors must be contiguous and live on %s" % device)
        for t in (means3D, shs, opacities, scales, rotations, cam, bg):
            if t.dtype != torch.float32:
                raise ValueError("PreparedForward: float32 tensors required")
        if (extra is None) != (extra_out is None):
            raise ValueError("extra and extra_out go together")
        self.keep = (means3D, shs, opacities, scales, rotations, cam, bg, out, extra, extra_out)
        color, depth, alpha, radii = out
        self.fr = _lib.gsr_frame()
        fr = self.fr
        fr.P, fr.D, fr.M, fr.W, fr.H = self.P, int(sh_degree), int(shs.shape[1]), self.W, self.H
        fr.scale_modifier = float(scale_modifier)
        fr.prefiltered, fr.debug = 0, 0
        fr.bg, fr.means3D, fr.shs, fr.colors_precomp = bg.data_ptr(), _ptr(means3D), _ptr(shs), None
        fr.opacities, fr.scales, fr.rotations, fr.cov3D_precomp = _ptr(opacities), _ptr(scales), _ptr(rotations), None
        base = cam.data_ptr()
        fr.viewmatrix, fr.projmatrix, fr.campos = base, base + 64, base + 128
        self.out_ptrs = (color.data_ptr(), depth.data_ptr(), alpha.data_ptr(), radii.data_ptr() if self.P > 0 else None)
        self.extra_ptrs = (_ptr(extra) if self.P > 0 else None, _ptr(extra_out) if extra is not None and self.P > 0 else None)
        self.extra_out = extra_out
        self.flags = _lib.GSR_FLAG_TIGHT_TILES if (_TIGHT_TILES if tight is None else tight) else 0
        if _EXACT_IMAGES if exact is None else exact:
            self.flags |= _lib.GSR_FLAG_EXACT_IMAGES
        self._cap = -1
        self.ws = None
        self._bufs = None

    def _bind_workspaces(self) -> None:
        st = self.st
        with torch.cuda.device(self.device):
            geom = st.workspace("geom", _L.gsr_geom_bytes(self.P), False)
            image = st.workspace("image", _L.gsr_image_bytes(self.W, self.H), False)
            st.ensure_capacity(self.P, self.W, self.H)
            binning = st.workspace("binning", _L.gsr_binning_bytes(st.capacity), False)
        self._bufs = (geom, binning, image)
        self._key = (geom.data_ptr(), geom.numel(), binning.data_ptr(), binning.numel(), image.data_ptr(), image.numel())
        self.ws = _lib.gsr_workspace(*self._key)
        self._cap = st.capacity
        self._counters = image[:32].view(torch.int32)
        self._capacity_instances = _L.gsr_binning_capacity(binning.numel())

    def launch(self, tanfovx: float, tanfovy: float) -> FrameTicket:
        """Issue the frame on the current stream; never synchronises.  Validate the returned ticket before trusting the images."""
        with torch.cuda.device(self.device):
            return self._launch(tanfovx, tanfovy)

    def _launch(self, tanfovx: float, tanfovy: float) -> FrameTicket:
        st = self.st
        stream = torch.cuda.current_stream(self.device)
        if self._cap != st.capacity or self.ws is None:
            self._bind_workspaces()
        else:  # the cached workspaces may have been re-allocated (grown) by another caller on this stream
            g2, b2, i2 = st.cache.get(("geom", stream.cuda_stream)), st.cache.get(("binning", stream.cuda_stream)), st.cache.get(("image", stream.cuda_stream))
            if g2 is not self._bufs[0] or b2 is not self._bufs[1] or i2 is not self._bufs[2]:
                self._bind_workspaces()
        st.geom_cache.pop(stream.cuda_stream, None)  # the shared workspaces are about to hold this frame
        fr = self.fr
        fr.tanfovx, fr.tanfovy = tanfovx, tanfovy
        if self.extra_out is not None and self.P == 0:
            self.extra_out.zero_()
        rc = _L.gsr_forward_multi(C.byref(fr), C.byref(self.ws), self.out_ptrs[0], self.out_ptrs[1], self.out_ptrs[2], self.out_ptrs[3],
                                  self.extra_ptrs[0], self.extra_ptrs[1], self.flags, C.c_void_p(stream.cuda_stream))
        _lib.check(rc, "gsr_forward")
        return st.issue_ticket(self._counters, stream, self._capacity_instances)


def _cpu_copy(items):
    """CPU clones of the tensors in ``items`` (the reference's cpu_deep_copy_tuple, __init__.py:16-18)."""
    return tuple(x.detach().cpu().clone() if isinstance(x, torch.Tensor) else x for x in items)


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings):
    # Whether a backward can follow is decided HERE: inside autograd.Function.forward grad mode is always off, and the
    # reference's eval loops (scene_representation.py:355 render_from_3DGS) pass nn.Parameters under torch.no_grad().
    need_bw = torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in
                                              (means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp))
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings,
                                     need_bw)


def _autograd_forward(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings, need_bw,
                      extra=None, extra_out=None):
    """forward_raw for the autograd front ends, with the reference's debug snapshot.  Returns (color, depth, alpha, radii,
    ticket, tensors to save for backward)."""
    if raster_settings.debug:
        # reference debug behaviour (__init__.py:83-90): keep a CPU copy of the arguments and dump it if the call fails
        cpu_args = _cpu_copy((raster_settings.bg, means3D, colors_precomp, opacities, scales, rotations, raster_settings.scale_modifier,
                              cov3Ds_precomp, raster_settings.viewmatrix, raster_settings.projmatrix, raster_settings.tanfovx,
                              raster_settings.tanfovy, raster_settings.image_height, raster_settings.image_width, sh,
                              raster_settings.sh_degree, raster_settings.campos, raster_settings.prefiltered, raster_settings.debug))
        try:
            res = forward_raw(means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings,
                              for_backward=need_bw, extra=extra, extra_out=extra_out)
        except Exception as ex:
            torch.save(cpu_args, "snapshot_fw.dump")
            print("\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.")
            raise ex
    else:
        res = forward_raw(means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings, for_backward=need_bw,
                          extra=extra, extra_out=extra_out)
    color, depth, alpha, radii, (geom, binning, image), ticket, keep = res
    k_means3D, k_shs, k_colors, _k_op, k_scales, k_rot, k_cov, k_bg, k_view, k_proj, k_campos, _k_extra = keep
    e = torch.empty(0, device=means3D.device)
    saved = (k_colors if k_colors is not None else e, k_means3D, k_scales if k_scales is not None else e,
             k_rot if k_rot is not None else e, k_cov if k_cov is not None else e, radii,
             k_shs if k_shs is not None else e, geom, binning, image, alpha, k_bg, k_view, k_proj, k_campos)
    if extra is not None:
        saved = saved + (_k_extra,)
    return color, depth, alpha, radii, ticket, saved


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings, need_bw=True):
        color, depth, alpha, radii, ticket, saved = _autograd_forward(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                                                      cov3Ds_precomp, raster_settings, need_bw)
        ctx.raster_settings = raster_settings
        ctx.ticket = ticket
        ctx.has = (sh.numel() != 0, colors_precomp.numel() != 0, scales.numel() != 0, cov3Ds_precomp.numel() != 0)
        ctx.needs = need_bw
        ctx.in_shapes = tuple(tuple(t.shape) for t in (means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp))
        ctx.save_for_backward(*saved)
        ctx.mark_non_differentiable(radii)
        return color, depth, alpha, radii

    @staticmethod
    def backward(ctx, grad_out_color, grad_out_depth, grad_out_alpha, _):
        if not ctx.needs:
            return (None,) * 10
        return _autograd_backward(ctx, ctx.saved_tensors, grad_out_color, grad_out_depth, grad_out_alpha) + (None, None)


def _autograd_backward(ctx, saved, grad_out_color, grad_out_depth, grad_out_alpha, extra=None, grad_out_extra=None):
    """gsr_backward (gsr_backward_multi when ``grad_out_extra`` is given) of a forward saved by ``_autograd_forward``.  Returns
    the gradients in the reference's input order: means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
    cov3Ds_precomp, plus dL/dextra_colors last when ``grad_out_extra`` is given."""
    s = ctx.raster_settings
    (colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom, binning, image, alpha, bg, view, proj, campos) = saved[:15]
    if _SYNC_MODE != "safe" and not ctx.ticket.ok():
        raise RuntimeError("autovfx_b200: the forward of this graph overflowed its binning buffer (async mode); re-run it")
    device = means3D.device
    P = means3D.size(0)
    H, W = int(s.image_height), int(s.image_width)
    M = sh.size(1) if sh.numel() else 0
    has_sh, has_col, has_scale, has_cov = ctx.has
    with_extra = grad_out_extra is not None
    if P == 0:  # empty scene: the reference returns empty gradients (rasterize_points.cu:158-168 with P = 0)
        zeros = tuple(torch.zeros(shp, dtype=torch.float32, device=device) for shp in ctx.in_shapes)
        return zeros + ((torch.zeros((0, 3), dtype=torch.float32, device=device),) if with_extra else ())
    with torch.cuda.device(device):
        def img_grad(g, c):
            if g is None:
                return torch.zeros((c, H, W), dtype=torch.float32, device=device)
            return _dev_f32(g, device)
        g_color, g_depth, g_alpha = img_grad(grad_out_color, 3), img_grad(grad_out_depth, 1), img_grad(grad_out_alpha, 1)
        f32 = dict(dtype=torch.float32, device=device)
        dL_dmeans3D = torch.empty((P, 3), **f32)
        dL_dmeans2D = torch.empty((P, 3), **f32)
        dL_dcolors = torch.empty((P, 3), **f32)
        dL_ddepths = torch.empty((P, 1), **f32)
        dL_dconic = torch.empty((P, 2, 2), **f32)
        dL_dopacity = torch.empty((P, 1), **f32)
        dL_dcov3D = torch.empty((P, 6), **f32)
        dL_dsh = torch.empty((P, M, 3), **f32)
        dL_dscales = torch.empty((P, 3), **f32)
        dL_drotations = torch.empty((P, 4), **f32)
        fr = _lib.gsr_frame()
        _fill_frame(fr, P, int(s.sh_degree), M, W, H, s, bg, means3D, sh, colors_precomp, None, scales, rotations, cov3Ds_precomp,
                    view, proj, campos)
        ws = _lib.gsr_workspace(geom.data_ptr(), geom.numel(), binning.data_ptr(), binning.numel(), image.data_ptr(), image.numel())
        gr = _lib.gsr_grads(_ptr(dL_dmeans2D), _ptr(dL_dconic), _ptr(dL_dopacity), _ptr(dL_dcolors), _ptr(dL_ddepths),
                            _ptr(dL_dmeans3D), _ptr(dL_dcov3D), _ptr(dL_dsh), _ptr(dL_dscales), _ptr(dL_drotations))
        stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        if with_extra:
            g_extra = _dev_f32(grad_out_extra, device)
            dL_dextra = torch.empty((P, 3), **f32)
            rc = _L.gsr_backward_multi(C.byref(fr), C.byref(ws), _ptr(radii), _ptr(alpha), _ptr(g_color), _ptr(g_depth), _ptr(g_alpha),
                                       _ptr(extra), _ptr(g_extra), C.byref(gr), _ptr(dL_dextra), stream)
        else:
            rc = _L.gsr_backward(C.byref(fr), C.byref(ws), _ptr(radii), _ptr(alpha), _ptr(g_color), _ptr(g_depth), _ptr(g_alpha),
                                 C.byref(gr), stream)
        if rc != 0 and s.debug:  # reference debug behaviour (__init__.py:135-142)
            torch.save(_cpu_copy((bg, means3D, radii, colors_precomp, scales, rotations, s.scale_modifier, cov3Ds_precomp, view, proj, s.tanfovx,
                                  s.tanfovy, g_color, g_depth, g_alpha, sh, s.sh_degree, campos, alpha, s.debug)), "snapshot_bw.dump")
            print("\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
        _lib.check(rc, "gsr_backward_multi" if with_extra else "gsr_backward")
    # reference order (__init__.py:146-156): means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp
    grads = (dL_dmeans3D, dL_dmeans2D, dL_dsh if has_sh else None, dL_dcolors if has_col else None, dL_dopacity,
             dL_dscales if has_scale else None, dL_drotations if has_scale else None, dL_dcov3D if has_cov else None)
    return grads + ((dL_dextra,) if with_extra else ())


def rasterize_gaussians_multi(means3D, means2D, sh, colors_precomp, extra_colors, opacities, scales, rotations, cov3Ds_precomp,
                              raster_settings):
    """Both rasterizer passes of one training frame in ONE autograd call: ``(color, depth, alpha, extra_image, radii)``, where
    ``extra_image`` [3,H,W] is the colour image a second ``rasterize_gaussians`` call with ``colors_precomp = extra_colors``
    ([P,3]) would return, bit for bit.  Gradients flow to every input, ``extra_colors`` included; they equal the sum of the two
    calls' gradients up to summation order.  One projection, binning, sort and blend forward, one blend backward
    (gsr_backward_multi) and one per-Gaussian backward serve both images.  Absent inputs are None or empty tensors."""
    def opt(t):
        return torch.Tensor([]) if t is None else t
    sh, colors_precomp, scales, rotations, cov3Ds_precomp = opt(sh), opt(colors_precomp), opt(scales), opt(rotations), opt(cov3Ds_precomp)
    need_bw = torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in
                                              (means3D, means2D, sh, colors_precomp, extra_colors, opacities, scales, rotations, cov3Ds_precomp))
    return _RasterizeGaussiansMulti.apply(means3D, means2D, sh, colors_precomp, extra_colors, opacities, scales, rotations, cov3Ds_precomp,
                                          raster_settings, need_bw)


class _RasterizeGaussiansMulti(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, extra_colors, opacities, scales, rotations, cov3Ds_precomp, raster_settings,
                need_bw=True):
        H, W = int(raster_settings.image_height), int(raster_settings.image_width)
        extra_out = torch.empty((3, H, W), dtype=torch.float32, device=means3D.device)
        color, depth, alpha, radii, ticket, saved = _autograd_forward(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                                                      cov3Ds_precomp, raster_settings, need_bw, extra=extra_colors,
                                                                      extra_out=extra_out)
        ctx.raster_settings = raster_settings
        ctx.ticket = ticket
        ctx.has = (sh.numel() != 0, colors_precomp.numel() != 0, scales.numel() != 0, cov3Ds_precomp.numel() != 0)
        ctx.needs = need_bw
        ctx.in_shapes = tuple(tuple(t.shape) for t in (means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp))
        ctx.extra_shape = tuple(extra_colors.shape)
        ctx.save_for_backward(*saved)
        ctx.mark_non_differentiable(radii)
        # outputs without a gradient arrive as None: an RGB-only loss runs the plain single-image backward
        ctx.set_materialize_grads(False)
        return color, depth, alpha, extra_out, radii

    @staticmethod
    def backward(ctx, grad_out_color, grad_out_depth, grad_out_alpha, grad_out_extra, _):
        if not ctx.needs:
            return (None,) * 11
        saved = ctx.saved_tensors
        g = _autograd_backward(ctx, saved, grad_out_color, grad_out_depth, grad_out_alpha, extra=saved[15], grad_out_extra=grad_out_extra)
        d_extra = g[8].view(ctx.extra_shape) if grad_out_extra is not None else None
        # input order: means3D, means2D, sh, colors_precomp, extra_colors, opacities, scales, rotations, cov3Ds_precomp, settings, need_bw
        return g[0], g[1], g[2], g[3], d_extra, g[4], g[5], g[6], g[7], None, None


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        """Boolean mask of the points in front of the near plane (__init__.py:179-188, rasterizer_impl.cu:54-66)."""
        with torch.no_grad():
            s = self.raster_settings
            if not positions.is_cuda:
                raise RuntimeError("autovfx_b200 rasterizer: positions must be a CUDA tensor")
            device = positions.device
            with torch.cuda.device(device):
                pos = _dev_f32(positions, device)
                view, proj = _dev_f32(s.viewmatrix, device), _dev_f32(s.projmatrix, device)
                P = pos.size(0)
                present = torch.zeros((P,), dtype=torch.bool, device=device)
                rc = _L.gsr_mark_visible(P, _ptr(pos), _ptr(view), _ptr(proj), _ptr(present),
                                         C.c_void_p(torch.cuda.current_stream(device).cuda_stream))
                _lib.check(rc, "gsr_mark_visible")
        return present

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None):
        raster_settings = self.raster_settings

        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')

        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')

        # absent inputs travel as empty tensors (their null data_ptr is the C side's "None", __init__.py:200-210)
        if shs is None:
            shs = torch.Tensor([])
        if colors_precomp is None:
            colors_precomp = torch.Tensor([])
        if scales is None:
            scales = torch.Tensor([])
        if rotations is None:
            rotations = torch.Tensor([])
        if cov3D_precomp is None:
            cov3D_precomp = torch.Tensor([])

        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, raster_settings)


def debug_views(workspaces, P: int, W: int, H: int) -> Dict[str, torch.Tensor]:
    """Typed tensor views into the opaque workspaces of a forward (parity tests: per-stage buffers, SURVEY §4)."""
    geom, binning, image = workspaces
    gx, gy = (W + 15) // 16, (H + 15) // 16
    tiles = gx * gy
    ws = _lib.gsr_workspace(geom.data_ptr(), geom.numel(), binning.data_ptr(), binning.numel(), image.data_ptr(), image.numel())
    v = _lib.gsr_views()
    _lib.check(_L.gsr_get_views(C.byref(ws), P, W, H, C.byref(v)), "gsr_get_views")
    cap = _L.gsr_binning_capacity(binning.numel())

    def view(base_t, ptr, nbytes, dtype, shape):
        off = ptr - base_t.data_ptr()
        return base_t[off:off + nbytes].view(dtype).view(*shape)

    return {
        "records": view(geom, v.records, 48 * P, torch.float32, (P, 12)),
        "cov3D": view(geom, v.cov3D, 24 * P, torch.float32, (P, 6)),
        "clamped": view(geom, v.clamped, P, torch.uint8, (P,)),
        "point_list": view(binning, v.point_list, 4 * cap, torch.int32, (cap,)),
        "sorted_keys": view(binning, v.sorted_keys, 8 * cap, torch.int64, (cap,)),
        "ranges": view(image, v.ranges, 8 * tiles, torch.int32, (tiles, 2)),
        "n_contrib": view(image, v.n_contrib, 4 * W * H, torch.int32, (H, W)),
        "tile_count": view(image, v.tile_count, 4 * tiles, torch.int32, (tiles,)) + view(image, v.tile_big, 4 * tiles, torch.int32, (tiles,)),
        "counters": view(image, v.counters, 32, torch.int32, (8,)),
    }
