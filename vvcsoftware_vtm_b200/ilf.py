"""ctypes binding of libilf_b200.so (include/ilf_b200.h).

No fallback of any kind: if the CUDA library is missing or no GPU is present the calls raise.  numpy arrays
in, numpy arrays out; pictures that are already on the GPU go in and out as torch CUDA tensors (upload_device,
set_original_device, download_device), on the caller's current torch stream.  Method names follow the reference entry points:
``loop_filter_pic`` = LoopFilter::loopFilterPic, ``sao_process`` = SampleAdaptiveOffset::SAOProcess,
``alf_process`` = AdaptiveLoopFilter::ALFProcess (DecLib.cpp:516-530).
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
STAGE_DEBLOCK, STAGE_SAO, STAGE_ALF, STAGE_ALL = 1, 2, 4, 7
SAO_CTU_BYTES = 32
MAX_SLICES = 64
BAND_HANDLE_BYTES = 192
BAND_ABOVE, BAND_BELOW = 0, 1


class IlfError(RuntimeError):
    pass


class IlfConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("width", "height", "bit_depth_luma", "bit_depth_chroma", "ctu_log2",
                                         "chroma_format", "device", "num_slots")]


class IlfBand(C.Structure):
    _fields_ = [("first_ctu_row", C.c_int32), ("num_ctu_rows", C.c_int32)]


class IlfSamples(C.Structure):
    """ilf_samples: sample type and the caller's (luma, chroma) bit depths of a device transfer."""
    _fields_ = [("type", C.c_int32), ("bit_depth", C.c_int32 * 2)]


SAMPLES_I16, SAMPLES_U8 = 0, 1   # ILF_SAMPLES_*


class IlfHashPart(C.Structure):
    """ilf_hash_part: a band's share of the decoded-picture hash (InLoopFilter.picture_hash_band, hash_combine)."""
    _fields_ = [(n, C.c_int32) for n in ("width", "height", "bd_luma", "bd_chroma", "first_row", "num_rows")] + \
               [("crc", C.c_uint32 * 3), ("sum", C.c_uint32 * 3)]


def lib_path():
    return os.environ.get("ILF_B200_LIB") or os.path.join(_HERE, "libilf_b200.so")


_LIB = None
NUM_KERNELS = 6   # ILF_NUM_KERNELS
ALF_STATS_WORDS = 25 * 105 + 36 + 36   # ILF_ALF_STATS_WORDS
DEBLOCK_SEARCH_MAX = 64   # ILF_DEBLOCK_SEARCH_MAX


def load_library():
    """Load libilf_b200.so; raises IlfError if it was not built (run ``python -c 'import __graft_entry__ as g; g.build()'``)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise IlfError(f"{path} is missing: the CUDA library was not built; there is no CPU fallback")
    lib = C.CDLL(path)
    vp, i, pd = C.c_void_p, C.c_int, C.c_ssize_t
    lib.ilf_abi_version.restype = i
    lib.ilf_create.argtypes = [C.POINTER(vp), C.POINTER(IlfConfig)]
    lib.ilf_create_band.argtypes = [C.POINTER(vp), C.POINTER(IlfConfig), C.POINTER(IlfBand)]
    lib.ilf_destroy.argtypes = [vp]
    lib.ilf_last_error.argtypes = [vp]
    lib.ilf_last_error.restype = C.c_char_p
    lib.ilf_get_config.argtypes = [vp, C.POINTER(IlfConfig)]
    lib.ilf_get_band.argtypes = [vp, C.POINTER(IlfBand), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.ilf_get_band_rows.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.ilf_upload_band.argtypes = [vp, i, vp, pd, vp, pd, vp, pd]
    lib.ilf_download_band.argtypes = [vp, i, vp, pd, vp, pd, vp, pd]
    lib.ilf_band_export.argtypes = [vp, i, C.c_char_p]
    lib.ilf_band_connect.argtypes = [vp, i, i, C.c_char_p]
    lib.ilf_band_exchange.argtypes = [vp, i]
    lib.ilf_band_exchange_batch.argtypes = [vp, i, i]
    lib.ilf_upload.argtypes = [vp, i, vp, pd, vp, pd, vp, pd]
    lib.ilf_download.argtypes = [vp, i, vp, pd, vp, pd, vp, pd]
    lib.ilf_sync.argtypes = [vp]
    lib.ilf_download_async.argtypes = [vp, i, vp, pd, vp, pd, vp, pd]
    lib.ilf_wait.argtypes = [vp, i]
    lib.ilf_upload_device.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, C.POINTER(IlfSamples), vp]
    lib.ilf_download_device.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, C.POINTER(IlfSamples), vp]
    lib.ilf_set_original_device.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, vp, C.POINTER(IlfSamples), vp]
    lib.ilf_host_alloc.argtypes = [C.c_size_t]
    lib.ilf_host_alloc.restype = vp
    lib.ilf_host_free.argtypes = [vp]
    lib.ilf_host_register.argtypes = [vp, C.c_size_t]
    lib.ilf_host_unregister.argtypes = [vp]
    lib.ilf_set_deblock_info.argtypes = [vp, i, vp, vp, vp, vp, vp, vp]
    lib.ilf_set_sao_params.argtypes = [vp, i, vp]
    lib.ilf_set_alf_params.argtypes = [vp, i, vp, vp]
    lib.ilf_run.argtypes = [vp, i, i, C.c_uint]
    for n in ("ilf_deblock", "ilf_sao", "ilf_alf"):
        getattr(lib, n).argtypes = [vp, i]
    lib.ilf_alf_classify.argtypes = [vp, i, vp]
    lib.ilf_set_original.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, vp]
    lib.ilf_sao_stats.argtypes = [vp, i, i]
    lib.ilf_get_sao_stats.argtypes = [vp, i, vp]
    lib.ilf_kernel_times.argtypes = [vp, C.POINTER(C.c_double * NUM_KERNELS), C.POINTER(C.c_longlong * NUM_KERNELS), C.POINTER(C.c_double * NUM_KERNELS)]
    lib.ilf_set_timing.argtypes = [vp, i]
    lib.ilf_alf_path.argtypes = [vp, i]
    lib.ilf_alf_stats.argtypes = [vp, i, i]
    lib.ilf_get_alf_stats.argtypes = [vp, i, vp]
    lib.ilf_deblock_search.argtypes = [vp, i, i, vp, i, vp]
    lib.ilf_get_deblock_search.argtypes = [vp, i, vp, i]
    lib.ilf_picture_hash.argtypes = [vp, i, i, C.POINTER(C.c_uint32 * 3)]
    lib.ilf_download_extended.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, i]
    lib.ilf_picture_hash_band.argtypes = [vp, i, C.POINTER(IlfHashPart)]
    lib.ilf_hash_combine.argtypes = [C.POINTER(IlfHashPart), i, i, C.POINTER(C.c_uint32 * 3)]
    lib.ilf_download_band_extended.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, i]
    lib.ilf_set_original_band.argtypes = [vp, i, vp, pd, vp, pd, vp, pd, vp]
    lib.ilf_launch_count.argtypes = [vp]
    lib.ilf_launch_count.restype = C.c_longlong
    lib.ilf_run_lanes.argtypes = [vp]
    lib.ilf_run_lanes.restype = C.c_int
    lib.ilf_slot_input_planes.argtypes = [vp, i, C.POINTER(vp * 3), C.POINTER(C.c_int32 * 3)]
    lib.ilf_slot_output_planes.argtypes = [vp, i, C.POINTER(vp * 3), C.POINTER(C.c_int32 * 3)]
    lib.ilf_stream.argtypes = [vp]
    lib.ilf_stream.restype = vp
    if lib.ilf_abi_version() != 1:
        raise IlfError("libilf_b200.so ABI version mismatch")
    _LIB = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _arr(a, dt):
    return None if a is None else np.ascontiguousarray(a, dtype=dt)


def hash_combine(parts, kind="crc"):
    """ilf_hash_combine: [Y, Cb, Cr] of the whole picture from the parts of all its bands (picture_hash_band), in any order.  A part
    is the bytes picture_hash_band returned (or an IlfHashPart), so parts can come from other processes."""
    kinds = {"crc": 1, "checksum": 2}
    if kind not in kinds:
        raise IlfError(f"unknown hash kind {kind!r}: 'crc' or 'checksum'")
    lib = load_library()
    arr = (IlfHashPart * max(1, len(parts)))()
    for j, p in enumerate(parts):
        b = bytes(p)
        if len(b) != C.sizeof(IlfHashPart):
            raise IlfError(f"a hash part is {C.sizeof(IlfHashPart)} bytes, got {len(b)}")
        C.memmove(C.byref(arr, j * C.sizeof(IlfHashPart)), b, len(b))
    out = (C.c_uint32 * 3)()
    rc = lib.ilf_hash_combine(arr, len(parts), kinds[kind], C.byref(out))
    if rc != 0:
        raise IlfError(f"ilf_hash_combine failed ({rc}): the parts do not tile one picture")
    return [int(v) for v in out]


def pinned_planes(width, height):
    """{"y","cb","cr"} int16 arrays in page-locked host memory (ilf_host_alloc); keep the dict alive while in use."""
    lib = load_library()
    out = {}
    for k, (h, w) in (("y", (height, width)), ("cb", (height // 2, width // 2)), ("cr", (height // 2, width // 2))):
        p = lib.ilf_host_alloc(h * w * 2)
        if not p:
            raise IlfError("ilf_host_alloc failed")
        out[k] = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int16)), shape=(h, w))
    return out


class InLoopFilter:
    """One context: a CUDA device plus ``num_slots`` resident pictures of one geometry."""

    def __init__(self, width, height, bit_depth_luma=10, bit_depth_chroma=10, ctu_log2=7, device=0, num_slots=1, band=None):
        self._lib = load_library()
        self.cfg = IlfConfig(width, height, bit_depth_luma, bit_depth_chroma, ctu_log2, 1, device, num_slots)
        self._h = C.c_void_p()
        if band is None:
            rc = self._lib.ilf_create(C.byref(self._h), C.byref(self.cfg))
        else:
            b = IlfBand(*band)
            rc = self._lib.ilf_create_band(C.byref(self._h), C.byref(self.cfg), C.byref(b))
        if rc != 0:
            msg = self._lib.ilf_last_error(None).decode()
            self._h = C.c_void_p()
            raise IlfError(f"ilf_create failed ({rc}): {msg}")
        r0, nr = C.c_int32(), C.c_int32()
        self._lib.ilf_get_band(self._h, None, C.byref(r0), C.byref(nr))
        self.row0, self.rows = r0.value, nr.value   # picture rows held by this context
        self._lib.ilf_get_band_rows(self._h, C.byref(r0), C.byref(nr))
        self.own_row0, self.own_rows = r0.value, nr.value   # picture rows this context produces (band mode: its own CTU rows)
        self.width, self.height = width, height
        ctu = 1 << ctu_log2
        self.ctus_w, self.ctus_h = (width + ctu - 1) // ctu, (height + ctu - 1) // ctu
        self.own_ctus = self.ctus_w * ((self.own_row0 + self.own_rows + ctu - 1) // ctu - self.own_row0 // ctu)   # statistics records

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.ilf_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise IlfError(f"libilf_b200 error {rc}: {self._lib.ilf_last_error(self._h).decode()}")

    # ---- transfers -------------------------------------------------------------------------------
    def upload(self, slot, y, cb, cr):
        y, cb, cr = (_arr(a, np.int16) for a in (y, cb, cr))
        assert y.shape == (self.rows, self.width) and cb.shape == cr.shape == (self.rows // 2, self.width // 2)
        self._ck(self._lib.ilf_upload(self._h, slot, _ptr(y), y.shape[1], _ptr(cb), cb.shape[1], _ptr(cr), cr.shape[1]))

    def download_async(self, slot, out):
        """Start the device -> host copy of `slot` into `out` (dict of page-locked int16 arrays); wait(slot) completes it."""
        y, cb, cr = out["y"], out["cb"], out["cr"]
        self._ck(self._lib.ilf_download_async(self._h, slot, _ptr(y), y.shape[1], _ptr(cb), cb.shape[1], _ptr(cr), cr.shape[1]))

    def wait(self, slot):
        self._ck(self._lib.ilf_wait(self._h, slot))

    def download(self, slot, out=None):
        """Filtered picture of `slot` as {"y","cb","cr"}; `out` = dict of preallocated int16 arrays to fill (e.g. pinned)."""
        if out is not None:
            y, cb, cr = out["y"], out["cb"], out["cr"]
            assert y.shape == (self.rows, self.width) and cb.shape == cr.shape == (self.rows // 2, self.width // 2)
            assert all(a.dtype == np.int16 and a.flags.c_contiguous for a in (y, cb, cr))
        else:
            y = np.empty((self.rows, self.width), np.int16)
            cb = np.empty((self.rows // 2, self.width // 2), np.int16)
            cr = np.empty_like(cb)
        self._ck(self._lib.ilf_download(self._h, slot, _ptr(y), y.shape[1], _ptr(cb), cb.shape[1], _ptr(cr), cr.shape[1]))
        return {"y": y, "cb": cb, "cr": cr}

    def sync(self):
        self._ck(self._lib.ilf_sync(self._h))

    # ---- pictures in device memory (torch CUDA tensors) -----------------------------------------------
    # Planes are 2-D CUDA tensors on the context's device with stride(-1) == 1, all int16 or all uint8 (which selects the sample
    # type), of the shapes of the rows the context produces (own_rows x width, chroma halved): the whole picture, or a band's own
    # rows.  bit_depth = the caller's depth: None (int16: the context's; uint8: 8), one int, or a (luma, chroma) pair.  Every call is
    # ordered on torch.cuda.current_stream of the context's device and returns without waiting.
    def _device_planes(self, planes, bit_depth):
        import torch
        shapes = ((self.own_rows, self.width), (self.own_rows // 2, self.width // 2), (self.own_rows // 2, self.width // 2))
        dtype = planes[0].dtype if isinstance(planes[0], torch.Tensor) else None
        if dtype not in (torch.int16, torch.uint8):
            raise IlfError("device planes are torch.int16 or torch.uint8 CUDA tensors")
        args = []
        for name, t, shape in zip(("y", "cb", "cr"), planes, shapes):
            if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dtype:
                raise IlfError(f"plane {name}: a CUDA tensor of dtype {dtype} is expected")
            if t.dim() != 2 or tuple(t.shape) != shape or t.stride(-1) != 1:
                raise IlfError(f"plane {name}: shape {tuple(t.shape)} strides {t.stride()}, expected shape {shape} with stride(-1) == 1")
            args += [C.c_void_p(t.data_ptr()), t.stride(0)]
        if bit_depth is None:
            bd = (0, 0)
        elif isinstance(bit_depth, int):
            bd = (bit_depth, bit_depth)
        else:
            bd = tuple(bit_depth)
        fmt = IlfSamples(SAMPLES_I16 if dtype == torch.int16 else SAMPLES_U8, (C.c_int32 * 2)(*bd))
        stream = torch.cuda.current_stream(torch.device("cuda", self.cfg.device)).cuda_stream
        return args, fmt, C.c_void_p(stream)

    def upload_device(self, slot, y, cb, cr, bit_depth=None):
        """ilf_upload_device: the picture (a band: its own rows) from CUDA tensors; side information must be set again after it."""
        args, fmt, stream = self._device_planes((y, cb, cr), bit_depth)
        self._ck(self._lib.ilf_upload_device(self._h, slot, *args, C.byref(fmt), stream))

    def set_original_device(self, slot, y, cb, cr, ctu_avail, bit_depth=None):
        """ilf_set_original_device: the encoder's source picture (a band: its own rows) from CUDA tensors, e.g. 8-bit frames
        (uint8) for a 10-bit context; ctu_avail (host, every CTU of the picture) as in set_original."""
        args, fmt, stream = self._device_planes((y, cb, cr), bit_depth)
        av = _arr(ctu_avail, np.uint8)
        assert av.size == self.ctus_w * self.ctus_h
        self._ck(self._lib.ilf_set_original_device(self._h, slot, *args, _ptr(av), C.byref(fmt), stream))

    def download_device(self, slot, dtype=None, bit_depth=None, out=None):
        """ilf_download_device: the slot's current picture (a band: its own rows) as {"y","cb","cr"} CUDA tensors of `dtype`
        (torch.int16, the default, or torch.uint8); `out` = such a dict to fill instead."""
        import torch
        if out is None:
            dev = torch.device("cuda", self.cfg.device)
            dt = torch.int16 if dtype is None else dtype
            out = {"y": torch.empty((self.own_rows, self.width), dtype=dt, device=dev)}
            out["cb"] = torch.empty((self.own_rows // 2, self.width // 2), dtype=dt, device=dev)
            out["cr"] = torch.empty_like(out["cb"])
        args, fmt, stream = self._device_planes((out["y"], out["cb"], out["cr"]), bit_depth)
        self._ck(self._lib.ilf_download_device(self._h, slot, *args, C.byref(fmt), stream))
        return out

    # ---- CTU-row band mode (one picture across several GPUs) ---------------------------------------
    def upload_band(self, slot, y, cb, cr):
        """Upload the band's OWN rows (own_rows x width); halo rows come from the neighbours (band_exchange)."""
        y, cb, cr = (_arr(a, np.int16) for a in (y, cb, cr))
        assert y.shape == (self.own_rows, self.width) and cb.shape == cr.shape == (self.own_rows // 2, self.width // 2)
        self._ck(self._lib.ilf_upload_band(self._h, slot, _ptr(y), y.shape[1], _ptr(cb), cb.shape[1], _ptr(cr), cr.shape[1]))

    def download_band(self, slot):
        y = np.empty((self.own_rows, self.width), np.int16)
        cb = np.empty((self.own_rows // 2, self.width // 2), np.int16)
        cr = np.empty_like(cb)
        self._ck(self._lib.ilf_download_band(self._h, slot, _ptr(y), y.shape[1], _ptr(cb), cb.shape[1], _ptr(cr), cr.shape[1]))
        return {"y": y, "cb": cb, "cr": cr}

    def download_band_extended(self, slot, margin, out=None):
        """The band's own rows, with Picture::extendPicBorder's margins, into full-picture planes of size (h + 2 m, w + 2 m),
        m = margin (luma) or margin / 2: only the own rows, their left / right margins and, for the first / last band, the margin
        rows above / below the picture are written.  `out`: such a dict to fill (every band into the same one), else new planes
        filled with -1."""
        if out is None:
            out = {k: np.full(((self.height >> sh) + 2 * (margin >> sh), (self.width >> sh) + 2 * (margin >> sh)), -1, np.int16)
                   for k, sh in (("y", 0), ("cb", 1), ("cr", 1))}
        ptrs = []
        for k, sh in (("y", 0), ("cb", 1), ("cr", 1)):
            m, a = margin >> sh, out[k]
            assert a.dtype == np.int16 and a.flags.c_contiguous and a.shape == ((self.height >> sh) + 2 * m, (self.width >> sh) + 2 * m)
            ptrs += [C.c_void_p(a.ctypes.data + 2 * ((m + (self.own_row0 >> sh)) * a.shape[1] + m)), a.shape[1]]
        self._ck(self._lib.ilf_download_band_extended(self._h, slot, *ptrs, margin))
        return out

    def picture_hash_band(self, slot=0):
        """The band's part of the decoded-picture hash (CRC and checksum of its own rows) as bytes of an ilf_hash_part: picklable,
        for hash_combine in whichever process gathers the bands."""
        part = IlfHashPart()
        self._ck(self._lib.ilf_picture_hash_band(self._h, slot, C.byref(part)))
        return bytes(part)

    def set_original_band(self, slot, y, cb, cr, ctu_avail):
        """Source picture of the band's OWN rows (own_rows x width) and the ILF_AVAIL_* flags of every CTU of the picture."""
        y, cb, cr = (_arr(a, np.int16) for a in (y, cb, cr))
        assert y.shape == (self.own_rows, self.width) and cb.shape == cr.shape == (self.own_rows // 2, self.width // 2)
        av = _arr(ctu_avail, np.uint8)
        assert av.size == self.ctus_w * self.ctus_h
        self._ck(self._lib.ilf_set_original_band(self._h, slot, _ptr(y), y.shape[1], _ptr(cb), cb.shape[1], _ptr(cr), cr.shape[1], _ptr(av)))

    def band_export(self, slot=0):
        """Opaque handle (bytes) of the slot's planes for the neighbouring band contexts, in this or another process."""
        buf = C.create_string_buffer(BAND_HANDLE_BYTES)
        self._ck(self._lib.ilf_band_export(self._h, slot, buf))
        return buf.raw

    def band_connect(self, slot, side, handle):
        assert len(handle) == BAND_HANDLE_BYTES
        self._ck(self._lib.ilf_band_connect(self._h, slot, side, handle))

    def band_exchange(self, slot=0, num_slots=1):
        """Pull the halo rows of slots [slot, slot + num_slots) from the connected neighbours (one kernel over NVLink P2P)."""
        self._ck(self._lib.ilf_band_exchange_batch(self._h, slot, num_slots))

    # ---- side information ------------------------------------------------------------------------
    def set_deblock_info(self, slot, params_bytes, info, info_chroma=None, mv16=None, mv32=None, ctu_slice=None):
        pb = np.frombuffer(bytes(params_bytes), dtype=np.uint8).copy()
        info = _arr(info, np.uint32); info_chroma = _arr(info_chroma, np.uint32)
        mv16 = _arr(mv16, np.int16); mv32 = _arr(mv32, np.int32); ctu_slice = _arr(ctu_slice, np.uint8)
        assert info.size == (self.rows // 4) * (self.width // 4)
        self._ck(self._lib.ilf_set_deblock_info(self._h, slot, _ptr(pb), _ptr(info), _ptr(info_chroma), _ptr(mv16), _ptr(mv32), _ptr(ctu_slice)))

    def set_sao_params(self, slot, sao_ctus):
        a = _arr(sao_ctus, np.uint8)
        assert a.size == self.ctus_w * self.ctus_h * SAO_CTU_BYTES
        self._ck(self._lib.ilf_set_sao_params(self._h, slot, _ptr(a)))

    def set_alf_params(self, slot, alf_params_bytes, ctu_enable):
        pb = np.frombuffer(bytes(alf_params_bytes), dtype=np.uint8).copy()
        en = _arr(ctu_enable, np.uint8)
        assert en.size == 3 * self.ctus_w * self.ctus_h
        self._ck(self._lib.ilf_set_alf_params(self._h, slot, _ptr(pb), _ptr(en)))

    # ---- execution -------------------------------------------------------------------------------
    def run(self, first_slot=0, num_slots=1, stages=STAGE_ALL):
        self._ck(self._lib.ilf_run(self._h, first_slot, num_slots, stages))

    def loop_filter_pic(self, slot=0):
        self._ck(self._lib.ilf_deblock(self._h, slot))

    def sao_process(self, slot=0):
        self._ck(self._lib.ilf_sao(self._h, slot))

    def alf_process(self, slot=0):
        self._ck(self._lib.ilf_alf(self._h, slot))

    def alf_classify(self, slot=0):
        """classIdx | transposeIdx << 5 per 4x4 luma block of the rows the context produces (a band context: its own rows)."""
        out = np.empty((self.rows // 4, self.width // 4), np.uint8)
        self._ck(self._lib.ilf_alf_classify(self._h, slot, _ptr(out)))
        u0 = (self.own_row0 - self.row0) // 4
        return out[u0:u0 + self.own_rows // 4].copy()

    # ---- encoder SAO statistics (EncSampleAdaptiveOffset::getStatistics) ---------------------------------
    def set_original(self, slot, y, cb, cr, ctu_avail):
        """Source picture of the slot and the per-CTU ILF_AVAIL_L/_A/_AL flags of the statistics pass."""
        y, cb, cr = (_arr(a, np.int16) for a in (y, cb, cr))
        av = _arr(ctu_avail, np.uint8)
        self._ck(self._lib.ilf_set_original(self._h, slot, _ptr(y), y.strides[0] // 2, _ptr(cb), cb.strides[0] // 2, _ptr(cr), cr.strides[0] // 2, _ptr(av)))

    def sao_stats(self, first_slot=0, num_slots=1):
        self._ck(self._lib.ilf_sao_stats(self._h, first_slot, num_slots))

    def get_sao_stats(self, slot=0):
        """int64 [num_ctus, 3, 5, 64]: per CTU, component and SAO type diff[32] then count[32] (SAOStatData); a band context: its own CTUs."""
        out = np.empty((self.own_ctus, 3, 5, 64), np.int64)
        self._ck(self._lib.ilf_get_sao_stats(self._h, slot, _ptr(out)))
        return out

    # ---- measurement -----------------------------------------------------------------------------
    def set_timing(self, on):
        self._ck(self._lib.ilf_set_timing(self._h, int(on)))

    KERNELS = ("deblock", "sao", "alf", "alf_chroma", "sao_stats", "alf_stats")   # "alf" = the whole ALF stage (one launch); "alf_chroma" is reserved, always zero

    def kernel_times(self):
        """{kernel: (total ms, launches, algorithmic bytes)} since set_timing(True); synchronises the context's stream."""
        ms = (C.c_double * NUM_KERNELS)(); n = (C.c_longlong * NUM_KERNELS)(); nb = (C.c_double * NUM_KERNELS)()
        self._ck(self._lib.ilf_kernel_times(self._h, C.byref(ms), C.byref(n), C.byref(nb)))
        return {k: (ms[i], n[i], nb[i]) for i, k in enumerate(self.KERNELS)}

    def alf_stats(self, first_slot=0, num_slots=1):
        """Encoder ALF statistics (EncAdaptiveLoopFilter::deriveStatsForFiltering) of the slots' current pictures against their originals."""
        self._ck(self._lib.ilf_alf_stats(self._h, first_slot, num_slots))

    def get_alf_stats(self, slot=0):
        """int64 [num_ctus, ALF_STATS_WORDS]; a band context: its own CTUs."""
        out = np.zeros((self.own_ctus, ALF_STATS_WORDS), np.int64)
        self._ck(self._lib.ilf_get_alf_stats(self._h, slot, _ptr(out)))
        return out

    # ---- encoder deblocking parameter search (EncGOP::applyDeblockingFilterParameterSelection) -----------
    def deblock_search(self, candidates, shift=(0, 0), first_slot=0, num_slots=1):
        """Score (beta_offset_div2, tc_offset_div2) pairs on the slots' uploaded pictures: per candidate and plane, the sum of
        ((deblocked - original)^2 >> shift[luma / chroma]) with every slice's offsets replaced by the candidate's."""
        c = np.asarray(candidates, dtype=np.int64).reshape(-1, 2)
        if c.size and (c.min() < -128 or c.max() > 127):
            raise IlfError("deblocking offsets must fit int8")
        c = np.ascontiguousarray(c.astype(np.int8))
        sh = np.ascontiguousarray(shift, dtype=np.int32)
        assert sh.shape == (2,)
        self._ck(self._lib.ilf_deblock_search(self._h, first_slot, num_slots, _ptr(c), len(c), _ptr(sh)))

    def get_deblock_search(self, slot=0):
        """uint64 [K, 3]: the sums of the slot's last deblock_search, per candidate and plane (Y, Cb, Cr)."""
        out = np.zeros((DEBLOCK_SEARCH_MAX, 3), np.uint64)
        r = self._lib.ilf_get_deblock_search(self._h, slot, _ptr(out), DEBLOCK_SEARCH_MAX)
        if r < 0:
            self._ck(r)
        return out[:r].copy()

    def picture_hash(self, slot=0, kind="crc"):
        """calcCRC / calcChecksum of the slot's current picture on the device: [Y, Cb, Cr]."""
        out = (C.c_uint32 * 3)()
        self._ck(self._lib.ilf_picture_hash(self._h, slot, 1 if kind == "crc" else 2, C.byref(out)))
        return [int(v) for v in out]

    def download_extended(self, slot, margin):
        """The slot's picture with Picture::extendPicBorder applied: dict of planes of size (h + 2 m, w + 2 m), m = margin (luma) or margin / 2."""
        out = {}
        ptrs = []
        for k, sh in (("y", 0), ("cb", 1), ("cr", 1)):
            m = margin >> sh
            a = np.full(((self.height >> sh) + 2 * m, (self.width >> sh) + 2 * m), -1, np.int16)
            out[k] = a
            ptrs += [C.c_void_p(a.ctypes.data + 2 * (m * a.shape[1] + m)), a.shape[1]]
        self._ck(self._lib.ilf_download_extended(self._h, slot, *ptrs, margin))
        return out

    def alf_path(self, slot=0):
        """Bits ILF_ALF_PATH_LUMA_DOT (1) / ILF_ALF_PATH_CHROMA_DOT (2): which arithmetic path the slot's ALF filters take."""
        r = self._lib.ilf_alf_path(self._h, slot)
        if r < 0:
            self._ck(r)
        return r

    def run_lanes(self):
        """Compute streams a chain over a large batch is dealt to (ilf_run_lanes; 1 = off)."""
        return int(self._lib.ilf_run_lanes(self._h))

    def launch_count(self):
        return int(self._lib.ilf_launch_count(self._h))

    def input_planes(self, slot):
        p = (C.c_void_p * 3)(); pitch = (C.c_int32 * 3)()
        self._ck(self._lib.ilf_slot_input_planes(self._h, slot, C.byref(p), C.byref(pitch)))
        return [int(v) for v in p], list(pitch)

    def output_planes(self, slot):
        p = (C.c_void_p * 3)(); pitch = (C.c_int32 * 3)()
        self._ck(self._lib.ilf_slot_output_planes(self._h, slot, C.byref(p), C.byref(pitch)))
        return [int(v) for v in p], list(pitch)

    def stream(self):
        return int(self._lib.ilf_stream(self._h) or 0)
