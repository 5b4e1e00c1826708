"""Host-side mirror of the reference's receive-chain interface over libt41rx.so (ctypes).

The reference exposes `void ProcessIQData(void)` working on globals (Process.h:15); here the
same call is `Receiver.process(iq)` on a bank of virtual receivers, with the globals the chain
samples (`bands[].mode/FLoCut/FHiCut`, `NCOFreq`, `AGCMode`, `spectrumZoom`, ...) set through
`Receiver.set_params`.  This module is plumbing only: every sample is processed by the CUDA
kernels inside libt41rx.so; if the library or a GPU is missing, construction raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("T41RX_LIB", os.path.join(_HERE, "libt41rx.so"))

DEMOD_USB, DEMOD_LSB, DEMOD_AM, DEMOD_NFM, DEMOD_PSK31, DEMOD_SAM = 0, 1, 2, 3, 5, 8
BLOCK = 2048
SPECTRUM_RES = 512
SPEC_FRAME_BYTES = 518    # specData[], t41Control.cpp:21
AUDIO_SPEC_PIXELS = 270   # AUDIO_SPEC_BOX_W - 2 (Display.h:45, Process.cpp:555)
FLAG_EXACT_NCO = 1       # bit-exact kernel, step-by-step FP64 oscillator
FLAG_PHASED_KERNEL = 2   # bit-exact kernel with the closed-form FP64 oscillator
FLAG_FAST_LMS = 8        # LMS / notch receivers on the throughput kernel too (audio SNR >= 70 dB instead of 90)
FLAG_FAST_SAM = 16       # SAM receivers on the throughput kernel too (acquisition transient differs, locked: >= 90 dB)
FLAG_FUSED_EXACT = 32    # bit-exact chain as the single fused kernel instead of front | serial | back kernels
FLAG_SCAN_ROWS = 4       # rows kernel: scan form of the ZoomFFT biquads (<= 1 LSB, < 1 % of pixels)
# flags = 0: the throughput kernel

# algorithmic HBM bytes per stream-block (SURVEY.md section 8(d))
BYTES_PER_BLOCK = 2 * BLOCK * 4 + BLOCK * 4        # 16 KiB I/Q in + 8 KiB audio out
BYTES_PER_BLOCK_Q15 = 2 * BLOCK * 2 + BLOCK * 2    # the firmware's q15 blocks: 8 KiB I/Q in + 4 KiB audio out
BYTES_PER_ROW = SPECTRUM_RES * 2 + SPECTRUM_RES * 2  # int16 spectrum row + RGB565 waterfall row


class Params(C.Structure):
    """t41rx_params (include/t41rx.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "mode", "f_lo_cut", "f_hi_cut", "nco_freq", "agc_mode", "agc_thresh", "audio_volume",
        "rf_gain_all_bands", "rf_gain", "spectrum_zoom", "current_scale", "pixel_offset",
        "current_nf", "spectrum_noise_floor", "nfm_filter_bw", "psk31_enable")] + [
        ("iq_amp_correction", C.c_float), ("iq_phase_correction", C.c_float),
        ("receive_eq_flag", C.c_int32), ("equalizer_rec", C.c_int32 * 14),
        ("nr_option", C.c_int32), ("anr_notch_on", C.c_int32), ("cw_receive", C.c_int32),
        ("cw_filter_index", C.c_int32), ("nb_on", C.c_int32)]

    def copy(self):
        p = Params()
        C.memmove(C.byref(p), C.byref(self), C.sizeof(Params))
        return p


class Debug(C.Structure):
    """t41rx_debug."""
    _fields_ = [(n, C.c_int32) for n in (
        "agc_state", "agc_decay_type", "agc_hang_counter", "agc_action", "rf_gain", "codec_timer",
        "zoom_sample_ptr", "first_block")] + [(n, C.c_float) for n in (
        "agc_volts", "agc_ring_max", "agc_save_volts", "agc_fast_backaverage", "agc_hang_backaverage",
        "sam_phzerror", "sam_omega2", "sam_fil_out")] + [
        ("dc_state", C.c_float * 2), ("am_wold", C.c_float),
        ("osc_vect_q", C.c_double), ("osc_vect_i", C.c_double)]


class Tables(C.Structure):
    """t41rx_tables."""
    _fields_ = [("dec1", C.c_float * 28), ("dec2", C.c_float * 46), ("int1", C.c_float * 48),
                ("int2", C.c_float * 32), ("mask", C.c_float * 1024), ("am_lp", C.c_float * 5),
                ("zoom_fir", C.c_float * 4), ("agc", C.c_float * 16),
                ("attack_buffsize", C.c_int32), ("hang_counter_load", C.c_int32)]

    def as_dict(self):
        d = {n: np.array(getattr(self, n), dtype=np.float32) for n in
             ("dec1", "dec2", "int1", "int2", "mask", "am_lp", "zoom_fir", "agc")}
        d["attack_buffsize"] = int(self.attack_buffsize)
        d["hang_counter_load"] = int(self.hang_counter_load)
        return d


EXPORTS = (
    "t41rx_default_params", "t41rx_mode_default_cuts", "t41rx_create", "t41rx_destroy",
    "t41rx_num_streams", "t41rx_set_params", "t41rx_set_params_each", "t41rx_get_params",
    "t41rx_get_tables", "t41rx_get_debug", "t41rx_design_tables", "t41rx_process", "t41rx_process_q15",
    "t41rx_process_device", "t41rx_process_device_q15", "t41rx_synchronize", "t41rx_kernel_launches", "t41rx_last_kernel_ms",
    "t41rx_stream_kernel_times", "t41rx_bind_audio_spectrum", "t41rx_bind_control_frames", "t41rx_smeter_dbm", "t41rx_smeter_bar",
    "t41rx_load_wav", "t41rx_read_wave", "t41rx_wav_sample_rate", "t41rx_wav_close",
    "t41rx_last_error", "t41rx_version",
    "t41rx_create_multi", "t41rx_destroy_multi", "t41rx_multi_num_devices", "t41rx_multi_num_streams", "t41rx_multi_shard",
    "t41rx_multi_set_params", "t41rx_multi_set_params_each", "t41rx_multi_get_debug", "t41rx_multi_process",
    "t41rx_multi_process_q15", "t41rx_multi_process_device", "t41rx_multi_synchronize", "t41rx_multi_gather_rows",
    "t41rx_multi_last_error", "t41rx_dc_refilter_count",
    "t41rx_chan_create", "t41rx_chan_destroy", "t41rx_chan_set_map", "t41rx_chan_process_device", "t41rx_chan_synchronize",
    "t41rx_chan_taps", "t41rx_chan_tune", "t41rx_chan_set_shift", "t41rx_chan_place",
    "t41rx_chan_create_real", "t41rx_chan_process_device_real", "t41rx_chan_tune_real", "t41rx_chan_place_real",
    "t41rx_chan_create_q15", "t41rx_chan_process_device_q15",
    "t41rx_chan_create_diversity", "t41rx_chan_set_weights", "t41rx_chan_process_device_diversity",
    "t41rx_chan_set_image", "t41rx_chan_get_image", "t41rx_chan_track_image", "t41rx_chan_image_stats")

CHAN_TAPS_PER_BRANCH = 10     # prototype length = 10 * n_channels
CHAN_SPACING = 96000.0        # channel spacing (Hz); every channel comes out at 192 kS/s
CHAN_FLOAT, CHAN_Q15, CHAN_REAL = 0, 1, 2   # capture kinds of t41rx_chan_create_diversity
CHAN_MAX_INPUTS = 4           # a diversity channelizer takes 2 ... 4 coherent captures
CHAN_DOMINANCE_DB = (3.0, 60.0)   # image tracking's dominance threshold T (dB), T41RX_CHAN_DOMINANCE_MIN/MAX_DB


def build_library():
    """Compile libt41rx.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(_HERE, "csrc"), "all"])


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libt41rx.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(LIB_PATH)
        vp, ip = C.c_void_p, C.c_int
        L.t41rx_default_params.argtypes = [C.POINTER(Params)]
        L.t41rx_mode_default_cuts.argtypes = [C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.t41rx_create.argtypes = [C.POINTER(vp), ip, ip]
        L.t41rx_destroy.argtypes = [vp]
        L.t41rx_num_streams.argtypes = [vp]
        L.t41rx_set_params.argtypes = [vp, ip, ip, C.POINTER(Params)]
        L.t41rx_set_params_each.argtypes = [vp, ip, ip, C.POINTER(Params)]
        L.t41rx_get_params.argtypes = [vp, ip, C.POINTER(Params)]
        L.t41rx_get_tables.argtypes = [vp, ip, C.POINTER(Tables)]
        L.t41rx_get_debug.argtypes = [vp, ip, C.POINTER(Debug)]
        L.t41rx_design_tables.argtypes = [C.POINTER(Params), ip, C.POINTER(Tables)]
        L.t41rx_process.argtypes = [vp, vp, vp, ip, ip, vp, vp, vp, vp, C.c_uint32]
        L.t41rx_process_q15.argtypes = [vp, vp, vp, ip, ip, vp, vp, vp, vp, C.c_uint32]
        L.t41rx_process_device.argtypes = [vp, vp, vp, ip, ip, vp, vp, vp, vp, C.c_uint32, vp]
        L.t41rx_process_device_q15.argtypes = [vp, vp, vp, ip, ip, vp, vp, vp, vp, C.c_uint32, vp]
        L.t41rx_synchronize.argtypes = [vp]
        L.t41rx_kernel_launches.argtypes = [vp]
        L.t41rx_kernel_launches.restype = C.c_int64
        L.t41rx_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.t41rx_stream_kernel_times.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
        L.t41rx_bind_audio_spectrum.argtypes = [vp, vp, vp]
        L.t41rx_bind_control_frames.argtypes = [vp, vp, vp]
        L.t41rx_smeter_dbm.argtypes = [C.c_float, C.c_float, C.c_int32, C.c_int32]
        L.t41rx_smeter_dbm.restype = C.c_float
        L.t41rx_smeter_bar.argtypes = [C.c_float]
        L.t41rx_smeter_bar.restype = C.c_int32
        L.t41rx_load_wav.argtypes = [C.POINTER(vp), C.c_char_p, C.c_uint32]
        L.t41rx_read_wave.argtypes = [vp, vp, ip]
        L.t41rx_wav_sample_rate.argtypes = [vp]
        L.t41rx_wav_sample_rate.restype = C.c_uint32
        L.t41rx_wav_close.argtypes = [vp]
        L.t41rx_wav_close.restype = None
        L.t41rx_last_error.restype = C.c_char_p
        L.t41rx_version.restype = C.c_char_p
        L.t41rx_create_multi.argtypes = [C.POINTER(vp), ip, C.POINTER(ip), ip]
        L.t41rx_destroy_multi.argtypes = [vp]
        L.t41rx_destroy_multi.restype = None
        L.t41rx_multi_num_devices.argtypes = [vp]
        L.t41rx_multi_num_streams.argtypes = [vp]
        L.t41rx_multi_shard.argtypes = [vp, ip, C.POINTER(ip), C.POINTER(ip), C.POINTER(ip), C.POINTER(vp)]
        L.t41rx_multi_set_params.argtypes = [vp, ip, ip, C.POINTER(Params)]
        L.t41rx_multi_set_params_each.argtypes = [vp, ip, ip, C.POINTER(Params)]
        L.t41rx_multi_get_debug.argtypes = [vp, ip, C.POINTER(Debug)]
        L.t41rx_multi_process.argtypes = [vp, vp, vp, ip, ip, vp, vp, vp, vp, C.c_uint32]
        L.t41rx_multi_process_q15.argtypes = [vp, vp, vp, ip, ip, vp, vp, vp, vp, C.c_uint32]
        L.t41rx_multi_process_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), ip, ip, C.POINTER(vp), C.POINTER(vp), C.c_uint32]
        L.t41rx_multi_synchronize.argtypes = [vp]
        L.t41rx_multi_gather_rows.argtypes = [vp, C.POINTER(vp), C.c_size_t, vp, C.POINTER(ip)]
        L.t41rx_multi_last_error.restype = C.c_char_p
        L.t41rx_dc_refilter_count.restype = C.c_int64
        L.t41rx_chan_create.argtypes = [C.POINTER(vp), ip, ip, ip]
        L.t41rx_chan_destroy.argtypes = [vp]
        L.t41rx_chan_destroy.restype = None
        L.t41rx_chan_set_map.argtypes = [vp, ip, ip, C.POINTER(C.c_int32)]
        L.t41rx_chan_process_device.argtypes = [vp, vp, vp, ip, vp]
        L.t41rx_chan_synchronize.argtypes = [vp]
        L.t41rx_chan_taps.argtypes = [ip, C.POINTER(C.c_float)]
        L.t41rx_chan_tune.argtypes = [ip, C.c_int32, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.t41rx_chan_set_shift.argtypes = [vp, ip, ip, C.POINTER(C.c_int32)]
        L.t41rx_chan_create_real.argtypes = [C.POINTER(vp), ip, ip, ip]
        L.t41rx_chan_process_device_real.argtypes = [vp, vp, vp, ip, vp]
        L.t41rx_chan_create_q15.argtypes = [C.POINTER(vp), ip, ip, ip]
        L.t41rx_chan_process_device_q15.argtypes = [vp, vp, vp, ip, vp]
        L.t41rx_chan_create_diversity.argtypes = [C.POINTER(vp), ip, ip, ip, ip, ip]
        L.t41rx_chan_set_weights.argtypes = [vp, ip, ip, C.POINTER(C.c_float)]
        L.t41rx_chan_process_device_diversity.argtypes = [vp, C.POINTER(vp), vp, ip, vp]
        L.t41rx_chan_set_image.argtypes = [vp, ip, ip, C.POINTER(C.c_float)]
        L.t41rx_chan_get_image.argtypes = [vp, C.POINTER(C.c_float)]
        L.t41rx_chan_track_image.argtypes = [vp, ip, C.c_float]
        L.t41rx_chan_image_stats.argtypes = [vp, C.POINTER(C.c_double)]
        L.t41rx_chan_tune_real.argtypes = [ip, C.c_int32, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.t41rx_chan_place_real.argtypes = [ip, C.c_int32, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                            C.POINTER(C.c_int32)]
        L.t41rx_chan_place.argtypes = [ip, C.c_int32, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                       C.POINTER(C.c_int32)]
        _lib = L
    return _lib


class T41RxError(RuntimeError):
    pass


def _check(rc, what):
    if rc != 0:
        raise T41RxError("%s failed (%d): %s" % (what, rc, lib().t41rx_last_error().decode()))


def default_params():
    p = Params()
    lib().t41rx_default_params(C.byref(p))
    return p


def mode_default_cuts(mode):
    lo, hi = C.c_int32(), C.c_int32()
    lib().t41rx_mode_default_cuts(mode, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


def make_params(**kw):
    """Reference defaults with the given fields replaced; a mode without explicit cut-offs takes the mode's preset
    (SetupMode, Filter.cpp:341-385)."""
    p = default_params()
    if "mode" in kw and "f_lo_cut" not in kw and "f_hi_cut" not in kw:
        kw["f_lo_cut"], kw["f_hi_cut"] = mode_default_cuts(kw["mode"])
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def design_tables(param_sequence):
    """Control path only (no GPU): tables of a fresh receiver after the given set_params calls."""
    arr = (Params * max(1, len(param_sequence)))(*param_sequence)
    t = Tables()
    _check(lib().t41rx_design_tables(arr, len(param_sequence), C.byref(t)), "t41rx_design_tables")
    return t.as_dict()


def smeter_dbm(audio_max_sq_ave, gain_correction=0.0, rf_gain=1, rf_gain_all_bands=1):
    """DrawSmeterBar()'s dBm reading from audioMaxSquaredAve (Display.cpp:959-981)."""
    return float(lib().t41rx_smeter_dbm(audio_max_sq_ave, gain_correction, rf_gain, rf_gain_all_bands))


def smeter_bar(dbm):
    """Pixels of the S-meter bar for a dBm reading (Display.cpp:995-998)."""
    return int(lib().t41rx_smeter_bar(dbm))


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class WavReader:
    """load_wav() / readWave() of the firmware (Utility.cpp:773-888) over t41rx_load_wav / t41rx_read_wave."""

    def __init__(self, path, num_samples):
        self._h = C.c_void_p()
        self.rc = lib().t41rx_load_wav(C.byref(self._h), os.fsencode(path), int(num_samples))

    @property
    def sample_rate(self):
        return int(lib().t41rx_wav_sample_rate(self._h)) if self._h else 0

    def read(self, size_buf):
        """float32 [size_buf] or None at the (reference's) end of file"""
        buf = np.empty(size_buf, np.float32)
        return buf if self._h and lib().t41rx_read_wave(self._h, _np_ptr(buf), size_buf) else None

    def close(self):
        if self._h:
            lib().t41rx_wav_close(self._h)
            self._h = C.c_void_p()


class Receiver:
    """A bank of n_streams virtual T41 receivers on one CUDA device."""

    def __init__(self, n_streams, device=0):
        self._h = C.c_void_p()
        self.n_streams = int(n_streams)
        self.device = int(device)
        _check(lib().t41rx_create(C.byref(self._h), self.n_streams, self.device), "t41rx_create")

    def close(self):
        if getattr(self, "_h", None):
            lib().t41rx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- parameters (the reference's globals) ----
    def set_params(self, p, first=0, count=None):
        count = self.n_streams - first if count is None else count
        _check(lib().t41rx_set_params(self._h, first, count, C.byref(p)), "t41rx_set_params")

    def set_params_each(self, plist, first=0):
        arr = (Params * len(plist))(*plist)
        _check(lib().t41rx_set_params_each(self._h, first, len(plist), arr), "t41rx_set_params_each")

    def get_params(self, stream):
        p = Params()
        _check(lib().t41rx_get_params(self._h, stream, C.byref(p)), "t41rx_get_params")
        return p

    def tables(self, stream):
        t = Tables()
        _check(lib().t41rx_get_tables(self._h, stream, C.byref(t)), "t41rx_get_tables")
        return t.as_dict()

    def debug(self, stream):
        d = Debug()
        _check(lib().t41rx_get_debug(self._h, stream, C.byref(d)), "t41rx_get_debug")
        return d

    # ---- ProcessIQData over host buffers ----
    def bind_audio_spectrum(self, ypixel_ptr, max_ave_ptr):
        """Raw pointers (host for process/process_q15, device for process_device) of the audio-spectrum by-product
        outputs: int32 [n_streams, n_rows, 270] and float32 [n_streams, n_rows]; None, None unbinds."""
        _check(lib().t41rx_bind_audio_spectrum(self._h, ypixel_ptr, max_ave_ptr), "t41rx_bind_audio_spectrum")

    def bind_control_frames(self, spec_frames_ptr, audio_frames_ptr):
        """Raw pointers of the control-app serial frames of the row-producing blocks: uint8 [n_streams, n_rows, 518]
        and uint8 [n_streams, n_rows, 270]; None, None unbinds."""
        _check(lib().t41rx_bind_control_frames(self._h, spec_frames_ptr, audio_frames_ptr), "t41rx_bind_control_frames")

    def _audio_spec_arrays(self, out, n_rows, want):
        """want_audio_spec: bind host arrays for every by-product of the row-producing blocks"""
        if not want or n_rows == 0:
            return False
        out.setdefault("audio_ypixel", np.zeros((self.n_streams, n_rows, AUDIO_SPEC_PIXELS), np.int32))
        out.setdefault("audio_max_sq_ave", np.zeros((self.n_streams, n_rows), np.float32))
        out.setdefault("spec_frames", np.zeros((self.n_streams, n_rows, SPEC_FRAME_BYTES), np.uint8))
        out.setdefault("audio_frames", np.zeros((self.n_streams, n_rows, AUDIO_SPEC_PIXELS), np.uint8))
        self.bind_audio_spectrum(_np_ptr(out["audio_ypixel"]), _np_ptr(out["audio_max_sq_ave"]))
        self.bind_control_frames(_np_ptr(out["spec_frames"]), _np_ptr(out["audio_frames"]))
        return True

    def process(self, iq, row_every=0, want_psk=False, flags=0, out=None, want_audio_spec=False):
        """iq: float32 [n_streams, n_blocks, 2048, 2] (host).  Returns dict of host arrays."""
        iq = np.ascontiguousarray(iq, dtype=np.float32)
        S, T = self.n_streams, iq.shape[1]
        if iq.shape != (S, T, BLOCK, 2):
            raise ValueError("iq must have shape [n_streams, n_blocks, 2048, 2]")
        n_rows = 0 if row_every <= 0 else (T + row_every - 1) // row_every
        if out is None:
            out = dict(audio=np.empty((S, T, BLOCK), np.float32),
                       spec=np.zeros((S, n_rows, SPECTRUM_RES), np.int16),
                       wf=np.zeros((S, n_rows, SPECTRUM_RES), np.uint16),
                       psk_bits=np.full((S, T), -1, np.int8) if want_psk else None,
                       psk_chars=np.zeros((S, T), np.uint8) if want_psk else None)
        bound = self._audio_spec_arrays(out, n_rows, want_audio_spec)
        try:
            _check(lib().t41rx_process(self._h, _np_ptr(iq), _np_ptr(out["audio"]), T, row_every,
                                       _np_ptr(out["spec"]) if n_rows else None,
                                       _np_ptr(out["wf"]) if n_rows else None,
                                       _np_ptr(out.get("psk_bits")), _np_ptr(out.get("psk_chars")), flags),
                   "t41rx_process")
        finally:
            if bound:
                self.bind_audio_spectrum(None, None)
                self.bind_control_frames(None, None)
        return out

    def process_q15(self, iq_q15, row_every=0, want_psk=False, flags=0, out=None, want_audio_spec=False):
        """The firmware's own block format: iq_q15 int16 [n_streams, n_blocks, 2048, 2] (host) in, audio int16
        [n_streams, n_blocks, 2048] out (arm_q15_to_float / arm_float_to_q15 run on the device)."""
        iq_q15 = np.ascontiguousarray(iq_q15, dtype=np.int16)
        S, T = self.n_streams, iq_q15.shape[1]
        if iq_q15.shape != (S, T, BLOCK, 2):
            raise ValueError("iq_q15 must have shape [n_streams, n_blocks, 2048, 2]")
        n_rows = 0 if row_every <= 0 else (T + row_every - 1) // row_every
        if out is None:
            out = dict(audio=np.empty((S, T, BLOCK), np.int16),
                       spec=np.zeros((S, n_rows, SPECTRUM_RES), np.int16),
                       wf=np.zeros((S, n_rows, SPECTRUM_RES), np.uint16),
                       psk_bits=np.full((S, T), -1, np.int8) if want_psk else None,
                       psk_chars=np.zeros((S, T), np.uint8) if want_psk else None)
        bound = self._audio_spec_arrays(out, n_rows, want_audio_spec)
        try:
            _check(lib().t41rx_process_q15(self._h, _np_ptr(iq_q15), _np_ptr(out["audio"]), T, row_every,
                                           _np_ptr(out["spec"]) if n_rows else None,
                                           _np_ptr(out["wf"]) if n_rows else None,
                                           _np_ptr(out.get("psk_bits")), _np_ptr(out.get("psk_chars")), flags),
                   "t41rx_process_q15")
        finally:
            if bound:
                self.bind_audio_spectrum(None, None)
                self.bind_control_frames(None, None)
        return out

    # ---- ProcessIQData over device buffers (raw pointers, e.g. torch.Tensor.data_ptr()) ----
    def process_device(self, iq_ptr, audio_ptr, n_blocks, row_every=0, spec_ptr=None, wf_ptr=None,
                       psk_bits_ptr=None, psk_chars_ptr=None, flags=0, cuda_stream=None):
        _check(lib().t41rx_process_device(self._h, iq_ptr, audio_ptr, n_blocks, row_every, spec_ptr, wf_ptr,
                                          psk_bits_ptr, psk_chars_ptr, flags, cuda_stream),
               "t41rx_process_device")

    def process_device_q15(self, iq16_ptr, audio16_ptr, n_blocks, row_every=0, spec_ptr=None, wf_ptr=None,
                           psk_bits_ptr=None, psk_chars_ptr=None, flags=0, cuda_stream=None):
        """process_device on q15 blocks resident in HBM (int16 [S, T, 2048, 2] in, int16 [S, T, 2048] out)"""
        _check(lib().t41rx_process_device_q15(self._h, iq16_ptr, audio16_ptr, n_blocks, row_every, spec_ptr, wf_ptr,
                                              psk_bits_ptr, psk_chars_ptr, flags, cuda_stream),
               "t41rx_process_device_q15")

    def synchronize(self):
        _check(lib().t41rx_synchronize(self._h), "t41rx_synchronize")

    def kernel_launches(self):
        return int(lib().t41rx_kernel_launches(self._h))

    def stream_kernel_times(self, max_n=32):
        """CUDA-event durations (ms) of the most recent t41rx_stream_rx_kernel launches, oldest first."""
        buf = (C.c_float * max_n)()
        n = lib().t41rx_stream_kernel_times(self._h, buf, max_n)
        if n < 0:
            _check(n, "t41rx_stream_kernel_times")
        return [float(buf[i]) for i in range(n)]

    def last_kernel_ms(self):
        ms = C.c_float()
        _check(lib().t41rx_last_kernel_ms(self._h, C.byref(ms)), "t41rx_last_kernel_ms")
        return float(ms.value)


def _check_multi(rc, what):
    if rc != 0:
        raise T41RxError("%s failed (%d): %s" % (what, rc, lib().t41rx_multi_last_error().decode()))


class MultiReceiver:
    """A bank of n_streams receivers sharded over several CUDA devices in ONE process (t41rx_create_multi): contiguous
    receiver ranges, one host thread per device inside every call, no inter-GPU traffic on the hot path."""

    def __init__(self, n_streams, devices):
        self._h = C.c_void_p()
        self.n_streams = int(n_streams)
        self.devices = [int(d) for d in devices]
        arr = (C.c_int * len(self.devices))(*self.devices)
        _check_multi(lib().t41rx_create_multi(C.byref(self._h), self.n_streams, arr, len(self.devices)), "t41rx_create_multi")

    def close(self):
        if getattr(self, "_h", None):
            lib().t41rx_destroy_multi(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def shards(self):
        """[(device, first, count)] of every shard"""
        out = []
        for g in range(lib().t41rx_multi_num_devices(self._h)):
            d, f, c = C.c_int(), C.c_int(), C.c_int()
            _check_multi(lib().t41rx_multi_shard(self._h, g, C.byref(d), C.byref(f), C.byref(c), None), "t41rx_multi_shard")
            out.append((d.value, f.value, c.value))
        return out

    def set_params_each(self, plist, first=0):
        arr = (Params * len(plist))(*plist)
        _check_multi(lib().t41rx_multi_set_params_each(self._h, first, len(plist), arr), "t41rx_multi_set_params_each")

    def set_params(self, p, first=0, count=None):
        count = self.n_streams - first if count is None else count
        _check_multi(lib().t41rx_multi_set_params(self._h, first, count, C.byref(p)), "t41rx_multi_set_params")

    def debug(self, stream):
        d = Debug()
        _check_multi(lib().t41rx_multi_get_debug(self._h, stream, C.byref(d)), "t41rx_multi_get_debug")
        return d

    def _out(self, T, row_every, want_psk, dtype):
        S = self.n_streams
        n_rows = 0 if row_every <= 0 else (T + row_every - 1) // row_every
        return n_rows, dict(audio=np.empty((S, T, BLOCK), dtype),
                            spec=np.zeros((S, n_rows, SPECTRUM_RES), np.int16),
                            wf=np.zeros((S, n_rows, SPECTRUM_RES), np.uint16),
                            psk_bits=np.full((S, T), -1, np.int8) if want_psk else None,
                            psk_chars=np.zeros((S, T), np.uint8) if want_psk else None)

    def process(self, iq, row_every=0, want_psk=False, flags=0):
        iq = np.ascontiguousarray(iq, dtype=np.float32)
        T = iq.shape[1]
        n_rows, out = self._out(T, row_every, want_psk, np.float32)
        _check_multi(lib().t41rx_multi_process(self._h, _np_ptr(iq), _np_ptr(out["audio"]), T, row_every,
                                               _np_ptr(out["spec"]) if n_rows else None, _np_ptr(out["wf"]) if n_rows else None,
                                               _np_ptr(out["psk_bits"]), _np_ptr(out["psk_chars"]), flags), "t41rx_multi_process")
        return out

    def process_q15(self, iq16, row_every=0, want_psk=False, flags=0):
        iq16 = np.ascontiguousarray(iq16, dtype=np.int16)
        T = iq16.shape[1]
        n_rows, out = self._out(T, row_every, want_psk, np.int16)
        _check_multi(lib().t41rx_multi_process_q15(self._h, _np_ptr(iq16), _np_ptr(out["audio"]), T, row_every,
                                                   _np_ptr(out["spec"]) if n_rows else None, _np_ptr(out["wf"]) if n_rows else None,
                                                   _np_ptr(out["psk_bits"]), _np_ptr(out["psk_chars"]), flags),
                     "t41rx_multi_process_q15")
        return out

    def process_device(self, iq_ptrs, audio_ptrs, n_blocks, row_every=0, spec_ptrs=None, wf_ptrs=None, flags=0):
        n = len(self.devices)
        arr = lambda ps: (C.c_void_p * n)(*ps) if ps is not None else None      # noqa: E731
        _check_multi(lib().t41rx_multi_process_device(self._h, arr(iq_ptrs), arr(audio_ptrs), n_blocks, row_every,
                                                      arr(spec_ptrs), arr(wf_ptrs), flags), "t41rx_multi_process_device")

    def synchronize(self):
        _check_multi(lib().t41rx_multi_synchronize(self._h), "t41rx_multi_synchronize")

    def gather_rows(self, row_ptrs, bytes_per_receiver, dst_ptr):
        """row buffers of the shards (device pointers) -> dst on the first device; returns True when NCCL carried it"""
        n = len(self.devices)
        used = C.c_int(0)
        _check_multi(lib().t41rx_multi_gather_rows(self._h, (C.c_void_p * n)(*row_ptrs), bytes_per_receiver, dst_ptr,
                                                   C.byref(used)), "t41rx_multi_gather_rows")
        return bool(used.value)


def chan_taps(n_channels):
    """The channelizer's prototype low-pass (float32 [10 * n_channels]); host only."""
    taps = np.empty(CHAN_TAPS_PER_BRANCH * int(n_channels), np.float32)
    _check(lib().t41rx_chan_taps(int(n_channels), taps.ctypes.data_as(C.POINTER(C.c_float))), "t41rx_chan_taps")
    return taps


def chan_centre(n_channels, channel):
    """Centre of a channel relative to the capture's centre (Hz)."""
    return (channel if channel < n_channels // 2 else channel - n_channels) * CHAN_SPACING


def chan_tune(n_channels, mode, offset_hz):
    """(channel, nco_freq) that put a receiver's carrier / dial point at offset_hz from the capture's centre; host only."""
    ch, nco = C.c_int32(), C.c_int32()
    _check(lib().t41rx_chan_tune(int(n_channels), int(mode), float(offset_hz), C.byref(ch), C.byref(nco)),
           "t41rx_chan_tune")
    return ch.value, nco.value


def chan_place(n_channels, mode, offset_hz):
    """(channel, shift, nco_freq) that put a receiver's carrier / dial point at offset_hz from the capture's centre with
    fine tuning: the receiver is mapped to channel, rotated by shift (Channelizer.set_shift) and runs at nco_freq, the
    chain's best operating point (0); host only."""
    ch, shift, nco = C.c_int32(), C.c_int32(), C.c_int32()
    _check(lib().t41rx_chan_place(int(n_channels), int(mode), float(offset_hz), C.byref(ch), C.byref(shift),
                                  C.byref(nco)), "t41rx_chan_place")
    return ch.value, shift.value, nco.value


def chan_centre_real(channel):
    """Centre of a real channelizer's channel (Hz from 0)."""
    return channel * CHAN_SPACING


def chan_tune_real(n_channels, mode, freq_hz):
    """chan_tune for a real capture (n_channels 128, 800, 1024 or 1280): freq_hz absolute, in [0, Fs/2]; host only."""
    ch, nco = C.c_int32(), C.c_int32()
    _check(lib().t41rx_chan_tune_real(int(n_channels), int(mode), float(freq_hz), C.byref(ch), C.byref(nco)),
           "t41rx_chan_tune_real")
    return ch.value, nco.value


def chan_place_real(n_channels, mode, freq_hz):
    """chan_place for a real capture (n_channels 128, 800, 1024 or 1280): freq_hz absolute, in [0, Fs/2]; host only."""
    ch, shift, nco = C.c_int32(), C.c_int32(), C.c_int32()
    _check(lib().t41rx_chan_place_real(int(n_channels), int(mode), float(freq_hz), C.byref(ch), C.byref(shift),
                                       C.byref(nco)), "t41rx_chan_place_real")
    return ch.value, shift.value, nco.value


class Channelizer:
    """Polyphase channelizer on one CUDA device: a wideband capture at n_channels x 96 kS/s in, the iq blocks of
    n_receivers receivers out (t41rx_process_device's layout).  Device pointers, e.g. torch.Tensor.data_ptr().
    real=True: an int16 real capture (n_channels 128, 800, 1024 or 1280: 12.288, 76.8, 98.304 or 122.88 MS/s; channels
    0 ... n_channels / 2); q15=True: a complex capture of interleaved int16 (I, Q) pairs, x = (I + jQ) / 32768
    (n_channels 64, 320, 512 or 640: 6.144, 30.72, 49.152 or 61.44 MS/s); else complex float (the same n_channels).
    n_inputs = 2 ... 4: a diversity channelizer (DESIGN §3.11) on that many coherent captures of the kind, receiver r
    getting rot_r(m) sum_a w[r][a] z^(a)_k[m] with its own weights (set_weights; default: input 0 alone)."""

    def __init__(self, n_channels, n_receivers, device=0, real=False, q15=False, n_inputs=1):
        if real and q15:
            raise ValueError("Channelizer: real and q15 are different capture kinds; pass at most one")
        if not isinstance(n_inputs, (int, np.integer)) or not 1 <= n_inputs <= CHAN_MAX_INPUTS:
            raise ValueError("Channelizer: n_inputs must be 1 (one capture) or 2 ... %d (diversity), not %r" % (
                CHAN_MAX_INPUTS, n_inputs))
        self._h = C.c_void_p()
        self.n_channels = int(n_channels)
        self.n_receivers = int(n_receivers)
        self.device = int(device)
        self.real = bool(real)
        self.q15 = bool(q15)
        self.n_inputs = int(n_inputs)
        if self.n_inputs > 1:
            self._create, self._process = "t41rx_chan_create_diversity", "t41rx_chan_process_device_diversity"
            kind = CHAN_REAL if self.real else CHAN_Q15 if self.q15 else CHAN_FLOAT
            _check(lib().t41rx_chan_create_diversity(C.byref(self._h), kind, self.n_channels, self.n_inputs,
                                                     self.n_receivers, self.device), self._create)
            return
        self._create, self._process = (("t41rx_chan_create_real", "t41rx_chan_process_device_real") if self.real else
                                       ("t41rx_chan_create_q15", "t41rx_chan_process_device_q15") if self.q15 else
                                       ("t41rx_chan_create", "t41rx_chan_process_device"))
        _check(getattr(lib(), self._create)(C.byref(self._h), self.n_channels, self.n_receivers, self.device),
               self._create)

    def close(self):
        if getattr(self, "_h", None):
            lib().t41rx_chan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_map(self, channels, first=0):
        """receivers first, first + 1, ... take channels[i] (-1: not written); effective from the next call"""
        arr = np.ascontiguousarray(channels, dtype=np.int32)
        _check(lib().t41rx_chan_set_map(self._h, int(first), int(arr.size), arr.ctypes.data_as(C.POINTER(C.c_int32))),
               "t41rx_chan_set_map")

    def set_shift(self, shifts, first=0):
        """receivers first, first + 1, ... rotated up by shifts[i] Hz (|shift| < 192000; 0 at creation); effective from
        the next call, with continuous phase"""
        arr = np.ascontiguousarray(shifts, dtype=np.int32)
        _check(lib().t41rx_chan_set_shift(self._h, int(first), int(arr.size), arr.ctypes.data_as(C.POINTER(C.c_int32))),
               "t41rx_chan_set_shift")

    def set_weights(self, w, first=0):
        """diversity: receivers first, first + 1, ... take the complex weights w[i] (array [count, n_inputs]), applied to
        each input's channel as delivered (after the channelizer's conjugate): an input-1 copy c x of an interferer x on
        input 0 is nulled by w[i][1] = -w[i][0] / conj(c).  Effective from the next call, in a step (no ramp)"""
        w = np.asarray(w, dtype=np.complex128)
        if w.ndim != 2 or w.shape[1] != self.n_inputs:
            raise ValueError("Channelizer.set_weights: w must be [count, %d], not %s" % (self.n_inputs, w.shape))
        arr = np.ascontiguousarray(np.stack([w.real, w.imag], axis=-1), dtype=np.float32)
        _check(lib().t41rx_chan_set_weights(self._h, int(first), int(w.shape[0]), arr.ctypes.data_as(C.POINTER(C.c_float))),
               "t41rx_chan_set_weights")

    def set_image(self, coef, first=0):
        """image correction (DESIGN §3.12, complex single-input channelizers): channels first, first + 1, ... take the
        complex coefficients coef[i], receivers on channel k getting z_k + c_k conj(z_(M - k) mod M) (0 at creation: no
        correction).  A frequency-independent imbalance x = mu s + nu conj(s) is removed by c_k = -conj(nu) / mu on every
        channel.  Effective from the next call"""
        c = np.atleast_1d(np.asarray(coef, dtype=np.complex128))
        arr = np.ascontiguousarray(np.stack([c.real, c.imag], axis=-1), dtype=np.float32)
        _check(lib().t41rx_chan_set_image(self._h, int(first), int(c.size), arr.ctypes.data_as(C.POINTER(C.c_float))),
               "t41rx_chan_set_image")

    def get_image(self):
        """all n_channels image coefficients (complex64), including what tracking has made of them"""
        arr = np.empty((self.n_channels, 2), np.float32)
        _check(lib().t41rx_chan_get_image(self._h, arr.ctypes.data_as(C.POINTER(C.c_float))), "t41rx_chan_get_image")
        return arr[:, 0] + 1j * arr[:, 1]

    def track_image(self, on=True, dominance_db=20.0):
        """image tracking on or off from the next call: each call measures every mirror pair and corrects the weak side
        of a pair whose other side is dominance_db (3 ... 60) or more stronger, for the next call"""
        _check(lib().t41rx_chan_track_image(self._h, int(bool(on)), float(dominance_db)), "t41rx_chan_track_image")

    def image_stats(self):
        """float64 [n_channels / 2 + 1, 4]: (Re A, Im A, P_k, P_kbar) of pair k from the last call with tracking on"""
        out = np.empty((self.n_channels // 2 + 1, 4), np.float64)
        _check(lib().t41rx_chan_image_stats(self._h, out.ctypes.data_as(C.POINTER(C.c_double))), "t41rx_chan_image_stats")
        return out

    def process_device(self, capture_ptr, iq_ptr, n_blocks, stream=None):
        """capture float32 [n_blocks * 2048 * n_channels / 2, 2] (real: int16 [n_blocks * 2048 * n_channels / 2];
        q15: int16 [n_blocks * 2048 * n_channels / 2, 2]; both 16-byte aligned) -> iq float32 [n_receivers, n_blocks,
        2048, 2].  Diversity: capture_ptr is a list of n_inputs such pointers, input 0 first"""
        if self.n_inputs > 1:
            ptrs = list(capture_ptr) if isinstance(capture_ptr, (list, tuple)) else None
            if ptrs is None or len(ptrs) != self.n_inputs:
                raise ValueError("Channelizer.process_device: a diversity channelizer takes a list of %d capture "
                                 "pointers" % self.n_inputs)
            _check(lib().t41rx_chan_process_device_diversity(self._h, (C.c_void_p * self.n_inputs)(*ptrs), iq_ptr,
                                                             int(n_blocks), stream), self._process)
            return
        _check(getattr(lib(), self._process)(self._h, capture_ptr, iq_ptr, int(n_blocks), stream), self._process)

    def synchronize(self):
        _check(lib().t41rx_chan_synchronize(self._h), "t41rx_chan_synchronize")
