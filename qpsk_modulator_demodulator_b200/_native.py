"""ctypes binding of libqpskcuda.so (include/qpskcuda.h).  No fallback: if the library is missing or
cannot be loaded, importing a compute entry point raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libqpskcuda.so")

OK = 0
ERR_NULL, ERR_ARG, ERR_RANGE, ERR_CUDA, ERR_NOMEM, ERR_CAPACITY, ERR_UNSUPPORTED, ERR_NO_DEVICE = -1, -2, -3, -4, -5, -6, -7, -8
FIR_FAST, FIR_EXACT, FIR_FMA, FIR_SPLIT = 0, 1, 2, 3


class ArgumentNullException(ValueError):
    pass


class ArgumentException(ValueError):
    pass


class ArgumentOutOfRangeException(ValueError):
    pass


class QpskCudaError(RuntimeError):
    pass


f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int)
u32p = C.POINTER(C.c_uint32)
i64p = C.POINTER(C.c_int64)
vpp = C.POINTER(C.c_void_p)


class ChanParams(C.Structure):
    _fields_ = [
        ("tx_freq_hz", C.c_double), ("rx_freq_hz", C.c_double), ("sample_rate_hz", C.c_double),
        ("tx_ppm", C.c_double), ("rx_ppm", C.c_double), ("tx_phase0", C.c_double), ("rx_phase0", C.c_double),
        ("noise_dbfs", C.c_float), ("mode", C.c_int), ("n_paths", C.c_int),
        ("path_gain_iq", C.c_float * 8), ("path_delay", C.c_int * 4), ("seed", C.c_uint64),
    ]


class ChainParams(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int), ("symbol_rate", C.c_int), ("rrc_span", C.c_double), ("rrc_alpha", C.c_double),
        ("fll_sps", C.c_float), ("fll_rolloff", C.c_float), ("fll_size", C.c_int), ("fll_bw", C.c_float),
        ("mm_sps", C.c_double), ("mm_kp", C.c_double), ("mm_ki", C.c_double),
        ("costas_sample_rate", C.c_double), ("costas_bw_hz", C.c_double), ("costas_damping", C.c_double),
    ]


def _signatures():
    i, i64, u64, d, f, vp, cp = C.c_int, C.c_int64, C.c_uint64, C.c_double, C.c_float, C.c_void_p, C.c_char_p
    return {
        "qpsk_version": (i, []),
        "qpsk_build_id": (cp, []),
        "qpsk_strerror": (cp, [i]),
        "qpsk_last_cuda_error": (cp, []),
        "qpsk_device_count": (i, [i32p]),
        "qpsk_set_device": (i, [i]),
        "qpsk_device_info": (i, [i32p, i32p, i32p, i64p]),
        "qpsk_host_alloc": (i, [vpp, i64]),
        "qpsk_host_free": (i, [vp]),
        "qpsk_host_register": (i, [vp, i64]),
        "qpsk_host_unregister": (i, [vp]),
        "qpsk_launch_count": (i64, []),
        "qpsk_launch_count_reset": (None, []),
        "qpsk_rrc_taps": (i, [d, d, i, i, f64p, i, i32p]),
        "qpsk_fir_create": (i, [f32p, i, vpp]),
        "qpsk_fir_create_batch": (i, [f32p, i, i, vpp]),
        "qpsk_fir_destroy": (i, [vp]),
        "qpsk_fir_reset": (i, [vp]),
        "qpsk_fir_set_mode": (i, [vp, i]),
        "qpsk_fir_num_taps": (i, [vp, i32p]),
        "qpsk_fir_last_kernel": (i, [vp, cp, i]),
        "qpsk_fir_filter": (i, [vp, vp, vp, i64, i64]),
        "qpsk_fir_fft_filter": (i, [vp, vp, vp, i64]),
        "qpsk_fir_filter_dev": (i, [vp, vp, vp, i64, i64, i64, vp]),
        "qpsk_fir_fft_filter_dev": (i, [vp, vp, vp, i64, i64, i64, vp]),
        "qpsk_fir_decimate": (i, [vp, vp, i64, i, vp, i64, i64p]),
        "qpsk_fir_decimate_dev": (i, [vp, vp, i64, i64, i, vp, i64, i64, i64p, vp]),
        "qpsk_fir_get_state": (i, [vp, f32p, i64]),
        "qpsk_fir_set_state": (i, [vp, f32p, i64]),
        "qpsk_fll_design": (i, [f, f, i, f32p, f32p]),
        "qpsk_fll_create": (i, [f, f, i, f, vpp]),
        "qpsk_fll_create_batch": (i, [f, f, i, f, i, vpp]),
        "qpsk_fll_destroy": (i, [vp]),
        "qpsk_fll_process": (i, [vp, vp, vp, i64, i64]),
        "qpsk_fll_process_dev": (i, [vp, vp, vp, i64, i64, i64, vp]),
        "qpsk_fll_get_state": (i, [vp, f32p, f32p]),
        "qpsk_fll_set_state": (i, [vp, f32p, f32p]),
        "qpsk_mm_create": (i, [d, d, d, vpp]),
        "qpsk_mm_create_batch": (i, [d, d, d, i, vpp]),
        "qpsk_mm_destroy": (i, [vp]),
        "qpsk_mm_process": (i, [vp, vp, i64, vp, i64, i32p]),
        "qpsk_mm_process_dev": (i, [vp, vp, i64, i64, vp, i64, i64, vp, vp]),
        "qpsk_mm_get_state": (i, [vp, i32p, f64p, f64p, i32p]),
        "qpsk_mm_gains_from_bw": (i, [d, f64p, f64p]),
        "qpsk_costas_create": (i, [d, d, d, vpp]),
        "qpsk_costas_create_batch": (i, [d, d, d, i, vpp]),
        "qpsk_costas_destroy": (i, [vp]),
        "qpsk_costas_process": (i, [vp, vp, vp, i64, i64]),
        "qpsk_costas_process_dev": (i, [vp, vp, vp, i64, i64, i64, vp, vp]),
        "qpsk_costas_get_state": (i, [vp, f64p, f64p]),
        "qpsk_eq_create": (i, [i, f, f, vpp]),
        "qpsk_eq_create_batch": (i, [i, f, f, i, vpp]),
        "qpsk_eq_create_fractional": (i, [i, f, f, i, i, vpp]),
        "qpsk_eq_destroy": (i, [vp]),
        "qpsk_eq_reset": (i, [vp]),
        "qpsk_eq_process": (i, [vp, vp, vp, i64, i64]),
        "qpsk_eq_process_dev": (i, [vp, vp, vp, i64, i64, i64, vp, vp]),
        "qpsk_eq_get_taps": (i, [vp, f32p, i64]),
        "qpsk_eq_set_taps": (i, [vp, f32p, i64]),
        "qpsk_pfb_taps": (i, [i, i, d, d, f64p, i, i32p]),
        "qpsk_pfb_create": (i, [f32p, i, i, vpp]),
        "qpsk_pfb_destroy": (i, [vp]),
        "qpsk_pfb_reset": (i, [vp]),
        "qpsk_pfb_process": (i, [vp, vp, i64, vp, i64, i64p]),
        "qpsk_pfb_process_dev": (i, [vp, vp, i64, vp, i64, i64p, vp]),
        "qpsk_ddc_create": (i, [f32p, i, f64p, i, i, vpp]),
        "qpsk_ddc_destroy": (i, [vp]),
        "qpsk_ddc_reset": (i, [vp]),
        "qpsk_ddc_process": (i, [vp, vp, i64, vp, i64, i64p]),
        "qpsk_ddc_process_dev": (i, [vp, vp, i64, vp, i64, i64p, vp]),
        "qpsk_agc_create_batch": (i, [i, f, f, i, vpp]),
        "qpsk_agc_destroy": (i, [vp]),
        "qpsk_agc_reset": (i, [vp]),
        "qpsk_agc_process": (i, [vp, vp, vp, i64, i64]),
        "qpsk_agc_process_dev": (i, [vp, vp, vp, i64, i64, i64, vp]),
        "qpsk_agc_gain": (i, [vp, f32p, i64]),
        "qpsk_agc_gain_dev": (i, [vp, vp, vp]),
        "qpsk_resamp_create": (i, [f32p, i, i, i, i, vpp]),
        "qpsk_resamp_destroy": (i, [vp]),
        "qpsk_resamp_reset": (i, [vp]),
        "qpsk_resamp_process": (i, [vp, vp, i64, vp, i64, i64p]),
        "qpsk_resamp_process_dev": (i, [vp, vp, i64, i64, vp, i64, i64p, vp]),
        "qpsk_conv_create": (i, [i, vpp]),
        "qpsk_conv_destroy": (i, [vp]),
        "qpsk_conv_reset": (i, [vp]),
        "qpsk_conv_encode": (i, [vp, vp, i64, vp]),
        "qpsk_conv_encode_dev": (i, [vp, vp, i64, i64, vp, i64, vp]),
        "qpsk_viterbi_create": (i, [i, i, f, vpp]),
        "qpsk_viterbi_destroy": (i, [vp]),
        "qpsk_viterbi_reset": (i, [vp]),
        "qpsk_viterbi_bits_bound": (i, [vp, i64, i64p]),
        "qpsk_viterbi_decode_dev": (i, [vp, vp, i64, vp, vp, i64, vp, vp]),
        "qpsk_viterbi_flush_dev": (i, [vp, vp, i64, vp, vp, i64, vp, vp]),
        "qpsk_viterbi_decode": (i, [vp, vp, i64, vp, vp, i64, vp]),
        "qpsk_viterbi_flush": (i, [vp, vp, i64, vp, vp, i64, vp]),
        "qpsk_fsync_create": (i, [i, i, f, vp, i, i, i, i, vpp]),
        "qpsk_fsync_destroy": (i, [vp]),
        "qpsk_fsync_reset": (i, [vp]),
        "qpsk_fsync_shape": (i, [vp, i32p, i32p, i32p, i32p]),
        "qpsk_fsync_slots_bound": (i, [vp, i64, i64p]),
        "qpsk_fsync_process_dev": (i, [vp, vp, i64, vp, i, vp, i64, vp, vp, vp, vp]),
        "qpsk_fsync_process": (i, [vp, vp, i64, vp, i, vp, i64, vp, vp, vp, i64p]),
        "qpsk_rs_create": (i, [i, i, i, vpp]),
        "qpsk_rs_destroy": (i, [vp]),
        "qpsk_rs_encode": (i, [vp, vp, i64, vp]),
        "qpsk_rs_decode": (i, [vp, vp, i64, vp, vp]),
        "qpsk_rs_encode_dev": (i, [vp, vp, i64, i, i64, vp, i64, vp]),
        "qpsk_rs_decode_dev": (i, [vp, vp, i64, vp, i, vp, i64, vp, vp, i64, vp]),
        "qpsk_mod_create": (i, [i, i, d, i, i, cp, vpp]),
        "qpsk_mod_destroy": (i, [vp]),
        "qpsk_mod_taps": (i, [vp, f64p, i, i32p]),
        "qpsk_mod_modulate_bits": (i, [vp, cp, i64, i, vp, i64, i64p]),
        "qpsk_mod_modulate_packed": (i, [vp, vp, i64, i, vp, i64, i64p]),
        "qpsk_mod_modulate_bytes": (i, [vp, vp, i64, vp, i64, vp, i64, i, vp, i64, i64p]),
        "qpsk_mod_modulate_frames": (i, [vp, vp, i64, i, vp, i64, vp, i64, vp, i64, i64p]),
        "qpsk_mod_modulate_frames_dev": (i, [vp, vp, i64, i, vp, i64, vp, i64, vp, i64, i64p, vp]),
        "qpsk_demod_create": (i, [i, i, f, i, d, d, d, i, cp, i, i64, vpp]),
        "qpsk_demod_create_batch": (i, [i, i, f, i, d, d, d, i, cp, i, i64, i, vpp]),
        "qpsk_demod_destroy": (i, [vp]),
        "qpsk_demod_set_fir_mode": (i, [vp, i]),
        "qpsk_demod_set_equalizer": (i, [vp, i, f, f]),
        "qpsk_demod_equalizer_taps": (i, [vp, f32p, i64]),
        "qpsk_demod_set_fractional_equalizer": (i, [vp, i, f, f]),
        "qpsk_demod_fractional_equalizer_taps": (i, [vp, f32p, i64]),
        "qpsk_demod_set_agc": (i, [vp, i, f, f]),
        "qpsk_demod_bits": (i, [vp, vp, i64, vp, i64, vp]),
        "qpsk_demod_bits_packed": (i, [vp, vp, i64, vp, i64, vp]),
        "qpsk_demod_bytes": (i, [vp, vp, i64, vp, i64, vp, i64, vp, i64, vp]),
        "qpsk_demod_bytes_cs16": (i, [vp, vp, i64, f, vp, i64, vp, i64, vp, i64, vp]),
        "qpsk_demod_last_payload": (i, [vp, vp, i64, vp]),
        "qpsk_demod_frame_bits": (i, [vp, vp, i64, vp, vp, i64, vp, i64, vp, i64, vp]),
        "qpsk_demod_constellation": (i, [vp, vp, i64, vp, i64, vp]),
        "qpsk_demod_bits_dev": (i, [vp, vp, i64, i64, vp, i64, vp, vp]),
        "qpsk_demod_bits_bound": (i, [vp, i64, i64p]),
        "qpsk_demod_bytes_dev": (i, [vp, vp, i64, i64, vp, i64, vp, i64, vp, i64, vp, vp]),
        "qpsk_demod_constellation_dev": (i, [vp, vp, i64, i64, vp, i64, vp, vp]),
        "qpsk_demod_frame_bits_dev": (i, [vp, vp, i64, vp, vp, i64, vp, i64, vp, i64, vp, vp]),
        "qpsk_demod_loop_state": (i, [vp, f64p, f64p, f64p, f64p, f32p, f32p]),
        "qpsk_demod_in_frame": (i, [vp, i32p]),
        "qpsk_demod_channels": (i, [vp, i32p]),
        "qpsk_demod_device": (i, [vp, i32p]),
        "qpsk_stream_create": (i, [vp, i64, i64, i, vp, i64, vp, i64, vpp]),
        "qpsk_stream_destroy": (i, [vp]),
        "qpsk_stream_push": (i, [vp, vp, i64]),
        "qpsk_stream_push_cs16": (i, [vp, vp, i64, f]),
        "qpsk_stream_poll": (i, [vp, i, vp, i64, i64p, i32p]),
        "qpsk_stream_pending": (i, [vp, i64p, i64p]),
        "qpsk_stream_flush": (i, [vp]),
        "qpsk_cf32_to_cs16": (i, [vp, i64, vp, f32p]),
        "qpsk_cs16_to_cf32": (i, [vp, i64, f, vp]),
        "qpsk_cf32_to_cs16_dev": (i, [vp, i64, vp, vp, vp]),
        "qpsk_cs16_to_cf32_dev": (i, [vp, i64, f, vp, vp]),
        "qpsk_chain_default_params": (i, [C.POINTER(ChainParams)]),
        "qpsk_chain_create": (i, [C.POINTER(ChainParams), i, vpp]),
        "qpsk_chain_destroy": (i, [vp]),
        "qpsk_chain_set_fir_mode": (i, [vp, i]),
        "qpsk_chain_symbols_bound": (i, [vp, i64, i64p]),
        "qpsk_chain_process": (i, [vp, vp, i64, vp, vp, vp, i64, i32p]),
        "qpsk_chain_process_dev": (i, [vp, vp, i64, i64, vp, i64, vp, i64, vp, i64, vp, vp]),
        "qpsk_chain_loop_state": (i, [vp, f32p, f32p, f64p, f64p, f64p]),
        "qpsk_unpack_bits_dev": (i, [vp, i64, i64, i, vp, i64, vp]),
        "qpsk_chan_create": (i, [C.POINTER(ChanParams), i, i, vpp]),
        "qpsk_chan_destroy": (i, [vp]),
        "qpsk_chan_apply_dev": (i, [vp, vp, i64, i64, vp, i64, vp]),
        "qpsk_chan_apply": (i, [vp, vp, i64, vp]),
        "qpsk_fill_uniform_dev": (i, [u64, u64, i64, i64, vp, vp]),
        "qpsk_fill_bytes_dev": (i, [u64, i, i, i64, vp, vp]),
        "qpsk_pack_bits_dev": (i, [vp, i64, vp, i64, i, vp, i64, vp]),
        "qpsk_ber_count_dev": (i, [vp, i64, vp, vp, i64, i64, i, vp, vp]),
        "qpsk_measure_fma_peak": (i, [f64p]),
        "qpsk_comm_unique_id": (i, [vp, i]),
        "qpsk_comm_create": (i, [vp, i, i, vpp]),
        "qpsk_comm_destroy": (i, [vp]),
        "qpsk_comm_info": (i, [vp, i32p, i32p, i32p]),
        "qpsk_ber_gather_dev": (i, [vp, vp, i, i, vp, vp]),
        "qpsk_ber_gather": (i, [vp, vp, i, i, vp]),
    }


_lib = None


def lib() -> C.CDLL:
    """Load libqpskcuda.so.  Raises if it has not been built — there is no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise QpskCudaError(f"{LIB_PATH} is missing: run `python -m qpsk_modulator_demodulator_b200.build` "
                                "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _signatures().items():
            fn = getattr(L, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _check_stamp(L)
        _lib = L
    return _lib


def build_id() -> str:
    """Stamp of the loaded library (hash of the sources, header, nvcc flags and version it was compiled from)."""
    return lib().qpsk_build_id().decode()


def _check_stamp(L):
    """A library that travels with a source tree must be the build of THAT tree: file times do not survive the copy to
    the GPU box, so the stamp compiled into the library is compared with the hash of the sources next to it."""
    if os.environ.get("QPSK_SKIP_BUILD_CHECK") == "1" or not os.path.isdir(os.path.join(_HERE, "csrc")):
        return
    from . import build as _b
    try:
        want = _b.source_id()
    except RuntimeError:          # no nvcc: the tree cannot be rebuilt here, nothing to compare against
        return
    got = L.qpsk_build_id().decode()
    if got != want:
        raise QpskCudaError(f"{LIB_PATH} carries build stamp {got} but the sources next to it hash to {want}: stale library, "
                            "run `python -m qpsk_modulator_demodulator_b200.build`")


def declared_symbols():
    return sorted(_signatures().keys())


def check(st: int):
    if st == OK:
        return
    if st == ERR_NULL:
        raise ArgumentNullException(lib().qpsk_strerror(st).decode())
    if st == ERR_ARG:
        raise ArgumentException(lib().qpsk_strerror(st).decode())
    if st == ERR_RANGE:
        raise ArgumentOutOfRangeException(lib().qpsk_strerror(st).decode())
    msg = lib().qpsk_strerror(st).decode()
    if st in (ERR_CUDA, ERR_NOMEM, ERR_NO_DEVICE):
        msg += ": " + lib().qpsk_last_cuda_error().decode()
    raise QpskCudaError(f"status {st}: {msg}")
