"""GPU parity of the host-buffer (end-to-end) entry points that bench.py's e2e legs time: the batch demodulator with the
samples in host memory (time-chunk copy pipeline, cf32 and CS16) and the batch modulator writing to host memory (frame-group
pipeline).  Payloads / frames must equal the device-resident path's and the oracle's."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"
FS, RS = 10_000_000, 5_000_000
ALPHA = float(np.float32(0.4))


def _bursts(gpu, C, n_payload, seed=77):
    """C impaired bursts generated on the device (the bench's generator), returned on the host with their payloads."""
    import torch
    mod = gpu.QPSKModulator(FS, RS, ALPHA, 10, True, TSC)
    pay = torch.empty((C, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(seed, 0, C, n_payload, pay.data_ptr(), 0)
    ff = mod.frame_floats(n_payload, b"S", b"E")
    tx = torch.empty((C, ff), dtype=torch.float32, device="cuda")
    mod.modulate_frames_dev(pay.data_ptr(), n_payload, C, b"S", b"E", tx.data_ptr(), ff, 0)
    ch = gpu.SimChannel(100e6, 100e6, FS, 1, 1, noise_dbfs=-40.0, mode=1, seed=seed, channels=C, first_channel=0)
    rx = torch.empty((C, ff), dtype=torch.float32, device="cuda")
    ch.apply_dev(tx.data_ptr(), ff, ff, rx.data_ptr(), ff, 0)
    torch.cuda.synchronize()
    return rx, pay.cpu().numpy()


@pytest.mark.parametrize("use_fll", [False, True])
def test_host_batch_demod_pipeline_matches_device_path_and_oracle(gpu, orc, use_fll):
    import torch
    C, n_payload = 600, 512                                     # 600 x 4196 samples x 8 B = 20 MB: several copy chunks
    rx, pay = _bursts(gpu, C, n_payload)
    ff = rx.shape[1]
    host = rx.cpu().numpy()
    kw = dict(tsc=TSC, use_fll=use_fll, channels=C, max_frame_bytes=2048)
    gh = gpu.QPSKDeModulator(FS, RS, ALPHA, 10, **kw)
    gdv = gpu.QPSKDeModulator(FS, RS, ALPHA, 10, **kw)
    payload = torch.zeros((C, 1024), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros(C, dtype=torch.int64, device="cuda")
    for rep in range(2):                                        # second burst: state carried
        got = gh.DeModulateBytes(host, b"S", b"E")
        gdv.demod_bytes_dev(rx.data_ptr(), ff, ff, b"S", b"E", payload.data_ptr(), 1024, nbytes.data_ptr())
        torch.cuda.synchronize()
        pd, nd = payload.cpu().numpy(), nbytes.cpu().numpy()
        for c in range(C):
            assert got[c] == pd[c, : nd[c]].tobytes(), (rep, c)
    assert sum(g == pay[c].tobytes() for c, g in enumerate(got)) > 0      # one-byte markers: many frames end early on a false 'E'
    for c in (0, 31, 32, 299, C - 1):
        od = orc.QPSKDeModulator(FS, RS, ALPHA, 10, tsc=TSC, use_fll=use_fll)
        for rep in range(2):
            w = od.DeModulateBytes(host[c], b"S", b"E")
        assert got[c] == w, c
    # bits and packed bits from the same host rows, through the same copy chunks, against the device-resident path
    gb, gp, gdb = (gpu.QPSKDeModulator(FS, RS, ALPHA, 10, **kw) for _ in range(3))
    cap = gdb.bits_bound(ff)
    d_bits = torch.zeros((C, cap), dtype=torch.uint8, device="cuda")
    d_nb = torch.zeros(C, dtype=torch.int64, device="cuda")
    for rep in range(2):
        bits, packed = gb.DeModulate(host), gp.DeModulatePacked(host)
        gdb.demod_bits_dev(rx.data_ptr(), ff, ff, d_bits.data_ptr(), cap, d_nb.data_ptr())
        torch.cuda.synchronize()
        db, dn = d_bits.cpu().numpy(), d_nb.cpu().numpy()
        for c in range(C):
            row = db[c, : dn[c]]
            assert bits[c] == (row + ord("0")).tobytes().decode("ascii"), (rep, c)
            assert packed[c] == (np.packbits(row).tobytes(), int(dn[c])), (rep, c)
    for c in (0, 299, C - 1):
        od = orc.QPSKDeModulator(FS, RS, ALPHA, 10, tsc=TSC, use_fll=use_fll)
        for rep in range(2):
            w = od.DeModulate(host[c])
        assert bits[c] == w and len(w) > 1000, c


def test_cs16_ingest_equals_cf32_of_the_same_values(gpu, orc):
    C, n_payload = 300, 512
    rx, pay = _bursts(gpu, C, n_payload, seed=5)
    host = rx.cpu().numpy()
    peak = float(np.abs(host).max())
    scale = float(np.float32(peak / 30000.0))
    x16 = np.clip(np.round(host / scale), -32768, 32767).astype(np.int16)
    xf = (x16.astype(np.float32) * np.float32(scale)).astype(np.float32)          # exactly what the device widens to
    kw = dict(tsc=TSC, channels=C, max_frame_bytes=2048)
    g16 = gpu.QPSKDeModulator(FS, RS, ALPHA, 10, **kw)
    g32 = gpu.QPSKDeModulator(FS, RS, ALPHA, 10, **kw)
    for rep in range(2):
        a = g16.DeModulateBytesCs16(x16, scale, b"S", b"E")
        b = g32.DeModulateBytes(xf, b"S", b"E")
        assert a == b, rep
    od = orc.QPSKDeModulator(FS, RS, ALPHA, 10, tsc=TSC)
    for rep in range(2):
        w = od.DeModulateBytes(xf[7], b"S", b"E")
    assert a[7] == w
    # one radio stream (single channel, one copy chunk)
    g1 = gpu.QPSKDeModulator(FS, RS, ALPHA, 10, tsc=TSC)
    o1 = orc.QPSKDeModulator(FS, RS, ALPHA, 10, tsc=TSC)
    for rep in range(2):
        assert g1.DeModulateBytesCs16(x16[3], scale, b"S", b"E") == o1.DeModulateBytes(xf[3], b"S", b"E")


def test_host_batch_modulator_pipeline(gpu, orc):
    import torch
    frames, n_payload = 700, 6000                               # 700 frames x 770 KB of samples: several frame groups
    m = gpu.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    rng = np.random.default_rng(2)
    pay = rng.integers(0, 256, (frames, n_payload), dtype=np.uint8)
    out = m.ModulateFrames(pay, b"START", b"END")
    ff = m.frame_floats(n_payload, b"START", b"END")
    assert out.shape == (frames, ff)
    dp = torch.from_numpy(pay).cuda()
    dout = torch.zeros((frames, ff), dtype=torch.float32, device="cuda")
    m.modulate_frames_dev(dp.data_ptr(), n_payload, frames, b"START", b"END", dout.data_ptr(), ff)
    torch.cuda.synchronize()
    assert np.array_equal(out.view(np.uint32), dout.cpu().numpy().view(np.uint32))
    om = orc.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    for f in (0, 350, frames - 1):
        w = om.ModulateBytes(pay[f].tobytes(), b"START", b"END")
        assert w.size == ff and float(np.abs(out[f] - w).max()) <= 1e-5 * float(np.abs(w).max())
    # padded rows: a stride wider than the frame leaves the padding untouched
    wide = np.full((frames, ff + 6), 7.0, np.float32)
    m.ModulateFrames(pay, b"START", b"END", out=wide)
    assert np.array_equal(wide[:, :ff], out) and (wide[:, ff:] == 7.0).all()
