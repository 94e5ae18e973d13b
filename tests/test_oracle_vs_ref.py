"""Pins the CPU oracle (oracle/srtb_oracle.cpp) against the reference's own operator/pipe headers, compiled through the
host shim (oracle/_ref/libsrtb_ref.so, see oracle/ref_shim/README.md). What the reference computed for the seeded
inputs below is stored in tests/golden/srtb_oracle_vs_ref.npz (tests/golden/make_golden.py writes it), so the test
needs nothing outside the repository: outputs compared bit for bit are stored as SHA-256 digests; outputs the SK and
average stages only zero are stored as their zero masks (plus the normalisation coefficient), rebuilt from the input
and checked against the digest of the reference's output; the whole-chain spectra as every 8th value. Bit-exact
wherever the reference's arithmetic order is fully specified, tolerance only where a reduction's order is the
runtime's choice."""
import functools
import hashlib
from pathlib import Path

import numpy as np
import pytest

GOLDEN = Path(__file__).resolve().parent / "golden" / "srtb_oracle_vs_ref.npz"
CHAIN_STRIDE = 8        # every 8th value of the whole-chain spectra is stored

UNPACK_BITS = [1, 2, 4, 8, -8, 16, -16, 32, 64]
WINDOWS = [0, 1, 2]
FFT_LOG2 = [1, 4, 10, 14]
S1_CASES = [(1 << 10, 16), ((1 << 14) + 3, 64), (1 << 18, 2048)]
S1_THRESHOLD, S1_FREQ_LIST = 1.5, "1100-1101, 1300.5-1302"
RANGE_STRINGS = ["11-12, 15-90, 233-235, 1176-1177", "", "1418-1422", "1-2-3, 5-6", " 7 - 8 ,9-10", "3-4,"]
MANUAL_CASES = [([(1418.0, 1422.0)], 1437.0, -64.0), ([(1422.0, 1418.0)], 1437.0, -64.0),
                ([(100.0, 200.0)], 1000.0, 500.0), ([(1400.0, 1600.0)], 1000.0, 500.0)]
DD_CASES = [(1 << 14, 1000.0, 500.0, 56.778), ((1 << 12) + 1, 1000.0, 400.0, 562.05),
            (1 << 16, 1437.0, -64.0, -478.80), (1 << 10, 1000.0, 500.0, 0.0)]
NSAMPS_CASES = [(1 << 26, 1 << 11, 1000.0, 500.0, 1e9, 5.0, True), (1 << 24, 1 << 11, 1000.0, 500.0, 1e9, 56.778, True),
                (1 << 30, 1 << 11, 1437.0, -64.0, 128e6, -478.80, True),
                (1 << 30, 1 << 11, 1437.0, -64.0, 128e6, -478.80, False),
                (1 << 28, 1 << 15, 1000.0, 500.0, 1e9, 100.0, True), (1 << 28, 1 << 15, 1000.0, 500.0, 1e9, 1.0, True)]
S2_THRESHOLD = 1.05
DETECT_CASES = [(16, 256, 16, False), (64, 2048, 256, False), (32, 1000, 64, True)]
DETECT_PARAMS = dict(f_low=1000.0, bw=500.0, fs=1e9, dm=0.005, snr=6.0, chan_thr=0.9)
CHAIN_CASES = [(14, 16, 0.0, -8), (15, 32, 0.02, -8), (14, 8, 0.0, 2)]
CHAIN_PARAMS = dict(f_low=1000.0, bw=500.0, fs=1e9, avg_thr=5.0, sk_thr=1.3, snr=6.0, chan_thr=0.9, maxbox=32,
                    freq_list="1200-1201")
SK_CASES = [(256, 64), (1000, 48)]
SK_THRESHOLD = 1.1
DETECT_V1_CASES = [(512, 64, 32), (1000, 128, 256)]
DETECT_V1_PARAMS = dict(sk_thr=1.4, snr=5.0, chan_thr=0.9)


def digest(a) -> str:
    """SHA-256 of an array's dtype, shape and bytes: equal digests <=> np.array_equal for arrays of one dtype"""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


@functools.lru_cache(maxsize=None)
def golden():
    with np.load(GOLDEN) as g:
        return {k: g[k] for k in g.files}


def g_str(key):
    return str(golden()[key])


def rel(a, b):
    a, b = np.asarray(a).astype(np.complex128).ravel(), np.asarray(b).astype(np.complex128).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


# --- seeded inputs (tests/golden/make_golden.py feeds the same ones to the reference)
def unpack_input(bits):
    rng = np.random.default_rng(abs(bits))
    nbytes = 1 << 12
    raw = (rng.standard_normal(nbytes // 4).astype(np.float32).view(np.uint8) if bits == 32 else
           rng.standard_normal(nbytes // 8).view(np.uint8) if bits == 64 else rng.integers(0, 256, nbytes, dtype=np.uint8))
    return raw, nbytes * 8 // abs(bits)


def multistream_input():
    return np.random.default_rng(9).integers(0, 256, 1 << 13, dtype=np.uint8)


def window_unpack_input():
    return np.random.default_rng(3).integers(0, 256, 512, dtype=np.uint8)


def fft_inputs(k):
    rng = np.random.default_rng(k)
    n = 1 << k
    x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
    xr = rng.uniform(-1, 1, 2 * n).astype(np.float32)
    return x, xr, (n // 2 if n > 1 else 1, 2 if n > 1 else 1)


def s1_input(nc):
    rng = np.random.default_rng(nc)
    x = ((rng.standard_normal(nc) + 1j * rng.standard_normal(nc)) * 100).astype(np.complex64)
    x[rng.integers(0, nc, 12)] *= 40
    return x


def dd_input(nc):
    rng = np.random.default_rng(nc)
    return (rng.standard_normal(nc) + 1j * rng.standard_normal(nc)).astype(np.complex64)


def dd_float32_params(nc, f_low, bw):
    f_min, f_c = np.float32(f_low), np.float32(np.float32(f_low) + np.float32(bw))
    df = np.float32(np.float32(bw) / np.float32(nc))
    return float(f_min), float(f_c), float(df)


def s2_input():
    rng = np.random.default_rng(21)
    C_, L = 48, 1024
    x = (rng.standard_normal((C_, L)) + 1j * rng.standard_normal((C_, L))).astype(np.complex64)
    x[5, :] = 3
    x[9, ::8] *= 9
    x[11, :] = 0
    return x


def detect_input(C_, L):
    rng = np.random.default_rng(C_ * L)
    x = (rng.standard_normal((C_, L)) + 1j * rng.standard_normal((C_, L))).astype(np.complex64)
    x[:, L // 8:L // 8 + 8] *= 10
    x[1, :] = 0
    return x


def chain_input(logn, C_, bits):
    n = 1 << logn
    rng = np.random.default_rng(logn * 7 + C_)
    if bits == -8:
        v = np.clip(np.round(rng.standard_normal(n) * 20), -127, 127)
        v[n // 2:n // 2 + 32] += np.round(rng.standard_normal(32) * 90)
        return np.clip(v, -127, 127).astype(np.int8).view(np.uint8)
    return rng.integers(0, 256, n * bits // 8, dtype=np.uint8)


def refft_layout_block(rng, nt, nf):
    """spectra [time][frequency]: noise, one steady tone (low kurtosis), one bursty channel (high kurtosis), one
    manually zapped channel, and a broadband burst over a few consecutive spectra"""
    x = (rng.standard_normal((nt, nf)) + 1j * rng.standard_normal((nt, nf))).astype(np.complex64)
    x[:, 5] = 3
    x[::8, 9] *= 9
    x[:, 11] = 0
    x[nt // 3:nt // 3 + 16, :] *= 1.6   # mild enough to stay inside the kurtosis thresholds of the detector tests
    return x


# --- the reference's outputs, rebuilt from the golden file
def ref_s1_pipe(x, nc):
    """kept bins are the input times the normalisation coefficient, the rest zero; the digest pins the result to the
    reference's output bit for bit"""
    g = golden()
    r = (x.view(np.float32) * g[f"s1_{nc}_coef"]).view(np.complex64)
    r[np.unpackbits(g[f"s1_{nc}_zero"], count=nc).astype(bool)] = 0
    assert digest(r) == g_str(f"s1_{nc}_digest")
    return r


def ref_zeroed(x, key, axis):
    """the SK stages zero whole channels and leave the others untouched; the stored mask is
    np.all(reference output == 0, axis=axis)"""
    r = x.copy()
    zero = golden()[f"{key}_zero"]
    if axis == 1:
        r[zero] = 0
    else:
        r[:, zero] = 0
    assert digest(r) == g_str(f"{key}_digest")
    return r


def ref_holders(key):
    g = golden()
    return [dict(boxcar=int(b), length=int(n), count=int(c), series=g.get(f"{key}_series_{b}"))
            for b, n, c in zip(g[f"{key}_boxcar"], g[f"{key}_length"], g[f"{key}_count"])]


@pytest.mark.parametrize("bits", UNPACK_BITS)
def test_unpack_bit_exact(oracle, bits):
    raw, n = unpack_input(bits)
    assert digest(oracle.unpack(raw, n, bits)) == g_str(f"unpack_{bits}")
    if bits in (1, 2, 4):     # generic == handwritten, as test-unpack.cpp:211-254 checks
        assert g_str(f"unpack_handwritten_{bits}") == g_str(f"unpack_{bits}")


def test_unpack_multistream_bit_exact(oracle):
    raw = multistream_input()
    for bits in (8, -8, 16, -16):
        n = raw.size * 8 // abs(bits) // 2
        for i, a in enumerate(oracle.unpack_interleaved_2(raw, n, bits)):
            assert digest(a) == g_str(f"il2_{bits}_{i}")
    n = raw.size // 2
    for i, a in enumerate(oracle.unpack_snap1(raw, n)):
        assert digest(a) == g_str(f"snap1_{i}")
    for streams in (2, 4):
        n = raw.size // streams
        for i, a in enumerate(oracle.unpack_gznupsr_a1(raw, n, streams)):
            assert digest(a) == g_str(f"gznu{streams}_{i}")


@pytest.mark.parametrize("window", WINDOWS)
def test_window_bit_exact(oracle, window):
    for n in (16, 1000):
        assert digest(np.array([oracle.window(window, i, n) for i in range(n)], np.float32)) == \
            g_str(f"window{window}_{n}")
    raw = window_unpack_input()
    assert digest(oracle.unpack(raw, 512, -8, window)) == g_str(f"window{window}_unpack")


@pytest.mark.parametrize("k", FFT_LOG2)
def test_naive_fft_bit_exact(oracle, k):
    x, xr, (length, batch) = fft_inputs(k)
    for d in (1, -1):
        assert digest(oracle.fft_c2c(x, d)) == g_str(f"fft{k}_c2c_{d}")
    assert digest(oracle.fft_r2c(xr)) == g_str(f"fft{k}_r2c")
    assert digest(oracle.watfft(x, length, batch)) == g_str(f"fft{k}_watfft")


@pytest.mark.parametrize("nc,C_", S1_CASES)
def test_rfi_s1_pipe(oracle, nc, C_):
    x = s1_input(nc)
    thr = S1_THRESHOLD
    r = ref_s1_pipe(x, nc)
    o, mean, mask = oracle.rfi_s1_average(x, thr, C_)
    o = oracle.rfi_manual(o, 1000.0, 500.0, oracle.eval_rfi_ranges(S1_FREQ_LIST))
    p = np.abs(x.astype(np.complex128)) ** 2
    border = np.abs(p / (thr * p.mean()) - 1) < 1e-4       # the mean's summation order is the runtime's
    assert np.array_equal((r == 0)[~border], (o == 0)[~border])
    keep = (r != 0) & (o != 0)
    assert np.array_equal(r[keep], o[keep])                 # normalised values are bit-identical
    assert ((o == 0) & (x != 0)).sum() >= 10


def test_rfi_ranges_and_manual_zap(oracle):
    g = golden()
    for i, s in enumerate(RANGE_STRINGS):
        assert oracle.eval_rfi_ranges(s) == [(float(a), float(b)) for a, b in g[f"ranges_{i}"]], s
    x = np.ones(1500, np.complex64)
    rr = [(float(a), float(b)) for a, b in g["ranges_0"]]
    assert digest(oracle.rfi_manual(x, 0.0, 1499.0, rr)) == g_str("manual_1500")
    x = np.ones(1 << 12, np.complex64)
    for i, (pairs, fl, bw) in enumerate(MANUAL_CASES):
        assert digest(oracle.rfi_manual(x, fl, bw, pairs)) == g_str(f"manual_{i}")


@pytest.mark.parametrize("nc,f_low,bw,dm", DD_CASES)
def test_dedisperse_pipe_bit_exact(oracle, nc, f_low, bw, dm):
    x = dd_input(nc)
    o = oracle.dedisperse(x, *dd_float32_params(nc, f_low, bw), dm)
    assert digest(o) == g_str(f"dd_{nc}_pipe")
    assert g_str(f"dd_{nc}_direct") == g_str(f"dd_{nc}_pipe")


def test_nsamps_reserved(oracle):
    for args, expected in zip(NSAMPS_CASES, golden()["nsamps_reserved"]):
        assert oracle.nsamps_reserved(*args) == int(expected), args


def test_rfi_s2_pipe(oracle):
    x = s2_input()
    C_, L = x.shape
    thr = S2_THRESHOLD
    r = ref_zeroed(x, "s2", axis=1)
    o, sk, zap = oracle.rfi_s2(x.reshape(-1), L, C_, thr)
    o = o.reshape(C_, L)
    lo, hi = oracle.sk_thresholds(L, thr)
    fin = np.isfinite(sk)
    border = np.zeros(C_, bool)
    border[fin] = (np.abs(sk[fin] / hi - 1) < 1e-4) | (np.abs(sk[fin] / lo - 1) < 1e-4)
    rz = np.all(r == 0, axis=1)
    oz = np.all(o == 0, axis=1)
    assert np.array_equal(rz[~border], oz[~border])
    assert rz[5] and rz[9] and rz[11] and zap[11] == 0     # q5: the all-zero row was left alone, not "zapped"
    same = rz == oz
    assert np.array_equal(r[same], o[same])


@pytest.mark.parametrize("C_,L,maxbox,reserve", DETECT_CASES)
def test_signal_detect_pipe(oracle, C_, L, maxbox, reserve):
    x = detect_input(C_, L)
    n_input = 2 * C_ * L
    p = DETECT_PARAMS
    snr, chan_thr = p["snr"], p["chan_thr"]
    key = f"det_{C_}_{L}"
    holders = ref_holders(key)
    reserved = oracle.nsamps_reserved(n_input, C_, p["f_low"], p["bw"], p["fs"], p["dm"], reserve) // C_
    if reserve:
        assert reserved > 0
    res, series = oracle.signal_detect(x.reshape(-1), L, C_, reserved, snr, chan_thr, maxbox)
    assert res.detect_enabled == 1
    got = {h["boxcar"]: h for h in holders}
    exp = {int(res.boxcar_length[b]): b for b in range(res.n_boxcars) if res.signal_count[b] > 0}
    # every series the reference emits exists in the oracle with (near-)identical values and counts
    for bc, h in got.items():
        b = [i for i in range(res.n_boxcars) if res.boxcar_length[i] == bc][0]
        assert h["length"] == res.series_length[b]
        scale = np.sqrt(np.mean(h["series"].astype(np.float64) ** 2))
        assert np.abs(h["series"] - series[b, :h["length"]]).max() < 1e-4 * scale * np.sqrt(bc)
        assert abs(h["count"] - int(res.signal_count[b])) <= 1
    assert set(exp) - set(got) <= {bc for bc, b in exp.items() if res.signal_count[b] <= 1}
    assert len(got) > 0
    # the reference's count_signal over the oracle's boxcar-1 series
    assert int(golden()[f"{key}_count_signal"]) == res.signal_count[0]


@pytest.mark.parametrize("logn,C_,dm,bits", CHAIN_CASES)
def test_whole_chain_composition(oracle, logn, C_, dm, bits):
    """The reference's pipes composed as main.cpp:170-204 wires them (unpack -> R2C -> drop Nyquist -> s1 pipe ->
    dedisperse pipe -> waterfall FFT -> s2 pipe -> signal_detect_pipe_2), each stage being the reference's OWN code
    through the shim, against the oracle's one-call chain: pins sizes, the Nyquist drop, the [C][L] row layout, the
    normalisation coefficient and the detector's view of the spectrum — not only the stages in isolation."""
    import ctypes as CT

    import oracle_lib
    n = 1 << logn
    L = n // 2 // C_
    raw = chain_input(logn, C_, bits)
    p = CHAIN_PARAMS
    key = f"chain_{logn}_{C_}_{bits}"
    g = golden()
    rz = g[f"{key}_zero_rows"]
    holders = ref_holders(key)
    cfg = oracle_lib.ChainConfig()
    cfg.baseband_input_count, cfg.baseband_input_bits, cfg.window = n, bits, 0
    cfg.baseband_freq_low, cfg.baseband_bandwidth, cfg.baseband_sample_rate, cfg.dm = p["f_low"], p["bw"], p["fs"], dm
    cfg.baseband_reserve_sample = 0
    cfg.rfi_average_threshold, cfg.rfi_sk_threshold = p["avg_thr"], p["sk_thr"]
    cfg.spectrum_channel_count = C_
    cfg.snr_threshold, cfg.channel_threshold, cfg.max_boxcar_length = p["snr"], p["chan_thr"], p["maxbox"]
    arr = (CT.c_float * 2)(1200.0, 1201.0)
    cfg.rfi_pairs, cfg.n_rfi_pairs = CT.cast(arr, CT.POINTER(CT.c_float)), 1
    work, res, series, _ = oracle.chain(raw, cfg)
    ospec = work[:n].view(np.complex64).reshape(C_, L)
    oz = np.all(ospec == 0, axis=1)
    assert (rz != oz).sum() <= 1                                  # SK border only
    idx = np.arange(0, C_ * L, CHAIN_STRIDE)
    same = (rz == oz)[idx // L]
    spec = g[f"{key}_spectrum"]
    assert rel(ospec.reshape(-1)[idx][same], spec[same]) < 2e-7   # same arithmetic; reduction order is the runtime's
    if np.array_equal(rz, oz):
        assert res.zero_count == int(g[f"{key}_zero_count"])
        got = {h["boxcar"]: h for h in holders}
        for b in range(res.n_boxcars):
            bc = int(res.boxcar_length[b])
            if res.signal_count[b] > 1:
                assert bc in got and abs(got[bc]["count"] - int(res.signal_count[b])) <= 1
        for bc, h in got.items():
            b = [i for i in range(res.n_boxcars) if res.boxcar_length[i] == bc][0]
            assert h["length"] == res.series_length[b]


@pytest.mark.parametrize("nt,nf", SK_CASES)
def test_sk_v1(oracle, nt, nf):
    """alternate f-4: mitigate_rfi_spectral_kurtosis_method (v1) on the [time][frequency] layout of the refft path"""
    x = refft_layout_block(np.random.default_rng(nt + nf), nt, nf)
    thr = SK_THRESHOLD
    r = ref_zeroed(x, f"sk_{nt}_{nf}", axis=0)
    o, sk, zap = oracle.sk_v1(x.reshape(-1), nf, nt, thr)
    o = o.reshape(nt, nf)
    lo, hi = oracle.sk_thresholds(nt, thr)
    fin = np.isfinite(sk)
    border = np.zeros(nf, bool)
    border[fin] = (np.abs(sk[fin] / hi - 1) < 1e-4) | (np.abs(sk[fin] / lo - 1) < 1e-4)
    rz, oz = np.all(r == 0, axis=0), np.all(o == 0, axis=0)
    assert np.array_equal(rz[~border], oz[~border])
    assert rz[5] and rz[9] and rz[11] and zap[11] == 0      # the all-zero channel is NaN -> left alone
    same = rz == oz
    assert np.array_equal(r[:, same], o[:, same])            # same serial fp32 sums: identical where decisions agree


@pytest.mark.parametrize("nt,nf,maxbox", DETECT_V1_CASES)
def test_signal_detect_pipe_v1(oracle, nt, nf, maxbox):
    """alternate f-4: the reference's signal_detect_pipe (v1: SK v1 + per-spectrum sums + boxcars) against the oracle.
    The spectrum length is a multiple of the device's work-group size here: multi_mapreduce cuts the flat array into
    pieces of ceil(size / (items * groups)) * items elements (algorithm/multi_reduce.hpp:93-101), which are the rows
    only then; the oracle restates the intended per-spectrum sum."""
    x = refft_layout_block(np.random.default_rng(7 * nt + nf), nt, nf)
    p = DETECT_V1_PARAMS
    key = f"det_v1_{nt}_{nf}"
    holders = ref_holders(key)
    ospec, res, series = oracle.signal_detect_v1(x.reshape(-1), nf, nt, p["sk_thr"], p["snr"], p["chan_thr"], maxbox)
    assert digest(ospec.reshape(nt, nf)) == g_str(f"{key}_spectrum")
    assert res.detect_enabled == 1 and res.zero_count == int(np.sum(np.abs(ospec.reshape(nt, nf)[0]) == 0))
    got = {h["boxcar"]: h for h in holders}
    exp = {int(res.boxcar_length[b]): b for b in range(res.n_boxcars) if res.signal_count[b] > 0}
    assert len(got) > 0
    for bc, h in got.items():
        b = [i for i in range(res.n_boxcars) if res.boxcar_length[i] == bc][0]
        assert h["length"] == res.series_length[b]
        if bc == 1:   # (the reference re-uses one device buffer for every boxcar > 1 and copies it asynchronously: SURVEY q3)
            scale = np.sqrt(np.mean(h["series"].astype(np.float64) ** 2))
            assert np.abs(h["series"] - series[b, :h["length"]]).max() < 1e-4 * scale
            assert abs(h["count"] - int(res.signal_count[b])) <= 1
    assert set(exp) - set(got) <= {bc for bc, b in exp.items() if res.signal_count[b] <= 1}
