#!/usr/bin/env python
"""Generates tests/golden/srtb_golden.npz, srtb_chain_golden.npz and srtb_oracle_vs_ref.npz from the REFERENCE'S OWN
code (oracle/_ref/libsrtb_ref.so, the reference headers compiled through oracle/ref_shim). Needs a checkout of the
reference project:   make -C oracle ref REF=<reference>/userspace && python tests/golden/make_golden.py
The tests read only the committed .npz files."""
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
import ref_lib  # noqa: E402
import test_oracle_vs_ref as t  # noqa: E402  (the seeded inputs and the digest of that test)


def main():
    ref = ref_lib.load()
    assert ref is not None, "build oracle/_ref first: make -C oracle ref"
    rng = np.random.default_rng(20260921)
    g = {}
    raw = rng.integers(0, 256, 512, dtype=np.uint8)
    g["unpack_raw"] = raw
    for bits in (1, 2, 4, 8, -8, 16, -16):
        g[f"unpack_b{bits}"] = ref.unpack(raw, raw.size * 8 // abs(bits), bits)
    g["unpack_b-8_hamming"] = ref.unpack(raw, raw.size, -8, 2)
    g["unpack_b2_hann"] = ref.unpack(raw, raw.size * 4, 2, 1)
    a, b = ref.unpack_interleaved_2(raw, raw.size // 2, -8)
    g["il2_a"], g["il2_b"] = a, b
    a, b = ref.unpack_snap1(raw, raw.size // 2)
    g["snap1_a"], g["snap1_b"] = a, b
    for s in (2, 4):
        for i, o in enumerate(ref.unpack_gznupsr_a1(raw, raw.size // s, s)):
            g[f"gznu{s}_{i}"] = o
    for w in (1, 2):
        g[f"window{w}_16"] = np.array([ref.window(w, i, 16) for i in range(16)], np.float32)
    x = (rng.uniform(-1, 1, 256) + 1j * rng.uniform(-1, 1, 256)).astype(np.complex64)
    g["fft_x"] = x
    g["fft_fwd"] = ref.fft_c2c(x, 1)
    g["fft_bwd"] = ref.fft_c2c(x, -1)
    xr = rng.integers(-128, 128, 512).astype(np.float32)
    g["r2c_x"] = xr
    g["r2c_X"] = ref.fft_r2c(xr)
    g["watfft_8x32"] = ref.watfft(x, 32, 8)
    spec = ((rng.standard_normal(2048) + 1j * rng.standard_normal(2048)) * 100).astype(np.complex64)
    spec[rng.integers(0, 2048, 8)] *= 40
    g["s1_x"] = spec
    g["s1_y"] = ref.rfi_s1_pipe(spec, 1.5, 16, 1000.0, 500.0, "1100-1110, 1300.5-1302")
    y = (rng.standard_normal(2048) + 1j * rng.standard_normal(2048)).astype(np.complex64)
    g["dd_x"] = y
    for tag, (fl, bw, dm) in {"a": (1000.0, 500.0, 56.778), "b": (1000.0, 400.0, 562.05), "c": (1437.0, -64.0, -478.80)}.items():
        g[f"dd_{tag}"] = ref.dedisperse_pipe(y, fl, bw, dm)
        g[f"dd_{tag}_params"] = np.array([fl, bw, dm], np.float64)
    C_, L = 16, 256
    d = (rng.standard_normal((C_, L)) + 1j * rng.standard_normal((C_, L))).astype(np.complex64)
    d[2, :] = 3
    d[5, ::8] *= 9
    d[7, :] = 0
    g["s2_x"] = d.reshape(-1)
    g["s2_y"] = ref.rfi_s2_pipe(d.reshape(-1), L, C_, 1.2)
    e = (rng.standard_normal((C_, L)) + 1j * rng.standard_normal((C_, L))).astype(np.complex64)
    e[:, 40:48] *= 10
    e[3, :] = 0
    g["det_x"] = e.reshape(-1)
    hs = ref.signal_detect_pipe(e.reshape(-1), L, C_, 2 * C_ * L, False, 1000.0, 500.0, 1e9, 0.0, 6.0, 0.9, 32)
    g["det_boxcar"] = np.array([h["boxcar"] for h in hs], np.int64)
    g["det_count"] = np.array([h["count"] for h in hs], np.int64)
    g["det_length"] = np.array([h["length"] for h in hs], np.int64)
    for h in hs:
        g[f"det_series_{h['boxcar']}"] = h["series"]
    np.savez_compressed(HERE / "srtb_golden.npz", **g)
    print("wrote", HERE / "srtb_golden.npz", sum(v.nbytes for v in g.values()), "bytes in", len(g), "arrays")
    chain_golden(ref)


def chain_golden(ref):
    """One block through the reference's pipes composed as main.cpp:170-204 wires them (every stage = the reference's
    own code through the shim): the fixture the GPU box checks srtb_b200_process_block against."""
    rng = np.random.default_rng(20260922)
    n, C_, dm = 1 << 15, 16, 0.0
    nc, L = n // 2, n // 2 // C_
    v = np.clip(np.round(rng.standard_normal(n) * 20), -127, 127)
    v[n // 2:n // 2 + 48] += np.round(rng.standard_normal(48) * 90)
    raw = np.clip(v, -127, 127).astype(np.int8).view(np.uint8)
    f_low, bw, fs, avg_thr, sk_thr, snr, chan_thr, maxbox = 1000.0, 500.0, 1e9, 5.0, 1.3, 6.0, 0.9, 64
    spec = ref.fft_r2c(ref.unpack(raw, n, -8))[:nc]
    spec = ref.rfi_s1_pipe(spec, avg_thr, C_, f_low, bw, "1200-1201")
    spec = ref.dedisperse_pipe(spec, f_low, bw, dm)
    spec = ref.watfft(spec, L, C_)
    spec = ref.rfi_s2_pipe(spec, L, C_, sk_thr)
    hs = ref.signal_detect_pipe(spec, L, C_, n, False, f_low, bw, fs, dm, snr, chan_thr, maxbox)
    g = {"raw": raw, "params": np.array([n, C_, dm, f_low, bw, fs, avg_thr, sk_thr, snr, chan_thr, maxbox], np.float64),
         "freq_pairs": np.array([1200.0, 1201.0], np.float32), "spectrum": spec.reshape(C_, L),
         "zero_count": np.array([int(np.sum(np.abs(spec.reshape(C_, L)[:, 0]) ** 2 == 0))], np.int64),
         "det_boxcar": np.array([h["boxcar"] for h in hs], np.int64),
         "det_count": np.array([h["count"] for h in hs], np.int64),
         "det_length": np.array([h["length"] for h in hs], np.int64)}
    np.savez_compressed(HERE / "srtb_chain_golden.npz", **g)
    print("wrote", HERE / "srtb_chain_golden.npz", sum(v_.nbytes for v_ in g.values()), "bytes;",
          "candidates at boxcars", g["det_boxcar"].tolist(), "counts", g["det_count"].tolist())
    oracle_vs_ref_golden(ref)


def _holders(g, key, hs, series_boxcars=None):
    g[f"{key}_boxcar"] = np.array([h["boxcar"] for h in hs], np.int64)
    g[f"{key}_length"] = np.array([h["length"] for h in hs], np.int64)
    g[f"{key}_count"] = np.array([h["count"] for h in hs], np.int64)
    for h in hs:
        if series_boxcars is None or h["boxcar"] in series_boxcars:
            g[f"{key}_series_{h['boxcar']}"] = h["series"]


def _zero_mask(g, key, x, r, axis):
    """the SK stages zero whole channels: store which, and the digest of the output they rebuild"""
    zero = np.all(r == 0, axis=axis)
    rebuilt = x.copy()
    if axis == 1:
        rebuilt[zero] = 0
    else:
        rebuilt[:, zero] = 0
    assert np.array_equal(rebuilt.view(np.uint32), r.view(np.uint32)), key
    g[f"{key}_zero"] = zero
    g[f"{key}_digest"] = np.array(t.digest(r))


def oracle_vs_ref_golden(ref):
    """What the reference computes for the seeded inputs of tests/test_oracle_vs_ref.py (see its docstring for the
    stored forms)."""
    import oracle_lib
    oracle = oracle_lib.load()
    g = {}
    d = t.digest
    for bits in t.UNPACK_BITS:
        raw, n = t.unpack_input(bits)
        g[f"unpack_{bits}"] = np.array(d(ref.unpack(raw, n, bits)))
        if bits in (1, 2, 4):
            g[f"unpack_handwritten_{bits}"] = np.array(d(ref.unpack_handwritten(raw, n, bits)))
    raw = t.multistream_input()
    for bits in (8, -8, 16, -16):
        for i, a in enumerate(ref.unpack_interleaved_2(raw, raw.size * 8 // abs(bits) // 2, bits)):
            g[f"il2_{bits}_{i}"] = np.array(d(a))
    for i, a in enumerate(ref.unpack_snap1(raw, raw.size // 2)):
        g[f"snap1_{i}"] = np.array(d(a))
    for streams in (2, 4):
        for i, a in enumerate(ref.unpack_gznupsr_a1(raw, raw.size // streams, streams)):
            g[f"gznu{streams}_{i}"] = np.array(d(a))
    for w in t.WINDOWS:
        for n in (16, 1000):
            g[f"window{w}_{n}"] = np.array(d(np.array([ref.window(w, i, n) for i in range(n)], np.float32)))
        g[f"window{w}_unpack"] = np.array(d(ref.unpack(t.window_unpack_input(), 512, -8, w)))
    for k in t.FFT_LOG2:
        x, xr, (length, batch) = t.fft_inputs(k)
        for direction in (1, -1):
            g[f"fft{k}_c2c_{direction}"] = np.array(d(ref.fft_c2c(x, direction)))
        g[f"fft{k}_r2c"] = np.array(d(ref.fft_r2c(xr)))
        g[f"fft{k}_watfft"] = np.array(d(ref.watfft(x, length, batch)))
    for nc, C_ in t.S1_CASES:
        x = t.s1_input(nc)
        r = ref.rfi_s1_pipe(x, t.S1_THRESHOLD, C_, 1000.0, 500.0, t.S1_FREQ_LIST)
        zero = r == 0
        coef = np.float32(float(np.float32(nc) * np.float32(nc) / np.float32(C_)) ** -0.5)
        rebuilt = (x.view(np.float32) * coef).view(np.complex64)
        rebuilt[zero] = 0
        assert np.array_equal(rebuilt.view(np.uint32), r.view(np.uint32)), nc
        g[f"s1_{nc}_zero"] = np.packbits(zero)
        g[f"s1_{nc}_coef"] = coef
        g[f"s1_{nc}_digest"] = np.array(d(r))
    for i, s in enumerate(t.RANGE_STRINGS):
        g[f"ranges_{i}"] = np.array(ref.eval_rfi_ranges(s), np.float32).reshape(-1, 2)
    rr = ref.eval_rfi_ranges(t.RANGE_STRINGS[0])
    g["manual_1500"] = np.array(d(ref.rfi_manual(np.ones(1500, np.complex64), 0.0, 1499.0, rr)))
    for i, (pairs, fl, bw) in enumerate(t.MANUAL_CASES):
        g[f"manual_{i}"] = np.array(d(ref.rfi_manual(np.ones(1 << 12, np.complex64), fl, bw, pairs)))
    for nc, f_low, bw, dm in t.DD_CASES:
        x = t.dd_input(nc)
        g[f"dd_{nc}_pipe"] = np.array(d(ref.dedisperse_pipe(x, f_low, bw, dm)))
        g[f"dd_{nc}_direct"] = np.array(d(ref.dedisperse(x, *t.dd_float32_params(nc, f_low, bw), dm)))
    g["nsamps_reserved"] = np.array([ref.nsamps_reserved(*a) for a in t.NSAMPS_CASES], np.int64)
    x = t.s2_input()
    C_, L = x.shape
    _zero_mask(g, "s2", x, ref.rfi_s2_pipe(x.reshape(-1), L, C_, t.S2_THRESHOLD).reshape(C_, L), axis=1)
    p = t.DETECT_PARAMS
    for C_, L, maxbox, reserve in t.DETECT_CASES:
        x = t.detect_input(C_, L).reshape(-1)
        key = f"det_{C_}_{L}"
        _holders(g, key, ref.signal_detect_pipe(x, L, C_, 2 * C_ * L, reserve, p["f_low"], p["bw"], p["fs"], p["dm"],
                                                p["snr"], p["chan_thr"], maxbox))
        reserved = oracle.nsamps_reserved(2 * C_ * L, C_, p["f_low"], p["bw"], p["fs"], p["dm"], reserve) // C_
        res, series = oracle.signal_detect(x, L, C_, reserved, p["snr"], p["chan_thr"], maxbox)
        g[f"{key}_count_signal"] = np.array(ref.count_signal(series[0, :int(res.series_length[0])], p["snr"]), np.int64)
    p = t.CHAIN_PARAMS
    for logn, C_, dm, bits in t.CHAIN_CASES:
        n = 1 << logn
        nc, L = n // 2, n // 2 // C_
        key = f"chain_{logn}_{C_}_{bits}"
        spec = ref.fft_r2c(ref.unpack(t.chain_input(logn, C_, bits), n, bits))[:nc]   # fft_pipe.hpp:75-77: count = N/2
        spec = ref.rfi_s1_pipe(spec, p["avg_thr"], C_, p["f_low"], p["bw"], p["freq_list"])
        spec = ref.dedisperse_pipe(spec, p["f_low"], p["bw"], dm)
        spec = ref.watfft(spec, L, C_)
        spec = ref.rfi_s2_pipe(spec, L, C_, p["sk_thr"])
        _holders(g, key, ref.signal_detect_pipe(spec, L, C_, n, False, p["f_low"], p["bw"], p["fs"], dm, p["snr"],
                                                p["chan_thr"], p["maxbox"]), series_boxcars=())
        spec = spec.reshape(C_, L)
        g[f"{key}_zero_rows"] = np.all(spec == 0, axis=1)
        g[f"{key}_zero_count"] = np.array(int(np.sum(np.abs(spec[:, 0]) ** 2 == 0)), np.int64)
        g[f"{key}_spectrum"] = spec.reshape(-1)[::t.CHAIN_STRIDE].copy()
    for nt, nf in t.SK_CASES:
        x = t.refft_layout_block(np.random.default_rng(nt + nf), nt, nf)
        _zero_mask(g, f"sk_{nt}_{nf}", x, ref.sk_v1(x.reshape(-1), nf, nt, t.SK_THRESHOLD).reshape(nt, nf), axis=0)
    p = t.DETECT_V1_PARAMS
    for nt, nf, maxbox in t.DETECT_V1_CASES:
        x = t.refft_layout_block(np.random.default_rng(7 * nt + nf), nt, nf)
        key = f"det_v1_{nt}_{nf}"
        rspec, hs = ref.signal_detect_pipe_v1(x.reshape(-1), nf, nt, p["sk_thr"], p["snr"], p["chan_thr"], maxbox)
        g[f"{key}_spectrum"] = np.array(d(rspec.reshape(nt, nf)))
        _holders(g, key, hs, series_boxcars=(1,))   # only boxcar 1's series is compared (see the test)
    np.savez_compressed(t.GOLDEN, **g)
    print("wrote", t.GOLDEN, t.GOLDEN.stat().st_size, "bytes in", len(g), "arrays")


if __name__ == "__main__":
    main()
