"""Every route by which the block path evaluates the coherent-dedispersion chirp, against float64 truth.

The host picks the route from the row length L = N / 2 / C, the band and the DM:

  L = 2^13, 2^14     whole-row kernel (fft_bigrow.cuh): tabulated phase (CHIRP = 5, process_block by default) or
                     on the fly with 1/f from Newton steps, variants 1 / 3 / 4, or the exact reciprocal, 2
                     (process_block_dm_sweep, and process_block under SRTB_B200_CHIRP_TABLE=0)
  L = 2^10 .. 2^12   sixteen-point row kernel (fft_engine.cuh): tabulated phase or chirp_factor on the fly
  L = 2^15 .. 2^18   long-row column sweep, Newton steps cp.newton = 0 (exact) / 1 / 2
  otherwise          the separate s1 + dedisperse kernel (in place; out of place in the DM sweep)

Each case runs one 8-bit noise block with s1 zapping off and a wide SK window, so that no threshold decision enters the
comparison, and bounds every row of the dynamic spectrum (rel-L2 <= 1e-5) and its largest element (<= 1e-4 RMS)
against a float64 evaluation of the same chain. The on-the-fly variants of the whole-row and row kernels are reachable
from process_block only with SRTB_B200_CHIRP_TABLE=0, which is read once per process: those cases run in one child
process (this file run as a script with --child OUTDIR). The DM sweep must return, trial by trial, exactly the result
header process_block returns at that DM through the same route.
"""
import json
import math
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")

if __name__ == "__main__":   # child process: the same imports as under pytest (tests/conftest.py)
    _ROOT = Path(__file__).resolve().parent.parent
    sys.path[:0] = [str(_ROOT), str(_ROOT / "tests"), str(_ROOT / "simple-radio-telescope-backend_b200")]

import srtb_b200  # noqa: E402
from test_gpu_parity import (_from_device_ptr, _row_rel_l2, chain_truth_float64, make_block_config,  # noqa: E402
                             oracle_chain_config, synth_baseband)

ROW_REL_L2 = 1e-5
MAX_ABS_RMS = 1e-4
D = 4.148808e3                      # coherent_dedispersion.hpp:67


# ----------------------------------------------------------------------------- host route selection, restated
def block_scalars(logn, C_, f_low, bw, dm):
    """(L, f_min, f_c, df, ddm) as block_enqueue hands them to the kernels: float32 band scalars (dedisperse_pipe.hpp:34)"""
    nc = 1 << (logn - 1)
    f_min = np.float32(f_low)
    f_c = np.float32(f_min + np.float32(bw))
    df = np.float32(np.float32(bw) / np.float32(nc))
    return nc // C_, float(f_min), float(f_c), float(df), (D * 1e6) * float(np.float32(dm))


def _newton_steps(delta, kmax):
    # one step when the squared spacing is within an ulp of fp64, two when its fourth power keeps |k| * error below
    # 1e-9 cycles, else 0 (the exact reciprocal): srtb_b200.cu:1723-1724 and 1786
    d2 = delta * delta
    return 1 if d2 <= 2.0 ** -52 else (2 if d2 * d2 * kmax < 1e-9 else 0)


def chirp_route(logn, C_, f_low, bw, dm, table=True):
    """the chirp route process_block takes for an 8-bit single-stream block: (kind, variant)"""
    L, f_min, f_c, df, ddm = block_scalars(logn, C_, f_low, bw, dm)
    fa = min(abs(f_min), abs(f_c))
    q = (f_c - f_min) * (1.0 / f_c)
    kmax = max(1.0, abs(ddm) / fa * q * q)
    if L in (8192, 16384):                                   # chirp_fusable: whole-row kernel (srtb_b200.cu:1638)
        if table:
            return ("whole-row", 5)                          # srtb_b200.cu:1728
        # srtb_b200.cu:1716-1727: far = B1 = L/16 bins along a butterfly's inputs, near = the pair's second bin
        far = _newton_steps((L // 16) * abs(df) / fa, kmax)
        near = _newton_steps(abs(df) / fa, kmax)
        return ("whole-row", 2 if far == 0 or near == 0 else (1 if far == 1 else (3 if near == 1 else 4)))
    if L in (1024, 2048, 4096):                              # chirp_fusable: row16 kernel (srtb_b200.cu:1639)
        return ("row16", "table" if table else "otf")
    if 2 ** 15 <= L <= 2 ** 18:                              # long_fusable (srtb_b200.cu:1760)
        # srtb_b200.cu:1768-1769, 1782-1786: consecutive points of a thread are (L1 / 16) * L2 bins apart
        lq = int(math.log2(L))
        l1 = (lq + 1) // 2
        l2 = lq - l1
        return ("long", _newton_steps(((1 << l1) // 16) * (1 << l2) * abs(df) / fa, kmax))
    return ("separate", None)                                # rfi_s1_dedisperse_fused (srtb_b200.cu:2221)


# (id, (log2 N, C, f_low, bw, DM), route with the phase table, route without it)
WHOLE_ROW = [
    ("wr14-exact-a", (22, 128, 1000.0, 400.0, 562.05), ("whole-row", 5), ("whole-row", 2)),
    ("wr14-exact-b", (24, 512, 1000.0, 400.0, 562.05), ("whole-row", 5), ("whole-row", 2)),
    ("wr13-exact", (23, 512, 1000.0, 400.0, 562.05), ("whole-row", 5), ("whole-row", 2)),
    ("wr14-n3-j1644", (24, 512, 1437.0, -64.0, -478.80), ("whole-row", 5), ("whole-row", 3)),
    ("wr13-n3", (26, 4096, 1000.0, 500.0, 56.78), ("whole-row", 5), ("whole-row", 3)),
    ("wr14-n4", (24, 512, 1000.0, 500.0, 56.78), ("whole-row", 5), ("whole-row", 4)),
    ("wr13-n4", (24, 1024, 1000.0, 500.0, 56.78), ("whole-row", 5), ("whole-row", 4)),
    ("wr13-n1-narrow", (27, 8192, 1000.0, 1.0, 1000.0), ("whole-row", 5), ("whole-row", 1)),
]
ROW16 = [
    ("row16-L10", (22, 2048, 1000.0, 400.0, 562.05), ("row16", "table"), ("row16", "otf")),
    ("row16-L11", (22, 1024, 1000.0, 400.0, 562.05), ("row16", "table"), ("row16", "otf")),
    ("row16-L12-j1644", (22, 512, 1437.0, -64.0, -478.80), ("row16", "table"), ("row16", "otf")),
]
OTHER = [
    ("long15-exact", (22, 64, 1000.0, 500.0, 562.05), ("long", 0), ("long", 0)),
    ("long15-n1-narrow", (25, 512, 1000.0, 0.1, 10000.0), ("long", 1), ("long", 1)),
    ("long17-n1-narrow", (26, 256, 1000.0, 0.01, 1.0e6), ("long", 1), ("long", 1)),
    ("long15-n2", (25, 512, 1000.0, 500.0, 56.78), ("long", 2), ("long", 2)),
    ("long16-n2-j1644", (24, 128, 1437.0, -64.0, -478.80), ("long", 2), ("long", 2)),
    ("sep-L9", (20, 1024, 1000.0, 400.0, 562.05), ("separate", None), ("separate", None)),
    ("sep-L19-j1644", (22, 4, 1437.0, -64.0, -478.80), ("separate", None), ("separate", None)),
]
TABLE_CASES = WHOLE_ROW + ROW16 + OTHER          # run in this process (phase table on)
CHILD_CASES = WHOLE_ROW + ROW16                  # run in the SRTB_B200_CHIRP_TABLE=0 child

# DM sweeps: (id, (log2 N, C, f_low, bw), format, trial DMs); one geometry per route
SNAP1 = srtb_b200.FORMAT_NAOCPSR_SNAP1
SIMPLE = srtb_b200.FORMAT_SIMPLE
PARENT_SWEEPS = [
    ("long15-config4", (25, 512, 1000.0, 500.0), SIMPLE, [0.0, 20.0, 56.78, -30.0]),
    ("long15-snap1", (22, 64, 1000.0, 400.0), SNAP1, [0.0, 3.0, 562.05, -100.0]),
    ("sep-L9", (20, 1024, 1000.0, 400.0), SIMPLE, [0.0, 10.0, 562.05, -478.8]),
]
CHILD_SWEEPS = [
    ("wr14", (24, 512, 1000.0, 500.0), SIMPLE, [0.0, 10.0, 56.78, 562.05]),
    ("wr13-j1644", (23, 512, 1437.0, -64.0), SIMPLE, [0.0, -30.0, -478.8, 100.0]),
    ("row16-L11", (22, 1024, 1000.0, 400.0), SIMPLE, [0.0, 10.0, 562.05, -200.0]),
]


def _case_params(cases):
    return [pytest.param(geom, table, id=cid) for cid, geom, table, _ in cases]


def test_route_selection_mirror():
    """every case lands on the route and Newton variant it exists to cover, so that a retuned constant in the host
    selection cannot silently move a case off its variant (the mirror restates srtb_b200.cu's rules)"""
    for cid, geom, table, otf in TABLE_CASES:
        assert chirp_route(*geom, table=True) == table, cid
        assert chirp_route(*geom, table=False) == otf, cid
        if table[0] == "whole-row":       # one CTA per row: the rows must outnumber the persistent grid
            assert geom[1] >= 512 or cid == "wr14-exact-a", cid
    covered = {r for _, _, t, o in TABLE_CASES for r in (t, o)}
    assert covered >= {("whole-row", v) for v in (1, 2, 3, 4, 5)} | {("long", v) for v in (0, 1, 2)}
    assert {("row16", "table"), ("row16", "otf"), ("separate", None)} <= covered
    kinds = {"long15": "long", "sep": "separate", "wr14": "whole-row", "wr13": "whole-row", "row16": "row16"}
    for sid, (logn, C_, f_low, bw), _, dms in PARENT_SWEEPS + CHILD_SWEEPS:
        for dm in dms:
            assert chirp_route(logn, C_, f_low, bw, dm)[0] == kinds[sid.split("-")[0]], (sid, dm)
    # the whole-row sweeps visit more than one Newton variant (the variant follows the DM)
    assert len({chirp_route(*g, dm, table=False) for _, g, _, dms in CHILD_SWEEPS[:1] for dm in dms}) >= 2


# ----------------------------------------------------------------------------- float64 truth
def chain_truth_torch(bb, cfg, device):
    """chain_truth_float64 in torch complex128 (on the device for blocks too large for a host FFT): the same
    parameter roundings, the same evaluation order of k"""
    n = cfg.baseband_input_count
    nc = n // 2
    C_ = min(cfg.spectrum_channel_count, nc)
    L = nc // C_
    X = torch.fft.rfft(torch.from_numpy(bb).to(device).to(torch.float64))[:nc]
    pw = X.real ** 2 + X.imag ** 2
    coef = float(srtb_b200.norm_coefficient(nc, cfg.spectrum_channel_count))
    limit = float(np.float32(cfg.mitigate_rfi_average_method_threshold)) * pw.mean()
    X = torch.where(pw > limit, torch.zeros_like(X), X * coef)
    del pw
    f_min = np.float32(cfg.baseband_freq_low)
    bw = np.float32(cfg.baseband_bandwidth)
    f_c = float(np.float32(f_min + bw))
    df = float(np.float32(bw / np.float32(nc)))
    f = float(f_min) + df * torch.arange(nc, dtype=torch.float64, device=device)
    k = (D * 1e6) * float(np.float32(cfg.dm)) / f * ((f - f_c) / f_c) ** 2
    del f
    X = X * torch.polar(torch.ones_like(k), -2 * math.pi * (k - torch.trunc(k)))
    del k
    return torch.fft.ifft(X.reshape(C_, L), dim=1) * L


def spectrum_errors(got, truth):
    """per-row rel-L2, whole-block rel-L2 and max |got - truth| / RMS(truth) of [C][L] complex arrays, in float64"""
    g = torch.as_tensor(got).to(truth.device, torch.complex128) if torch.is_tensor(truth) else None
    if g is None:
        rows = _row_rel_l2(got, truth)
        d = np.abs(got.astype(np.complex128) - truth)
        p = np.abs(truth) ** 2
        return rows, float(np.sqrt((d ** 2).sum() / p.sum())), float(d.max() / np.sqrt(p.mean()))
    d = (g - truth).abs()
    p = truth.abs() ** 2
    rows = (d ** 2).sum(1).sqrt() / p.sum(1).sqrt().clamp_min(1e-300)
    return rows.cpu().numpy(), float(((d ** 2).sum() / p.sum()).sqrt()), float(d.max() / p.mean().sqrt())


def _noise_block(logn, C_):
    return synth_baseband(1 << logn, seed=1000 * logn + C_, tone=False, pulse=False)


def run_route_case(ctx, geom):
    """process_block on one noise block at `geom`; returns (report, dynamic spectrum [C][L] complex64)"""
    logn, C_, f_low, bw, dm = geom
    n = 1 << logn
    L = n // 2 // C_
    bb = _noise_block(logn, C_)
    cfg = make_block_config(n, -8, SIMPLE, C_, dm, f_low=f_low, bw=bw, fs=2e6 * abs(bw), avg_thr=1e9, sk_thr=1.95,
                            snr=50.0)
    res = ctx.process_block(cfg, torch.from_numpy(bb.view(np.uint8)).pin_memory(), n, None)
    torch.cuda.synchronize()
    got = _from_device_ptr(ctx.block_spectrum_ptr(0), n // 2).reshape(C_, L)
    if logn >= 25:
        truth = chain_truth_torch(bb, cfg, "cuda")
    else:
        truth = chain_truth_float64(bb, cfg)
    rows, total, maxabs = spectrum_errors(got, truth)
    del truth
    worst = int(np.argmax(rows))
    rep = dict(zero_count=int(res[0].zero_count), rows=int(C_), L=int(L), row_rel_l2=float(rows[worst]), worst_row=worst,
               rel_l2=total, maxabs_rms=maxabs)
    return rep, got


def _check_route_report(cid, route, rep):
    print(f"{cid:18s} {str(route):22s} L=2^{int(math.log2(rep['L'])):<2d} rows={rep['rows']:5d}  rel-L2 {rep['rel_l2']:.2e}"
          f"  worst row {rep['row_rel_l2']:.2e} (row {rep['worst_row']})  max-abs/RMS {rep['maxabs_rms']:.2e}")
    assert rep["zero_count"] == 0, f"{cid}: a channel was zapped; the comparison needs none"
    assert rep["row_rel_l2"] <= ROW_REL_L2, f"{cid}: row {rep['worst_row']} has rel-L2 {rep['row_rel_l2']:.3e}"
    assert rep["maxabs_rms"] <= MAX_ABS_RMS, f"{cid}: max-abs {rep['maxabs_rms']:.3e} x RMS"


@pytest.mark.gpu
@pytest.mark.parametrize("cid,geom,route", [pytest.param(c, g, t, id=c) for c, g, t, _ in TABLE_CASES])
def test_chirp_route_vs_float64(ctx, cid, geom, route):
    """process_block with the phase table (the default): whole-row and row16 tabulated, long Newton 0/1/2, separate"""
    rep, _ = run_route_case(ctx, geom)
    _check_route_report(cid, route, rep)


# ----------------------------------------------------------------------------- the SRTB_B200_CHIRP_TABLE=0 child
def _header_bytes(res):
    return np.frombuffer(bytes(res), np.uint8).copy()


def _sweep_block(logn, fmt, seed):
    n = 1 << logn
    if fmt == SIMPLE:
        return synth_baseband(n, seed)
    a, b = synth_baseband(n, seed), synth_baseband(n, seed + 1, tone=False)
    raw = np.empty(2 * n, np.int8)               # naocpsr_snap1 "1 1 2 2"
    raw.reshape(-1, 4)[:, 0:2] = a.reshape(-1, 2)
    raw.reshape(-1, 4)[:, 2:4] = b.reshape(-1, 2)
    return raw


def run_sweep(ctx, geom, fmt, dms):
    """(sweep headers, process_block headers) as uint8 arrays [n_dm][streams][sizeof(DetectResult)]"""
    logn, C_, f_low, bw = geom
    n = 1 << logn
    raw = _sweep_block(logn, fmt, seed=logn * 10 + C_)
    cfg = make_block_config(n, -8, fmt, C_, 0.0, f_low=f_low, bw=bw, fs=2e6 * abs(bw), avg_thr=10.0, sk_thr=1.3,
                            snr=6.0, maxbox=64)
    pinned = torch.from_numpy(raw.view(np.uint8)).pin_memory()
    sweep = ctx.process_block_dm_sweep(cfg, pinned, raw.size, dms)
    got = np.array([[_header_bytes(r) for r in trial] for trial in sweep])
    single = []
    for dm in dms:
        cfg.dm = dm
        single.append([_header_bytes(r) for r in ctx.process_block(cfg, pinned, raw.size, None)])
    return got, np.array(single)


def _child(outdir):
    out = Path(outdir)
    torch.cuda.set_device(0)
    ctx = srtb_b200.Context(0, torch.cuda.current_stream().cuda_stream)
    report = {}
    for cid, geom, _, otf in CHILD_CASES:
        rep, got = run_route_case(ctx, geom)
        report[cid] = rep
        if otf == ("whole-row", 2):
            np.save(out / f"spectrum_{cid}.npy", got)
        del got
    for sid, geom, fmt, dms in CHILD_SWEEPS:
        got, single = run_sweep(ctx, geom, fmt, dms)
        np.save(out / f"sweep_{sid}.npy", got)
        np.save(out / f"single_{sid}.npy", single)
    (out / "report.json").write_text(json.dumps(report))
    ctx.close()


@pytest.fixture(scope="module")
def no_table_run(tmp_path_factory):
    """one child process with SRTB_B200_CHIRP_TABLE=0 (read once per process): the on-the-fly cases and sweeps"""
    out = tmp_path_factory.mktemp("chirp_on_the_fly")
    env = {**os.environ, "SRTB_B200_CHIRP_TABLE": "0", "PYTHONPATH": os.pathsep.join(sys.path)}
    p = subprocess.run([sys.executable, str(Path(__file__).resolve()), "--child", str(out)], capture_output=True,
                       text=True, timeout=1500, env=env)
    assert p.returncode == 0, p.stderr[-3000:]
    return out, json.loads((out / "report.json").read_text())


@pytest.mark.gpu
@pytest.mark.parametrize("cid,geom,route", [pytest.param(c, g, o, id=c) for c, g, _, o in CHILD_CASES])
def test_chirp_route_on_the_fly_vs_float64(no_table_run, cid, geom, route):
    """process_block without the phase table: whole-row Newton variants 1 / 3 / 4 and exact 2, row16 chirp_factor"""
    _, report = no_table_run
    _check_route_report(cid, route, report[cid])


def _explain_header_diff(a, b):
    ra = srtb_b200.DetectResult.from_buffer_copy(a.tobytes())
    rb = srtb_b200.DetectResult.from_buffer_copy(b.tobytes())
    diff = []
    for name, _ in srtb_b200.DetectResult._fields_:
        va, vb = getattr(ra, name), getattr(rb, name)
        if hasattr(va, "__len__"):
            va, vb = list(va), list(vb)
        if name in ("variance", "threshold"):
            va = np.asarray(va, np.float32).view(np.uint32).tolist()
            vb = np.asarray(vb, np.float32).view(np.uint32).tolist()
        if va != vb:
            diff.append((name, va, vb))
    return diff


def _check_sweep(sid, dms, got, single):
    assert got.shape == single.shape and got.shape[0] == len(dms)
    for j, dm in enumerate(dms):
        for s in range(got.shape[1]):
            assert np.array_equal(got[j, s], single[j, s]), \
                f"{sid}: DM {dm} stream {s}: the sweep differs from process_block in {_explain_header_diff(got[j, s], single[j, s])}"
    # not vacuous: the trials differ from one another, and the detector ran
    assert len({got[j, 0].tobytes() for j in range(len(dms))}) > 1, f"{sid}: every trial returned the same header"
    hdr = [srtb_b200.DetectResult.from_buffer_copy(got[j, 0].tobytes()) for j in range(len(dms))]
    assert all(h.detect_enabled == 1 and h.n_boxcars > 0 for h in hdr)
    print(f"sweep {sid}: {len(dms)} DMs x {got.shape[1]} stream(s) bit-identical to process_block; "
          f"signal counts {[sum(h.signal_count[:h.n_boxcars]) for h in hdr]}")


@pytest.mark.gpu
@pytest.mark.parametrize("sid,geom,fmt,dms", [pytest.param(*c, id=c[0]) for c in PARENT_SWEEPS])
def test_dm_sweep_bit_identical_per_trial(ctx, sid, geom, fmt, dms):
    """long and separate routes (and a dual-stream snap1 block): every trial's header equals process_block's at that DM"""
    got, single = run_sweep(ctx, geom, fmt, dms)
    _check_sweep(sid, dms, got, single)


@pytest.mark.gpu
@pytest.mark.parametrize("sid,dms", [pytest.param(c[0], c[3], id=c[0]) for c in CHILD_SWEEPS])
def test_dm_sweep_bit_identical_per_trial_on_the_fly(no_table_run, sid, dms):
    """whole-row and row16 routes, both evaluating the chirp on the fly (no phase table)"""
    out, _ = no_table_run
    _check_sweep(sid, dms, np.load(out / f"sweep_{sid}.npy"), np.load(out / f"single_{sid}.npy"))


# ----------------------------------------------------------------------------- table against exact on-the-fly, table cache
@pytest.mark.gpu
@pytest.mark.parametrize("cid,geom", [pytest.param(c, g, id=c) for c, g, _, o in WHOLE_ROW if o == ("whole-row", 2)])
def test_phase_table_equals_exact_on_the_fly(ctx, no_table_run, cid, geom):
    """at a whole-row geometry that selects the exact reciprocal (variant 2) the tabulated and on-the-fly routes
    evaluate the same k, round it to nearest the same way and hand the SFU the same fp32 angle: bit-identical spectra"""
    out, _ = no_table_run
    _, tab = run_route_case(ctx, geom)
    otf = np.load(out / f"spectrum_{cid}.npy")
    nd = int((tab != otf).sum())
    assert nd == 0, f"{cid}: {nd} of {tab.size} values differ, max |diff| {np.abs(tab - otf).max():.3e}"


def _spectra(c, cfg, bb, streams=1):
    n = cfg.baseband_input_count
    c.process_block(cfg, torch.from_numpy(bb.view(np.uint8)).pin_memory(), bb.size, None)
    torch.cuda.synchronize()
    return [_from_device_ptr(c.block_spectrum_ptr(s), n // 2) for s in range(streams)]


@pytest.mark.gpu
def test_phase_table_rebuilt_on_dm_band_and_size_change(ctx):
    """one context runs DM a, b, a, then DM a with another f_low, then the same DM and band with another N (L = 2^14
    throughout): every spectrum is bit-identical to a fresh context's, so the cached table follows all of them"""
    a, b = 562.05, 56.78
    seq = [(22, 128, 1000.0, a), (22, 128, 1000.0, b), (22, 128, 1000.0, a), (22, 128, 1100.0, a), (23, 256, 1100.0, a)]
    for logn, C_, f_low, dm in seq:
        n = 1 << logn
        assert chirp_route(logn, C_, f_low, 400.0, dm) == ("whole-row", 5)
        bb = _noise_block(logn, C_)
        cfg = make_block_config(n, -8, SIMPLE, C_, dm, f_low=f_low, bw=400.0, fs=8e8, avg_thr=1e9, sk_thr=1.95, snr=50.0)
        got = _spectra(ctx, cfg, bb)[0]
        fresh = srtb_b200.Context(0, torch.cuda.current_stream().cuda_stream)
        try:
            expect = _spectra(fresh, cfg, bb)[0]
        finally:
            fresh.close()
        nd = int((got != expect).sum())
        assert nd == 0, f"N=2^{logn} f_low={f_low} DM={dm}: {nd} values differ from a fresh context's"


@pytest.mark.gpu
def test_ring_dm_alternating_matches_process_block(ctx):
    """dual-polarisation snap1 blocks at L = 2^14 through the ring with the DM alternating per submission and up to
    three blocks in flight: both streams of every block are bit-identical to process_block at its DM (a table rebuilt
    under an in-flight block, or read by the second lane before it is built, would show here)"""
    logn, C_ = 22, 128
    n = 1 << logn
    slots = 3
    dms = [562.05, 56.78, -100.0, 562.05, 0.0, 56.78, 10.0]
    cfgs = [make_block_config(n, -8, SNAP1, C_, dm, f_low=1000.0, bw=400.0, fs=8e8, avg_thr=10.0, sk_thr=1.3, snr=6.0)
            for dm in dms]
    blocks = [torch.from_numpy(_sweep_block(logn, SNAP1, seed=500 + i).view(np.uint8)).pin_memory() for i in range(len(dms))]
    expect = [_spectra(ctx, cfg, blk.numpy(), streams=2) for cfg, blk in zip(cfgs, blocks)]
    got, tickets = [], []
    for cfg, blk in zip(cfgs, blocks):
        tickets.append(ctx.submit_block_ex(cfg, blk, blk.numel(), False))
        if len(tickets) == slots:
            _, _, ptrs = ctx.collect_block_ex(tickets.pop(0))
            got.append([_from_device_ptr(p, n // 2) for p in ptrs])
    while tickets:
        _, _, ptrs = ctx.collect_block_ex(tickets.pop(0))
        got.append([_from_device_ptr(p, n // 2) for p in ptrs])
    assert len(got) == len(expect)
    for i, (g, e) in enumerate(zip(got, expect)):
        for s in range(2):
            nd = int((g[s] != e[s]).sum())
            assert nd == 0, f"block {i} (DM {dms[i]}) stream {s}: {nd} values differ from process_block"


# ----------------------------------------------------------------------------- the truth function itself (CPU)
@pytest.mark.parametrize("f_low,bw,dm", [(1000.0, 400.0, 562.05), (1437.0, -64.0, -478.80)])
def test_truth_function_vs_oracle(oracle, f_low, bw, dm):
    """chain_truth_float64 (and its torch twin) against the CPU oracle's chain under the same settings, so that a
    wrong truth function cannot make the GPU comparisons above vacuous"""
    logn, C_ = 16, 8                        # L = 2^12
    n = 1 << logn
    bb = synth_baseband(n, seed=77, tone=False, pulse=False)
    cfg = make_block_config(n, -8, SIMPLE, C_, dm, f_low=f_low, bw=bw, fs=2e6 * abs(bw), avg_thr=1e9, sk_thr=1.95,
                            snr=50.0)
    work, _, _, _ = oracle.chain(bb.view(np.uint8), oracle_chain_config(cfg))
    espec = work[:n].view(np.complex64).reshape(C_, n // 2 // C_)
    truth = chain_truth_float64(bb, cfg)
    assert not np.all(espec == 0, axis=1).any()
    rows, total, _ = spectrum_errors(espec, truth)
    print(f"oracle vs float64 truth ({f_low}, {bw}, DM {dm}): rel-L2 {total:.2e}, worst row {rows.max():.2e}")
    assert rows.max() <= ROW_REL_L2
    # the chirp matters at this DM: truth without it is far from the oracle
    cfg0 = make_block_config(n, -8, SIMPLE, C_, 0.0, f_low=f_low, bw=bw, fs=2e6 * abs(bw), avg_thr=1e9, sk_thr=1.95)
    assert spectrum_errors(espec, chain_truth_float64(bb, cfg0))[1] > 0.5
    # the torch twin agrees to the fp64 rounding of k (|k| reaches 2e8 cycles here: a few roundings of 2e8 x 2^-53
    # cycles each, ~1e-7 rad of phase), 50 times below the tolerance of the GPU comparisons
    t = chain_truth_torch(bb, cfg, "cpu").numpy()
    assert spectrum_errors(t, truth)[1] < 2e-7


if __name__ == "__main__":
    assert sys.argv[1] == "--child", "usage: test_gpu_chirp_routes.py --child OUTDIR"
    _child(sys.argv[2])
