"""Pin the port (oracle/rx_oracle.c) against the UNMODIFIED reference.

The reference ships no tests or golden vectors (SURVEY.md §4), so what the reference code itself computed, executed
over these inputs, is the pin: tests/golden/make_ref_pin.py (and make_golden.py for the per-case rx_fm outputs and the
rx_sdr conversions) recorded it under tests/golden/, so the comparison runs anywhere."""
import dataclasses
import json
import os

import numpy as np
import pytest

import oracle
from cases import fm_cases, fm_optional_cases
from rx_tools_b200.synth import digest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PIN = json.load(open(os.path.join(G, "ref_pin.json")))
FM_GOLD = json.load(open(os.path.join(G, "fm_golden.json")))


def test_tables_match_reference(port):
    assert digest(port.atan_table()) == PIN["tables"]["atan_sha256"]
    for row in range(11):
        assert [int(v) for v in port.droop9(row)] == PIN["tables"]["cic9"][row]


def test_scale_integer_form(port):
    # SURVEY F5: (int16)(x/32767.0*128.0+0.4) == trunc((1280x+131068)/327670) for all x
    tab = port.scale_table()
    x = np.arange(-32768, 32768, dtype=np.int64)
    num = 1280 * x + 131068
    q = np.where(num >= 0, num // 327670, -((-num) // 327670))
    assert np.array_equal(q.astype(np.int16), tab)
    assert tab.min() == -127 and tab.max() == 128


@pytest.mark.parametrize("case", fm_cases() + fm_optional_cases(), ids=lambda c: c.name)
def test_fm_port_equals_reference(case, port):
    g = FM_GOLD[case.name]
    x = case.make_input()
    assert digest(x) == g["input_sha256"], "synthetic generator drifted"
    a, la, ha = port.fm_run(case.params, x, case.chunk_int16, return_chunks=True)
    assert [int(v) for v in la] == g["chunk_result_len"]
    assert [int(v) for v in ha] == g["squelch_hits"]
    assert a.size == g["n_out"]
    assert digest(a) == g["output_sha256"]      # bit-exact incl. the atan2 path


@pytest.mark.parametrize("case", (fm_cases() + fm_optional_cases())[::2], ids=lambda c: c.name)
def test_fm_levels_port_equals_reference(case, port):
    # the per-chunk `sr` behind the -L statistics (src/rtl_fm.c:792-806)
    x = case.make_input()
    a = port.fm_levels(case.params, x, case.chunk_int16)
    b = np.array(PIN["fm_levels"][case.name])
    assert a.size == b.size and a.size >= 1
    assert np.array_equal(a, b)
    assert b.max() > 0 or case.name.startswith("zeros")      # an all-zero capture has level 0


def test_derivation_matches_optimal_settings():
    from rx_tools_b200 import fm
    combos = [dict(rate_s=1024000, rate_r=24000), dict(wbfm=1), dict(wbfm=1, rate_s=2400000, rate_r=48000),
              dict(wbfm=1, rate_s=300000, rate_r=48000, use_F=1, comp_fir_size=9), dict(rate_s=24000),
              dict(rate_s=24000, custom_atan=2), dict(mode=oracle.MODE_AM, rate_s=12000),
              dict(mode=oracle.MODE_USB, rate_s=48000, use_F=1, comp_fir_size=0),
              dict(wbfm=1, time_constant_us=50), dict(rate_s=170000, post_downsample=4, deemph=1)]
    assert [g["cli"] for g in PIN["derive"]] == combos
    for kw, g in zip(combos, PIN["derive"]):
        want = oracle.FmParams(**g["params"])
        got = fm.derive_params(**kw)
        mine = dataclasses.asdict(got.params)
        assert mine.pop("report_levels") == 0          # library-only switch, not a reference field
        assert mine == dataclasses.asdict(want), (kw, got.params, want)
        assert got.capture_rate == g["capture_rate"] and got.capture_freq_offset == g["capture_freq_offset"], kw


# ------------------------------------------------------------------------- rx_power
from cases import power_cases, power_input  # noqa: E402


def _window_table(port, case, n):
    return port.window_table(case.window, n)


@pytest.mark.parametrize("case", power_cases(), ids=lambda c: c.name)
def test_power_port_equals_reference(case, port):
    g = PIN["power"][case.name]
    n = 1 << g["bin_e"]
    win = _window_table(port, case, n)
    assert digest(win) == g["window_sha256"]
    if g["bin_e"] > 0:
        assert digest(port.sine_table(g["bin_e"])) == g["sine_sha256"]
    x = power_input(case, g["tune_count"], g["buf_len"])
    p = oracle.PowerParams(bin_e=g["bin_e"], buf_len=g["buf_len"], downsample=g["downsample"],
                           downsample_passes=g["downsample_passes"], comp_fir_size=case.comp_fir_size,
                           boxcar=case.boxcar, peak_hold=case.peak_hold)
    avg_p, smp_p = port.power_scan(p, win, x, case.n_pass, g["tune_count"])
    assert [int(v) for v in smp_p] == g["samples"]
    assert digest(avg_p) == g["avg_sha256"]
    assert avg_p.any()


@pytest.mark.parametrize("m", [1, 2, 5, 10, 12])
def test_fix_fft_port_equals_reference(m, port):
    g = PIN["fix_fft"][str(m)]
    rng = np.random.default_rng(m)
    iq = rng.integers(-32768, 32768, size=2 << m, dtype=np.int32).astype(np.int16)
    assert digest(port.fix_fft(iq, m)) == g["sha256"]
    # smaller transform inside a larger sine table (fix_fft allows n < N_WAVE)
    if m > 2:
        iq2 = iq[: 2 << (m - 2)]
        assert digest(port.fix_fft(iq2, m - 2, m)) == g["inner_sha256"]


# ---- rx_sdr conversions (src/rtl_sdr.c:348-391): they live inline in main(), so the pin is what the reference's own
# executable wrote recording from the replay device (tests/golden/sdr_golden.json)
def _port_sdr(port, name, src, dst, count):
    import ctypes as C
    f = getattr(port.L, name)
    f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
    f.restype = None
    f(src.ctypes.data, count, dst.ctypes.data)
    return dst


def test_sdr_conversions_port_equals_reference_executable(port):
    import sdr_inputs as SI
    g = json.load(open(os.path.join(G, "sdr_golden.json")))
    x = SI.cs16_capture()
    n = SI.N_ELEMS
    for fmt, name, dt in (("CS8", "orx_sdr_cs16_to_cs8", np.uint8), ("CU8", "orx_sdr_cs16_to_cu8", np.uint8),
                          ("CF32", "orx_sdr_cs16_to_cf32", np.float32)):
        ref = g["CS16_" + fmt]
        assert (digest(x), ref["n_elems"]) == (ref["input_sha256"], n)
        mine = _port_sdr(port, name, np.ascontiguousarray(x[:2 * n]), np.empty(2 * n, dt), 2 * n).view(np.uint8)
        assert (mine.size, digest(mine)) == (ref["n_bytes"], ref["output_sha256"]), fmt
    y = SI.cs12_capture()
    n12 = SI.N_ELEMS_12
    ref = g["CS12_CS16"]
    assert (digest(y), ref["n_elems"]) == (ref["input_sha256"], n12)
    mine = _port_sdr(port, "orx_sdr_cs12_to_cs16", y, np.empty(2 * n12, np.int16), n12).view(np.uint8)
    assert (mine.size, digest(mine)) == (ref["n_bytes"], ref["output_sha256"])


def test_sdr_conversions_port_equals_golden(port):
    import json
    import sdr_inputs as SI
    from rx_tools_b200.synth import digest
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sdr_golden.json")))
    x, n = SI.cs16_capture(), SI.N_ELEMS
    assert digest(x) == g["CS16_CS8"]["input_sha256"]
    for fmt, name, dt in (("CS8", "orx_sdr_cs16_to_cs8", np.uint8), ("CU8", "orx_sdr_cs16_to_cu8", np.uint8),
                          ("CF32", "orx_sdr_cs16_to_cf32", np.float32)):
        mine = _port_sdr(port, name, np.ascontiguousarray(x[:2 * n]), np.empty(2 * n, dt), 2 * n)
        assert digest(mine.view(np.uint8)) == g["CS16_" + fmt]["output_sha256"], fmt
    y, n12 = SI.cs12_capture(), SI.N_ELEMS_12
    mine = _port_sdr(port, "orx_sdr_cs12_to_cs16", y, np.empty(2 * n12, np.int16), n12)
    assert digest(mine.view(np.uint8)) == g["CS12_CS16"]["output_sha256"]


@pytest.mark.parametrize("freq", ["100M:102.8M:40", "100M:100.4M:2"])
def test_power_port_equals_reference_beyond_65536_bins(freq, port):
    """bin_e 17 / 18 (hop buffers of 0.5 / 7 MB, the second one boxcar-decimated by 7): the shapes the library serves from
    global memory (tests/test_power_gpu.py::test_hop_buffers_beyond_shared_memory)."""
    g = PIN["power_big_bins"][freq]
    assert g["bin_e"] >= 17
    rng = np.random.default_rng(g["bin_e"])
    x = rng.integers(-3000, 3001, size=(2, g["tune_count"], g["buf_len"]), dtype=np.int32).astype(np.int16)
    win = port.window_table("blackman", 1 << g["bin_e"])
    assert digest(win) == g["window_sha256"]
    pp = oracle.PowerParams(bin_e=g["bin_e"], buf_len=g["buf_len"], downsample=g["downsample"],
                            downsample_passes=g["downsample_passes"])
    a2, s2 = port.power_scan(pp, win, x, 2, g["tune_count"])
    assert [int(v) for v in s2] == g["samples"] and digest(a2) == g["avg_sha256"]
