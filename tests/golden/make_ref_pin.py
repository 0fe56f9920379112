"""Mint tests/golden/ref_pin.json from the UNMODIFIED reference (oracle/_ref): what tests/test_oracle_pin.py and
tests/test_host_logic.py::test_planner_and_csv_match_reference compare the port and the host planner against, beyond
what fm_golden.json / power_golden.json / sdr_golden.json already hold (tables, per-chunk levels, the parameter
derivation, sine tables, fix_fft, the plans and hop frequencies, the CSV text).

Run where the reference sources are available (oracle/_ref built):  python tests/golden/make_ref_pin.py"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import oracle  # noqa: E402
from cases import fm_cases, fm_optional_cases, power_cases, power_input  # noqa: E402
from rx_tools_b200.synth import digest  # noqa: E402

# the CLI combinations of test_derivation_matches_optimal_settings
DERIVE_COMBOS = [dict(rate_s=1024000, rate_r=24000), dict(wbfm=1), dict(wbfm=1, rate_s=2400000, rate_r=48000),
                 dict(wbfm=1, rate_s=300000, rate_r=48000, use_F=1, comp_fir_size=9), dict(rate_s=24000),
                 dict(rate_s=24000, custom_atan=2), dict(mode=oracle.MODE_AM, rate_s=12000),
                 dict(mode=oracle.MODE_USB, rate_s=48000, use_F=1, comp_fir_size=0),
                 dict(wbfm=1, time_constant_us=50), dict(rate_s=170000, post_downsample=4, deemph=1)]
# the ranges of test_planner_and_csv_match_reference: (freq_arg, crop, boxcar, comp_fir_size)
PLANNER_ARGS = [("24M:1766M:1k", 0.285, 1, 0), ("24M:1766M:1k", 0.0, 1, 0), ("88M:108M:10k", 0.1, 1, 0),
                ("100M:100.2M:50", 0.0, 0, 9), ("433M:434M:100", 0.2, 1, 0), ("100M:120M:2M", 0, 1, 0)]
BIG_BINS = ["100M:102.8M:40", "100M:100.4M:2"]
FFT_M = [1, 2, 5, 10, 12]


def _plan_fields(p):
    return dict(tune_count=p.tune_count, bin_e=p.bin_e, buf_len=p.buf_len, downsample=p.downsample,
                downsample_passes=p.downsample_passes, rate=p.rate)


def main():
    oracle.build()
    assert oracle.have_ref(), "needs oracle/_ref"
    rf, rp, port = oracle.RefFm(), oracle.RefPower(), oracle.port()
    out = {}
    out["tables"] = dict(atan_sha256=digest(rf.atan_table()), cic9=[[int(v) for v in rf.cic9(r)] for r in range(11)])

    fm_gold = json.load(open(os.path.join(HERE, "fm_golden.json")))
    levels = {}
    for c in fm_cases() + fm_optional_cases():
        x = c.make_input()
        y, lens, hits = rf.run(c.params, x, c.chunk_int16, return_chunks=True)
        g = fm_gold[c.name]          # the pin of test_fm_port_equals_reference lives in fm_golden.json
        assert (digest(x), digest(y), [int(v) for v in lens], [int(v) for v in hits]) == \
            (g["input_sha256"], g["output_sha256"], g["chunk_result_len"], g["squelch_hits"]), c.name
    for c in (fm_cases() + fm_optional_cases())[::2]:
        levels[c.name] = [int(v) for v in rf.levels(c.params, c.make_input(), c.chunk_int16)]
    out["fm_levels"] = levels

    derive = []
    for kw in DERIVE_COMBOS:
        want, cap_rate, cap_off = rf.derive(**kw)
        derive.append(dict(cli=kw, params=want.__dict__, capture_rate=cap_rate, capture_freq_offset=cap_off))
    out["derive"] = derive

    pw = {}
    for c in power_cases():
        custom = None
        if c.window == "hann":
            p0 = rp.setup(c.freq_arg, c.crop, c.boxcar, c.comp_fir_size, c.peak_hold, "rectangle")
            custom = port.window_table("hann", 1 << p0.bin_e)
        plan = rp.setup(c.freq_arg, c.crop, c.boxcar, c.comp_fir_size, c.peak_hold,
                        c.window if custom is None else "rectangle", custom)
        n = 1 << plan.bin_e
        win, sine = rp.tables()
        avg, smp = rp.scan(power_input(c, plan.tune_count, plan.buf_len), c.n_pass)
        pw[c.name] = dict(_plan_fields(plan), window_sha256=digest(win), sine_sha256=digest(sine[: n * 3 // 4]),
                          avg_sha256=digest(avg), samples=[int(v) for v in smp])
    out["power"] = pw

    fft = {}
    for m in FFT_M:
        rng = np.random.default_rng(m)
        iq = rng.integers(-32768, 32768, size=2 << m, dtype=np.int32).astype(np.int16)
        fft[str(m)] = dict(sha256=digest(rp.fix_fft(iq, m)))
        if m > 2:
            fft[str(m)]["inner_sha256"] = digest(rp.fix_fft(iq[: 2 << (m - 2)], m - 2, m))
    out["fix_fft"] = fft

    big = {}
    for freq in BIG_BINS:
        plan = rp.setup(freq, 0.0, 1, 0, 0, "blackman")
        rng = np.random.default_rng(plan.bin_e)
        x = rng.integers(-3000, 3001, size=(2, plan.tune_count, plan.buf_len), dtype=np.int32).astype(np.int16)
        avg, smp = rp.scan(x, 2)
        win, _ = rp.tables()
        big[freq] = dict(_plan_fields(plan), window_sha256=digest(win), avg_sha256=digest(avg),
                         samples=[int(v) for v in smp])
    out["power_big_bins"] = big

    planner = []
    for arg, crop, boxcar, fir in PLANNER_ARGS:
        plan = rp.setup(arg, crop, boxcar, fir, 0, "hamming")
        planner.append(dict(freq_arg=arg, crop_arg=crop, boxcar=boxcar, comp_fir_size=fir, **_plan_fields(plan),
                            crop=plan.crop, hop_freqs_sha256=digest(rp.hop_freqs().astype(np.int64))))
    out["planner"] = planner
    # csv_dbm() text over the accumulators of a seeded scan
    import tempfile
    rp.setup("24M:60M:1k", 0.285, 1, 0, 0, "hamming")
    rng = np.random.default_rng(5)
    x = rng.integers(-100, 101, size=(2, rp.plan.tune_count, rp.plan.buf_len), dtype=np.int32).astype(np.int16)
    avg, smp = rp.scan(x, 2)
    with tempfile.TemporaryDirectory() as td:
        text = rp.csv(os.path.join(td, "ref.csv"))
    out["csv"] = dict(freq_arg="24M:60M:1k", crop=0.285, seed=5, avg_sha256=digest(avg), samples=[int(v) for v in smp],
                      text_sha256=digest(np.frombuffer(text.encode(), dtype=np.uint8)))

    with open(os.path.join(HERE, "ref_pin.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote ref_pin.json:", {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
