"""Host-side arithmetic of librxb200 (planner, tables, CSV formatter, scale identity) against the
port oracle and the golden files.  CPU only."""
import json
import os

import numpy as np
import pytest

from cases import power_cases
from rx_tools_b200 import power
from rx_tools_b200.synth import digest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PW_GOLD = json.load(open(os.path.join(G, "power_golden.json")))


@pytest.mark.parametrize("case", power_cases(), ids=lambda c: c.name)
def test_planner_matches_reference_plan(case):
    g = PW_GOLD[case.name]
    plan = power.plan_range(case.freq_arg, case.crop, case.boxcar, case.comp_fir_size, case.peak_hold)
    assert (plan.n_hops, plan.bin_e, plan.buf_len, plan.downsample, plan.downsample_passes, plan.rate) == \
        (g["tune_count"], g["bin_e"], g["buf_len"], g["downsample"], g["downsample_passes"], g["rate"])
    if plan.bin_e:
        assert digest(power.window_table(case.window, 1 << plan.bin_e)) == g["window_sha256"]


def test_cfg4_plan_is_871_hops():
    plan = power.plan_range("24M:1766M:1k", 0.285)
    assert (plan.n_hops, plan.bin_e, plan.buf_len, plan.rate) == (871, 12, 16384, 2797202)


@pytest.mark.parametrize("log2n", [1, 4, 10, 12, 15])
def test_sine_table_matches_port(log2n, port):
    assert np.array_equal(power.sine_table(log2n), port.sine_table(log2n))


@pytest.mark.parametrize("name", sorted(power.WINDOWS))
def test_window_tables_match_port(name, port):
    for n in (2, 256, 1024, 4096):
        assert np.array_equal(power.window_table(name, n), port.window_table(name, n))


def test_planner_and_csv_match_reference(port):
    """Plans, hop frequencies and csv_dbm() text against what the reference computed (tests/golden/ref_pin.json)."""
    import oracle
    pin = json.load(open(os.path.join(G, "ref_pin.json")))
    args = [("24M:1766M:1k", 0.285, 1, 0), ("24M:1766M:1k", 0.0, 1, 0), ("88M:108M:10k", 0.1, 1, 0),
            ("100M:100.2M:50", 0.0, 0, 9), ("433M:434M:100", 0.2, 1, 0), ("100M:120M:2M", 0, 1, 0)]
    assert [(g["freq_arg"], g["crop_arg"], g["boxcar"], g["comp_fir_size"]) for g in pin["planner"]] == args
    for (arg, crop, boxcar, fir), rp in zip(args, pin["planner"]):
        plan = power.plan_range(arg, crop, boxcar, fir, 0)
        assert (plan.n_hops, plan.bin_e, plan.buf_len, plan.downsample, plan.downsample_passes, plan.rate) == \
            (rp["tune_count"], rp["bin_e"], rp["buf_len"], rp["downsample"], rp["downsample_passes"], rp["rate"]), arg
        assert abs(plan.crop - rp["crop"]) < 1e-15
        freqs = np.array([plan.hop_freq(i) for i in range(plan.n_hops)], dtype=np.int64)
        assert digest(freqs) == rp["hop_freqs_sha256"]
    # CSV text identical for the same accumulators
    g = pin["csv"]
    plan = power.plan_range(g["freq_arg"], g["crop"])
    rng = np.random.default_rng(g["seed"])
    x = rng.integers(-100, 101, size=(2, plan.n_hops, plan.buf_len), dtype=np.int32).astype(np.int16)
    pp = oracle.PowerParams(bin_e=plan.bin_e, buf_len=plan.buf_len, downsample=plan.downsample,
                            downsample_passes=plan.downsample_passes)
    avg, smp = port.power_scan(pp, port.window_table("hamming", 1 << plan.bin_e), x, 2, plan.n_hops)
    assert digest(avg) == g["avg_sha256"] and [int(v) for v in smp] == g["samples"]
    mine = power.csv_rows(plan, avg, smp)
    assert digest(np.frombuffer(mine.encode(), dtype=np.uint8)) == g["text_sha256"]


def test_wbfm_preset_keeps_a_later_squelch_level():
    """-M wbfm zeroes squelch_level when it is parsed (src/rtl_fm.c:1331-1341); `-M wbfm -l 50` keeps 50.  The parse-order
    rule lives in the shell (host/rx_fm_b200.c), rxb200_fm_derive passes cli.squelch_level through."""
    from rx_tools_b200 import fm
    assert fm.derive_params(wbfm=1, squelch_level=50).params.squelch_level == 50
    assert fm.derive_params(wbfm=1).params.squelch_level == 0


def test_deemph_fp32_identity():
    """The CUDA back end runs deemph_filter (src/rtl_fm.c:667-682) for odd a as  U' = fma(X - U, fl(1/a), U)  in FP32
    with U = 2^23 + 32768 + avg (csrc/fm_kernels.cu, DeemphOp<false, true>).  That is exact iff rounding d * fl(1/a) to
    the nearest integer equals the reference's trunc((d +- a/2) / a) for every difference d of two int16 values: checked
    here for every d and a spread of odd a (the kernels' own parity tests cover a = 23 and a = 181 on the GPU)."""
    d = np.arange(-65535, 65536, dtype=np.int64)
    for a in list(range(1, 400, 2)) + [1023, 1801, 4095, 18001, 32767]:
        inv = np.float64(np.float32(1.0) / np.float32(a))
        h = a // 2
        num = np.where(d > 0, d + h, d - h)
        ref = np.sign(num) * (np.abs(num) // a)            # C's truncating division
        y = d.astype(np.float64) * inv                     # exact: 17 x 24 significant bits
        assert np.array_equal(np.rint(y).astype(np.int64), ref), a
        # no tie in sight: the nearest half-integer is further away than any rounding of the fma could reach
        assert np.min(np.abs((y - np.floor(y)) - 0.5)) > 65536 * 2.0 ** -24 / a


def _fast_atan2_ref(y, x):
    """fast_atan2 (src/rtl_fm.c:485-506) on int64 arrays, C's truncating division."""
    ya = np.abs(y)
    num = np.where(x >= 0, 4096 * (x - ya), 4096 * (x + ya))
    den = np.where(x >= 0, x + ya, ya - x)
    den1 = np.where(den == 0, 1, den)
    q = np.sign(num) * (np.abs(num) // den1)
    ang = np.where(x >= 0, 4096 - q, 12288 - q)
    ang = np.where(y < 0, -ang, ang)
    return np.where((x == 0) & (y == 0), 0, ang)


def _fast_atan2_f32(y, x, ulp_shift):
    """The FP32 restatement the CUDA front end uses where the operands are exact in a float (fast_atan2_f32,
    csrc/fm_kernels.cu), step for step in numpy float32; `ulp_shift` moves the reciprocal estimate by that many ulps
    (the hardware's rcp.approx is within one ulp of the rounded reciprocal)."""
    f = np.float32
    x = x.astype(f); y = y.astype(f)
    ax, ay = np.abs(x), np.abs(y)
    den = ax + ay
    n = ax - ay
    an = np.abs(n) * f(4096.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        rc = (f(1.0) / den).astype(f)
        rc = np.where(np.isfinite(rc), (rc.view(np.int32) + ulp_shift).view(f), rc)
        te = (an * rc).astype(f)
        te = (te.astype(np.float64) * (1.0 - 2.0 ** -20)).astype(f)          # fma(te, -2^-20, te)
        T = np.floor(te).astype(f)                                            # round-down add of 1.5 * 2^23, minus it
        rem = an.astype(np.float64) - T.astype(np.float64) * den.astype(np.float64)   # fma(-T, den, an): exact
        T = np.where(rem >= den, T + f(1.0), T)
        Ts = np.where(n < 0, -T, T)
        ang = np.where(x >= 0, f(4096.0) - Ts, f(12288.0) + Ts)
        r = np.where(y < 0, -ang, ang)
    return np.where(den == 0, 0, r).astype(np.int64)


def test_fast_atan2_fp32_form():
    rng = np.random.default_rng(7)
    # every pair of small operands, then random pairs over the whole range the undecimated shape can produce (|.| <= 2^15),
    # the quadrant edges and the ratios whose quotient is an exact integer
    g = np.arange(-260, 261, dtype=np.int64)
    xs, ys = [np.repeat(g, g.size)], [np.tile(g, g.size)]
    xs.append(rng.integers(-32768, 32769, 4_000_000)); ys.append(rng.integers(-32768, 32769, 4_000_000))
    k = rng.integers(1, 4097, 500_000); d = rng.integers(1, 16, 500_000) * 4096          # n / den = k / 4096 exactly
    xs.append((d + k * (d // 4096)) // 2); ys.append((d - k * (d // 4096)) // 2)
    edge = np.array([-32768, -32767, -1, 0, 1, 32767, 32768], dtype=np.int64)
    xs.append(np.repeat(edge, edge.size)); ys.append(np.tile(edge, edge.size))
    x = np.concatenate(xs); y = np.concatenate(ys)
    want = _fast_atan2_ref(y, x)
    for shift in (-1, 0, 1):
        assert np.array_equal(_fast_atan2_f32(y, x, shift), want), shift


def test_row_discriminator_operands_fit_fp32():
    """The row front end (csrc/fm_rows.cuh) runs fast_atan2 in FP32 without a range check: its operands must stay below 2^24.
    The chain from the 8-bit-range samples (|x| <= 128, src/rtl_fm.c:846) to the discriminator is linear with non-negative
    half-band taps (fifth_order, :411-440) followed by the droop FIR (generic_fir, :442-465; the product's copy of
    cic_9_tables is read from csrc/fm_kernels.cu), so |d| <= 128 * sum|g| for the combined response g, plus the floors'
    slack; the conjugate product's components obey |cr| + |cj| <= (|di| + |dq|)(|bi| + |bq|) <= 4 d^2."""
    import re
    src = open(os.path.join(os.path.dirname(__file__), "..", "rx_tools_b200", "csrc", "fm_kernels.cu")).read()
    body = re.search(r"k_droop9_host\[11\]\[10\] = \{(.*?)\n\};", src, re.S).group(1)
    table = [[int(v) for v in row.split(",") if v.strip()] for row in re.findall(r"\{(\s*-?\d+\s*(?:,\s*-?\d+\s*)*)\}", body)]
    b = np.array([1, 5, 10, 10, 5, 1], dtype=np.float64) / 16.0

    def up(v, k):
        o = np.zeros((len(v) - 1) * k + 1)
        o[::k] = v
        return o

    for P in (1, 2, 3):                                    # the row front end's instantiations
        h = np.array([1.0])
        for lvl in range(P):
            h = np.convolve(h, up(b, 2 ** lvl))
        assert abs(128 * np.abs(h).sum() - 128 * 2 ** P) < 1e-9          # without the FIR: |d| <= 128 << P
        c = np.array(table[P][1:10], dtype=np.float64) / 32768.0
        assert table[P][0] == 9 and np.array_equal(c, c[::-1])
        g = np.convolve(up(c, 2 ** P), h)
        floors = sum(2 ** (P - 1 - lvl) for lvl in range(P)) * np.abs(c).sum() + 1      # one unit per floor, amplified downstream
        dmax = 128 * np.abs(g).sum() + floors
        assert 4 * dmax * dmax < 2 ** 24, (P, dmax)


def test_resampler_group_closed_form():
    """fm_back_kernel knows where a lane stops before it starts: n outputs of low_pass_real (src/rtl_fm.c:396-407) end with the
    first sample that takes the running phase to n * fast, i.e. after ceil((n * fast - phase) / slow) samples (win_outputs,
    csrc/fm_kernels.cu).  Checked against the reference's loop for integer and fractional rate ratios."""
    rng = np.random.default_rng(3)
    for fast, slow in [(2_400_000, 48_000), (300_000, 48_000), (170_000, 32_000), (1_024_000, 24_000), (1_200_000, 44_100)]:
        for _ in range(50):
            phase = int(rng.integers(0, slow))             # a piece starts right after an emission: phase < slow
            n = int(rng.integers(1, 200))
            ph, samples, outs = phase, 0, 0
            while outs < n:                                # the reference's loop
                samples += 1
                ph += slow
                if ph >= fast:
                    ph -= fast
                    outs += 1
            assert samples == (n * fast - phase + slow - 1) // slow, (fast, slow, phase, n)


def test_polar_disc_fp32_form():
    """polar_discriminant (src/rtl_fm.c:476-483: (int)(atan2(cj, cr) / 3.14159 * 2^14)) as the CUDA path evaluates it for operands
    that are exact in a float (disc_std_f32, csrc/fm_kernels.cu): an FP32 estimate assembled as integer part + fraction, and a
    guard band inside which the fp64 form decides.  Restated here step for step in numpy float32 (constants copied from the
    kernel); outside the guard band the result must equal the fp64 truncation for every operand pair, whatever the reciprocal
    estimate's last bit, and the guard band must stay a small fraction of the samples."""
    f = np.float32
    q_coef = [f(c) for c in (-0.3333333134651184, 0.1999976634979248, -0.14279110729694366, 0.11037992686033249,
                             -0.08673165738582611, 0.06284350901842117, -0.03627006709575653, 0.013750223442912102,
                             -0.002447017002850771)]
    khi, klo = f(5215.193359375), f(0.00022094578889664263)
    one_c2, one_c4, delta = f(1.0069195032119751), f(1.0138390064239502), f(1.5e-3)
    src = open(os.path.join(os.path.dirname(__file__), "..", "rx_tools_b200", "csrc", "fm_kernels.cu")).read()
    for lit in ("-0.002447017002850771f", "5215.193359375f", "0.00022094578889664263f", "1.0069195032119751f",
                "1.0138390064239502f", "1.5e-3f", "0.1999976634979248f"):
        assert lit in src, lit                         # the kernel still uses these constants

    def fma(a, b, c):
        return (a.astype(np.float64) * np.float64(b) + np.float64(c)).astype(f) if np.isscalar(b) or np.ndim(b) == 0 else \
            (a.astype(np.float64) * b.astype(np.float64) + (c.astype(np.float64) if np.ndim(c) else np.float64(c))).astype(f)

    def form(y, x, ulp):
        ax, ay = np.abs(x.astype(f)), np.abs(y.astype(f))
        a, b = np.minimum(ax, ay), np.maximum(ax, ay)
        r = (f(1) / b).astype(f)
        r = (r.view(np.int32) + ulp).view(f)
        t0 = (a * r).astype(f)
        t = fma(fma(-t0, b, a), r, t0)
        u = (t * t).astype(f)
        q = np.full_like(u, q_coef[-1])
        for c in q_coef[-2::-1]:
            q = fma(q, u, np.full_like(u, c))
        p = fma((t * u).astype(f), q, t)
        n1 = np.floor((p * khi).astype(f)).astype(f)
        fr = fma(p, np.full_like(p, klo), fma(p, np.full_like(p, khi), -n1))
        n = n1.astype(np.int64)
        swap, neg = ay > ax, x < 0
        n = np.where(swap, 8191 - n, n)
        fr = np.where(swap, (one_c2 - fr).astype(f), fr)
        n = np.where(neg, 16383 - n, n)
        fr = np.where(neg, (one_c4 - fr).astype(f), fr)
        rr = np.rint(fr)
        sure = np.abs(fr - rr) >= delta
        k = n + rr.astype(np.int64) - (fr < rr)
        return np.where(y < 0, -k, k), sure

    rng = np.random.default_rng(5)
    g = np.arange(-150, 151, dtype=np.int64)
    sets = [(np.repeat(g, g.size), np.tile(g, g.size)),
            (rng.integers(-32768, 32769, 3_000_000), rng.integers(-32768, 32769, 3_000_000)),
            (rng.integers(-300, 301, 1_000_000), rng.integers(-32768, 32769, 1_000_000)),
            (rng.integers(-(1 << 24) + 1, 1 << 24, 1_000_000), rng.integers(-(1 << 24) + 1, 1 << 24, 1_000_000))]
    total = unsure = 0
    for y, x in sets:
        keep = ~((y == 0) & (x >= 0))                  # the kernel returns 0 for these before anything else
        y, x = y[keep], x[keep]
        want = np.trunc(np.arctan2(y.astype(np.float64), x.astype(np.float64)) / 3.14159 * 16384).astype(np.int64)
        for ulp in (-1, 0, 1):
            k, sure = form(y, x, ulp)
            assert np.array_equal(k[sure], want[sure]), ulp
            total += y.size
            unsure += int((~sure).sum())
    assert unsure < 0.006 * total
