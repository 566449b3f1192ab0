"""-m "not gpu": the CPU oracle against (a) the committed golden fixtures produced by the reference itself,
(b) the stored outputs of the reference built as a library (tests/golden/reference_runs.json), (c) known-answer vectors."""
import json
import zlib
from pathlib import Path

import numpy as np
import pytest

from oraclelib import Oracle
from paritylib import diff_bufres, diff_digests, diff_frames, diff_stats, digest, record_digests, reference_runs
from readsb_b200 import synth

GOLDEN = sorted(p for p in (Path(__file__).parent / "golden").glob("*.npz") if p.stem not in ("beast_stream", "sc16_converters"))


def load_golden(path):
    z = np.load(path)
    meta = json.loads(bytes(z["meta"]).decode())
    return z, meta


@pytest.mark.parametrize("path", GOLDEN, ids=[p.stem for p in GOLDEN])
def test_oracle_matches_golden(path):
    z, meta = load_golden(path)
    o = Oracle(**meta["options"])
    frames, bufres = o.run_stream(np.ascontiguousarray(z["iq"]), meta["buf_samples"])
    # flags (ICAO_ADDED) is this repo's annotation, everything else is the reference's own output
    problems = diff_frames(frames, z["frames"], fields=("timestamp", "j", "crc", "addr", "score", "buffer_seq", "signal_len",
                                                        "phase", "msgtype", "msgbits", "correctedbits", "fix_bit", "msg"))
    assert not problems, "\n".join(problems)
    # signalLevel: same fp64 expression as demod_2400.c:448-449
    level = frames["sigpow_sum"] / 65535.0 / 65535.0 / frames["signal_len"]
    assert np.array_equal(level, z["signal_level"])
    # converter outputs (convert.c:100-107)
    assert np.array_equal(bufres["sum_level"] / 65536.0 / bufres["length"], z["mean_level"])
    assert np.array_equal(bufres["sum_power"] / 65535.0 / 65535.0 / bufres["length"], z["mean_power"])
    assert np.array_equal(bufres["n_frames"], z["bufres"]["n_frames"])
    assert np.array_equal(bufres["icao_flipped"], z["bufres"]["icao_flipped"])
    st = o.stats()
    for k, v in meta["stats"].items():
        if k in ("sum_signal_power", "reserved_", "demod_modeac", "peak_signal_power"):
            continue
        assert st[k] == v, k
    assert st["peak_signal_power"] == meta["dstats"]["peak_signal_power"]
    # noise_power_sum (demod_2400.c:474-479) re-accumulated in the reference's order from the exact integers
    noise = 0.0
    for b in bufres:
        noise += (b["sum_power"] / 65535.0 / 65535.0 / b["length"]) * b["length"] - b["sum_signal_power"] / 65535.0 / 65535.0
    assert noise == meta["dstats"]["noise_power_sum"]


@pytest.mark.parametrize("path", GOLDEN, ids=[p.stem for p in GOLDEN])
def test_oracle_modeac_matches_golden(path):
    """demodulate2400AC (demod_2400.c:575-761): the reference's replies on every fixture (most hold none, modeac_mix many)."""
    z, meta = load_golden(path)
    got = Oracle(**meta["options"]).run_stream_ac(np.ascontiguousarray(z["iq"]), meta["buf_samples"])
    want = z["modeac"]
    assert len(got) == len(want)
    assert np.array_equal(got["timestamp"], want["timestamp"]) and np.array_equal(got["modeac"], want["modeac"])
    assert np.array_equal(got["buffer_idx"], want["buffer_idx"])
    if path.stem == "modeac_mix":
        assert len(want) > 15


def test_oracle_beast_matches_reference_network_output():
    """SURVEY 8(f) row 4: the bytes the reference program itself sent to a beast_out TCP client (--net-verbatim --modeac,
    tests/golden/make_beast_golden.py) == oracle frames + Mode A/C replies through the oracle's Beast encoder."""
    z = np.load(Path(__file__).parent / "golden" / "beast_stream.npz")
    meta = json.loads(bytes(z["meta"]).decode())
    iq = np.concatenate([np.full(2 * meta["silence_samples"], 127, np.uint8), z["traffic"]])
    buf = 131072                                               # the reference's default --sdr-buffer-size
    frames, _ = Oracle().run_stream(iq, buf)
    modeac = Oracle().run_stream_ac(iq, buf)
    got = Oracle.beast(frames, modeac, verbatim=True)
    assert meta["n_records"] == len(frames) + len(modeac) > 100
    assert got == bytes(z["beast"])
    assert Oracle.beast(frames, modeac, verbatim=False) != got   # the fixture holds repaired frames: corrected bytes differ


def test_beast_escaping_and_signal_byte():
    from readsb_b200.abi import FRAME_DTYPE, MODEAC_DTYPE
    f = np.zeros(1, FRAME_DTYPE)
    f["timestamp"] = 0x1A001A1A00FF; f["msgbits"] = 56; f["signal_len"] = 134; f["fix_bit"] = -1
    f["msg"][0, :7] = [0x1A, 0x5D, 0x1A, 0, 0, 0, 0x1A]
    f["sigpow_sum"] = int(0.25 * 65535 * 65535 * 134)          # signalLevel 0.25 -> sqrt 0.5 -> 127.5 -> nearbyint: 128 (half to even)
    rec = Oracle.beast(f)
    assert rec[:2] == b"\x1a2" and rec[2:].count(b"\x1a\x1a") == 6
    body = rec[2:].replace(b"\x1a\x1a", b"\x1a")
    assert body[:6] == bytes([0x1A, 0x00, 0x1A, 0x1A, 0x00, 0xFF]) and body[6] in (127, 128) and body[7:] == bytes([0x1A, 0x5D, 0x1A, 0, 0, 0, 0x1A])
    f["sigpow_sum"] = 1                                         # tiny but non-zero power: the byte is clamped up to 1
    assert Oracle.beast(f)[2:].replace(b"\x1a\x1a", b"\x1a")[6] == 1
    a = np.zeros(1, MODEAC_DTYPE); a["timestamp"] = 5; a["modeac"] = 0x1A7F
    assert Oracle.beast(np.zeros(0, FRAME_DTYPE), a) == bytes([0x1A, 0x31, 0, 0, 0, 0, 0, 5, 0, 0x1A, 0x1A, 0x7F])


@pytest.mark.parametrize("q11", [0, 1])
def test_oracle_sc16_converters_match_golden(q11):
    z = np.load(Path(__file__).parent / "golden" / "sc16_converters.npz")
    iq = z[f"iq{q11}"]; n = iq.size // 2
    mag, sl, sp = Oracle.convert_sc16(iq, bool(q11))
    assert np.array_equal(mag, z[f"mag{q11}"])
    assert float(np.float32(sl) / np.float32(n)) == z[f"means{q11}"][0] and float(np.float32(sp) / np.float32(n)) == z[f"means{q11}"][1]


def test_lut_known_answer():
    lut = Oracle.lut()
    assert zlib.crc32(lut.tobytes()) == 0x8E9D21E1            # SURVEY.md 8a a1, probed on the reference
    assert lut.min() == 363 and lut.max() == 65535
    full = lut.reshape(256, 256)
    assert np.array_equal(full, full.T) and np.array_equal(full, full[::-1, :]) and np.array_equal(full, full[:, ::-1])


CRC_KATS = [  # SURVEY.md 8a a11
    ("8D4840D6202CC371C32CE0576098", 0), ("8D40621D58C382D690C8AC2863A7", 0), ("5D4840D6F8740F", 0),
]
BIT_SYNDROMES_112 = {0: 0x3935EA, 1: 0x1C9AF5, 5: 0x9E31E9, 8: 0x2C38BC, 31: 0x7EDA22, 32: 0x3F6D11, 87: 0xFFF409, 88: 0x800000, 111: 0x000001}
BIT_SYNDROMES_56 = {0: 0x018567, 5: 0xAFF54C, 8: 0xEA04AD}


def test_crc_known_answers():
    for hexmsg, want in CRC_KATS:
        assert Oracle.crc24(bytes.fromhex(hexmsg)) == want
    for nbits, table in ((112, BIT_SYNDROMES_112), (56, BIT_SYNDROMES_56)):
        for bit, syn in table.items():
            m = bytearray(nbits // 8)
            m[bit >> 3] = 1 << (7 - (bit & 7))
            assert Oracle.crc24(bytes(m)) == syn
            assert Oracle.diagnose1(syn, nbits) == (bit if bit >= 5 else -2)   # DF bits are never corrected (crc.c:210)
    assert Oracle.diagnose1(0, 112) == -1 and Oracle.diagnose1(0x123456, 112) == -2


def test_synth_frames_have_valid_parity():
    iq, truth = synth.generate(200000, seed=5, frames_per_sec=3000, df_mask=synth.DF17 | synth.DF11 | synth.DF18, want_truth=True)
    assert len(truth) > 100
    for _, msg, errors in truth:
        assert errors == 0 and Oracle.crc24(msg) == 0


def test_empty_and_tiny_buffers():
    o = Oracle()
    frames, bufres = o.run_stream(np.zeros(0, dtype=np.uint8), 65536)
    assert len(frames) == 0 and len(bufres) == 0
    iq = synth.config5_stream(2, 3000)
    frames, bufres = Oracle().run_stream(iq, 1000)           # buffers shorter than the 326-sample halo are legal
    assert len(bufres) == 3


# What the reference's own demodulator, converters, CRC tables and ICAO filter returned for the inputs of the tests below
# (tests/golden/make_reference_runs.py runs them where the reference is built as a library, oracle/_ref); the tests hold the
# oracle to those outputs on machines without the reference tree.
FRAME_FIELDS = ("timestamp", "j", "crc", "addr", "score", "buffer_seq", "signal_len", "phase", "msgtype", "msgbits", "correctedbits",
                "fix_bit", "msg")
LIVE_GEN = {"cfg2": synth.config2_stream, "cfg5": synth.config5_stream, "mixed": synth.mixed_stream}
LIVE_INPUTS = [("cfg2", 1), ("cfg5", 2), ("mixed", 3), ("mixed", 4)]
LIVE_BUFS = [65536, 131072]
# what each demodulate2400() call added to Modes.stats_current (the per-buffer counters of b200_buffer_result)
LIVE_BUFRES_FIELDS = ("sample_timestamp", "length", "n_frames", "buffer_seq", "icao_flipped", "demod_preambles", "demod_rejected_bad",
                      "demod_rejected_unknown_icao", "demod_accepted", "demod_preamblePhase", "demod_bestPhase")
OPTION_CASES = [(58, 0, 1), (58, 1, 0), (40, 1, 1), (120, 1, 1)]
OPTION_FIELDS = ("timestamp", "crc", "score", "msgtype", "correctedbits", "fix_bit", "msg")
MODEAC_CASES = [(1, 65536), (2, 131072), (3, 20000)]
ICAO_TTL_MS = 500           # ms of stream time instead of 60 s, same mechanism
BUSY_CASES = [(120, 3000.0), (400, 6000.0)]
BUSY_TTL_MS = 400
BUSY_FIELDS = ("timestamp", "crc", "addr", "score", "msgtype", "correctedbits", "msg")
MODEAC_SC16_CASES = [(False, 65536), (True, 20000)]


def table_probes(crc24, diagnose1) -> dict:
    """crc24 of 200 random messages and diagnose1 of every single-bit syndrome, per frame length."""
    rng = np.random.default_rng(1)
    out = {}
    for nbits in (56, 112):
        crcs = [crc24(rng.integers(0, 256, nbits // 8, dtype=np.uint8).tobytes()) for _ in range(200)]
        diag = []
        for bit in range(nbits):
            m = bytearray(nbits // 8); m[bit >> 3] = 1 << (7 - (bit & 7))
            diag.append(diagnose1(Oracle.crc24(bytes(m)), nbits))
        out[str(nbits)] = {"crc24": crcs, "diagnose1": diag}
    return out


def test_reference_tables_match():
    assert digest(Oracle.lut()) == reference_runs()["tables"]["lut"]
    assert table_probes(Oracle.crc24, Oracle.diagnose1) == reference_runs()["tables"]["probes"]


@pytest.mark.parametrize("kind,seed", LIVE_INPUTS)
@pytest.mark.parametrize("buf", LIVE_BUFS)
def test_oracle_matches_reference_live(kind, seed, buf):
    want = reference_runs()[f"live/{kind}/{seed}/{buf}"]
    o = Oracle()
    fo, bo = o.run_stream(LIVE_GEN[kind](seed, 1_500_000), buf)
    problems = diff_digests(record_digests(fo, FRAME_FIELDS), want["frames"], "frames ")
    problems += diff_digests({"signal_level": digest(fo["sigpow_sum"] / 65535.0 / 65535.0 / fo["signal_len"]),
                              "mean_level": digest(bo["sum_level"] / 65536.0 / bo["length"])}, want["levels"])
    problems += diff_digests(record_digests(bo, LIVE_BUFRES_FIELDS), want["bufres"], "bufres ")
    so = o.stats()
    problems += diff_stats(so, dict(want["stats"], sum_signal_power=so["sum_signal_power"]))   # the reference keeps this one as fp64 only
    assert not problems, "\n".join(problems)


def options_input():
    return synth.mixed_stream(9, 1_000_000)


@pytest.mark.parametrize("thr,nfix,fixdf", OPTION_CASES)
def test_oracle_matches_reference_options(thr, nfix, fixdf):
    want = reference_runs()[f"options/{thr}/{nfix}/{fixdf}"]
    fo = Oracle(thr, nfix, fixdf).run_stream(options_input(), 65536)[0]
    problems = diff_digests(record_digests(fo, OPTION_FIELDS), want["frames"])
    assert want["n_frames"] > 50 and not problems, "\n".join(problems)


@pytest.mark.parametrize("seed,buf", MODEAC_CASES)
def test_oracle_modeac_matches_reference_live(seed, buf):
    want = reference_runs()[f"modeac/{seed}/{buf}"]
    o = Oracle()
    ao = o.run_stream_ac(synth.modeac_stream(seed, 1_500_000), buf)
    assert want["n"] > 80 and len(ao) == want["n"] == want["modeac_count"] == o.stats()["demod_modeac"]
    problems = diff_digests(record_digests(ao, ("timestamp", "modeac")), want["replies"])
    assert not problems, "\n".join(problems)


def icao_ttl_input():
    return synth.generate(6_000_000, seed=77, frames_per_sec=40, df_mask=synth.DF17 | synth.AP, n_icao=2)


def test_icao_ttl_two_flips():
    """An address added by a clean DF17 lives until the second filter flip (SURVEY.md 8a, ICAO-filter timing)."""
    fo, bo = Oracle(icao_ttl_ms=ICAO_TTL_MS).run_stream(icao_ttl_input(), 131072)
    assert not diff_digests(record_digests(fo, ("timestamp", "msg", "score")), reference_runs()["icao_ttl_two_flips"])
    assert bo["icao_flipped"].sum() >= 3


def icao_filter_probes(f) -> list[str]:
    """Random add / test / expire sequences on one ICAO filter; per step, a digest of the answers to 700 tests."""
    rng = np.random.default_rng(11)
    pool = rng.choice(1 << 24, size=6000, replace=False).astype(np.uint32)
    known, out = [], []
    for step in range(40):
        for a in rng.choice(pool, size=int(rng.integers(1, 700))):
            f.icao_add(int(a)); known.append(int(a))
        probe = list(rng.choice(pool, size=300)) + known[-200:] + known[:200]
        out.append(digest(np.array([f.icao_test(int(a)) for a in probe])))
        if rng.random() < 0.35:
            f.icao_expire()
    return out


def older_generation_is_forgotten(f):
    """An address of the older generation dies with the 86th new address of the next one."""
    f.icao_add(0xABCDEF); f.icao_expire()
    for a in range(1, 86):
        f.icao_add(a)
    assert f.icao_test(0xABCDEF)
    f.icao_add(86)
    assert not f.icao_test(0xABCDEF) and f.icao_test(1) and f.icao_test(86)


def test_icao_filter_resize_forgets_the_older_generation():
    """icao_filter.c:112-130: once the active generation holds more than buckets / 3 addresses (86, 171, 342 ... from 2^8
    buckets) icaoFilterResize re-inserts the ACTIVE generation only (:66-92) - whatever the older one held is gone; and
    icaoFilterExpire halves the tables when the active generation is small (:97-99).  The oracle's sets follow the same
    state machine: random add / test / expire sequences against the reference's own icao_filter.c."""
    got, want = icao_filter_probes(Oracle()), reference_runs()["icao_filter_probes"]
    assert got == want, f"first differing step: {next(i for i, (a, b) in enumerate(zip(got, want)) if a != b)}"
    older_generation_is_forgotten(Oracle())          # the reference passes the same check (make_reference_runs.py)


def busy_input(n_icao, fps):
    return synth.generate(5_000_000, seed=5, frames_per_sec=fps, df_mask=synth.DF17 | synth.DF11 | synth.AP | synth.DF11_IID, n_icao=n_icao)


@pytest.mark.parametrize("n_icao,fps", BUSY_CASES)
def test_oracle_matches_reference_in_busy_airspace(n_icao, fps):
    """More aircraft than the reference's filter keeps without resizing (> 85, > 170, > 341): address/parity replies of
    aircraft that only the older generation knew are rejected after a resize (score -1), and the scan goes on where the
    reference's does."""
    want = reference_runs()[f"busy/{n_icao}/{fps}"]
    o = Oracle(icao_ttl_ms=BUSY_TTL_MS)
    fo, bo = o.run_stream(busy_input(n_icao, fps), 65536)
    so = o.stats()
    problems = diff_digests(record_digests(fo, BUSY_FIELDS), want["frames"])
    problems += diff_stats(so, dict(want["stats"], sum_signal_power=so["sum_signal_power"]))
    assert want["n_frames"] > 1000 and not problems, "\n".join(problems)
    assert bo["icao_flipped"].sum() >= 3


def sc16_input(q11):
    rng = np.random.default_rng(5 + q11)
    n = 70001
    lim = 2048 if q11 else 32768
    iq = rng.integers(-lim, lim, size=2 * n, dtype=np.int32)
    iq[:64] = [-lim, lim - 1] * 32                       # saturating corner: magsq clamps at 1
    iq[64:128] = 0
    iq[128:4000] = rng.integers(-lim // 50, lim // 50, size=3872)   # noise floor
    return iq.astype(np.int16)


@pytest.mark.parametrize("q11", [False, True])
def test_oracle_sc16_converters_match_reference(q11):
    """SURVEY 8(f) row 3: convert_sc16_nodc (convert.c:212-250) / convert_sc16q11_nodc (:329-367), magnitudes and the two
    sequential float accumulators, against the reference's own converters reached through init_converter."""
    want = reference_runs()[f"sc16/{int(q11)}"]
    iq = sc16_input(q11); n = iq.size // 2
    mag_o, sl_o, sp_o = Oracle.convert_sc16(iq, q11)
    assert digest(mag_o) == want["mag"] and mag_o.max() == 65535 and mag_o[32:64].min() == 0
    assert float(np.float32(sl_o) / np.float32(n)) == want["mean_level"] and float(np.float32(sp_o) / np.float32(n)) == want["mean_power"]


def _to_sc16(iq8: np.ndarray, q11: bool, seed: int) -> np.ndarray:
    """The uc8 synthetic capture as a 16-bit frontend would deliver it (plus a little sub-LSB dither)."""
    rng = np.random.default_rng(seed)
    scale = 16 if q11 else 256
    v = (iq8.astype(np.int32) - 128) * scale + rng.integers(0, scale, size=iq8.size)
    return np.clip(v, -2048 if q11 else -32768, 2047 if q11 else 32767).astype(np.int16)


def modeac_sc16_input(q11):
    return _to_sc16(synth.modeac_stream(31 + q11, 1_200_000), q11, 9)


@pytest.mark.parametrize("q11,buf", MODEAC_SC16_CASES)
def test_oracle_modeac_with_converter_levels_matches_reference(q11, buf):
    """demodulate2400AC takes its noise floor from mag_buf.mean_level / mean_power (demod_2400.c:580-581); for an sc16 frontend
    those are float-accumulated means (convert.c:243-249), not the exact integer sums: the reference's converter + the
    reference's demodulate2400AC against the oracle's converter + oracle_demodulate2400AC_levels."""
    want = reference_runs()[f"modeac_sc16/{int(q11)}/{buf}"]
    o = Oracle()
    ao = o.run_stream_ac_sc16(modeac_sc16_input(q11), buf, q11)
    assert want["n"] > 80 and len(ao) == want["n"] == o.stats()["demod_modeac"]
    # the reference harness cannot see f1_sample
    problems = diff_digests(record_digests(ao, ("timestamp", "modeac", "buffer_idx")), want["replies"])
    assert not problems, "\n".join(problems)


def dropped_input():
    return synth.mixed_stream(21, 6 * 65536)


def test_dropped_samples_raise_the_threshold_to_75():
    """demod_2400.c:334-338: while stats_15min.samples_dropped is set the reference uses max(75, preambleThreshold); the
    boundary exposes that as a threshold the caller sets between buffers."""
    want = reference_runs()["dropped_samples"]
    iq = dropped_input()
    o = Oracle(preamble_threshold=58)
    o.set_preamble_threshold(75)
    fo, _ = o.run_stream(iq, 65536)
    o58 = Oracle(preamble_threshold=58)
    o58.run_stream(iq, 65536)
    assert want["n_frames"] > 50 and not diff_digests(record_digests(fo, ("timestamp", "msg", "score")), want["frames"])
    assert want["demod_preambles"] == o.stats()["demod_preambles"] < o58.stats()["demod_preambles"]


def syndrome_ffffff_input():
    z = np.load(Path(__file__).resolve().parent / "golden" / "regress" / "syndrome_ffffff.npz")
    return z["iq"], int(z["preamble_threshold"])


def test_reference_rejects_the_all_ones_syndrome():
    """tests/golden/regress/syndrome_ffffff.npz holds a DF17 candidate with syndrome 0xFFFFFF (no single-bit error has it): the
    reference and the oracle both find nothing to accept in that window (the CUDA path once did, see tests/test_gpu_edges.py)."""
    want = reference_runs()["syndrome_ffffff"]
    iq, thr = syndrome_ffffff_input()
    o = Oracle(preamble_threshold=thr)
    fo, _ = o.run_stream(iq, 65536)
    assert want["n_frames"] == len(fo) == 0
    assert want["demod_preambles"] == o.stats()["demod_preambles"] > 10
    assert Oracle.diagnose1(0xFFFFFF, 112) < 0 and Oracle.diagnose1(0xFFFFFF, 56) < 0


def test_aggressive_error_tables_match_reference():
    """--aggressive (nfix_crc = 2, crc.c:180-378 with max_correct 2 / max_detect 4): the oracle's table — preparation, the
    demodulator path does not use it yet — holds exactly the syndromes the reference's modesChecksumDiagnose knows, with the same
    bit positions: 51 + 1275 entries for 56-bit frames, 107 + 3724 (of 5671 two-bit patterns: the rest collide with 3- or 4-bit
    patterns and are dropped) for 112-bit frames; digest over every entry, reference side taken over all 2^24 syndromes."""
    import ctypes as C
    L = Oracle.lib()
    L.oracle_crc_table2_digest.argtypes = [C.c_int, C.POINTER(C.c_uint64)]
    L.oracle_crc_diagnose2.argtypes = [C.c_uint32, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    for bits, n_expected in ((56, 51 + 1275), (112, 107 + 3724)):
        do = C.c_uint64()
        no = L.oracle_crc_table2_digest(bits, C.byref(do))
        assert [no, do.value] == reference_runs()["crc_table2_digest"][str(bits)] and no == n_expected
    b0, b1 = C.c_int(), C.c_int()
    assert L.oracle_crc_diagnose2(0x3935EA, 112, C.byref(b0), C.byref(b1)) == -2          # bit 0 is a DF bit: never corrected
    assert L.oracle_crc_diagnose2(0xFFF409, 112, C.byref(b0), C.byref(b1)) == 1 and (b0.value, b1.value) == (87, -1)
    assert L.oracle_crc_diagnose2(0xFFF409 ^ 0x000001, 112, C.byref(b0), C.byref(b1)) in (2, -2)
    assert L.oracle_crc_diagnose2(0, 112, C.byref(b0), C.byref(b1)) == 0
