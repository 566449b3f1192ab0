"""-m gpu: BASELINE-size batches (256 receivers x 65536-sample buffers) checked through size-independent properties,
plus the committed golden fixtures (reference output) through the CUDA path."""
import json
from pathlib import Path

import numpy as np
import pytest

from oraclelib import Oracle
from paritylib import diff_bufres, diff_digests, diff_frames, diff_stats, record_digests, reference_runs
from readsb_b200 import synth
from readsb_b200.abi import FRAME_DTYPE

pytestmark = pytest.mark.gpu
GOLDEN = sorted(p for p in (Path(__file__).parent / "golden").glob("*.npz") if p.stem not in ("beast_stream", "sc16_converters"))


@pytest.mark.parametrize("path", GOLDEN, ids=[p.stem for p in GOLDEN])
def test_cuda_matches_reference_golden(cuda, path):
    from readsb_b200.demod import Demodulator
    z = np.load(path)
    meta = json.loads(bytes(z["meta"]).decode())
    d = Demodulator(n_streams=1, buf_samples=meta["buf_samples"], max_buffers_per_run=2, mode_ac=True, **meta["options"])
    frames, bufres, modeac = d.replay(np.ascontiguousarray(z["iq"]), want_modeac=True)
    assert len(modeac) == len(z["modeac"]) and np.array_equal(modeac["timestamp"], z["modeac"]["timestamp"])
    assert np.array_equal(modeac["modeac"], z["modeac"]["modeac"]) and np.array_equal(modeac["buffer_idx"], z["modeac"]["buffer_idx"])
    problems = diff_frames(frames, z["frames"], fields=("timestamp", "j", "crc", "addr", "score", "buffer_seq", "signal_len",
                                                        "phase", "msgtype", "msgbits", "correctedbits", "fix_bit", "msg"))
    assert not problems, "\n".join(problems)
    assert np.array_equal(frames["sigpow_sum"] / 65535.0 / 65535.0 / frames["signal_len"], z["signal_level"])
    assert np.array_equal(bufres["sum_level"] / 65536.0 / bufres["length"], z["mean_level"])
    assert np.array_equal(bufres["sum_power"] / 65535.0 / 65535.0 / bufres["length"], z["mean_power"])
    st = d.stats(0)
    for k, v in meta["stats"].items():
        if k not in ("sum_signal_power", "reserved_", "demod_modeac", "peak_signal_power"):
            assert st[k] == v, k
    assert st["peak_signal_power"] == meta["dstats"]["peak_signal_power"]
    d.close()


def _crc24_numpy(msgs: np.ndarray, nbytes: int) -> np.ndarray:
    """Vectorised Mode-S syndrome of N frames (bit-serial, MSB first)."""
    rem = np.zeros(len(msgs), dtype=np.uint32)
    for i in range(nbytes - 3):
        for b in range(7, -1, -1):
            bit = (msgs[:, i] >> b) & 1
            fb = ((rem >> 23) & 1) ^ bit
            rem = (rem << 1) & 0xFFFFFF
            rem ^= np.where(fb == 1, 0xFFF409, 0).astype(np.uint32)
    tail = (msgs[:, nbytes - 3].astype(np.uint32) << 16) | (msgs[:, nbytes - 2].astype(np.uint32) << 8) | msgs[:, nbytes - 1]
    return rem ^ tail


@pytest.mark.parametrize("workload", ["config3", "config5"])
def test_full_size_batch_properties(cuda, workload):
    """256 streams x 2 buffers of 65536 samples per launch (BASELINE configs[2] / configs[4] shapes)."""
    import devbuf
    from readsb_b200.demod import Demodulator
    S, BUF, NB = 256, 65536, 2
    gen = synth.config2_stream if workload == "config3" else synth.config5_stream
    host = np.empty((S, 2 * NB * BUF), dtype=np.uint8)
    # 32 distinct seeds, each receiver's stream rotated differently: cheap to generate, all receivers still differ
    base = [gen(500 + i, NB * BUF) for i in range(32)]
    for s in range(S):
        host[s] = np.roll(base[s % 32], 2 * 997 * (s // 32))
    pad = 4096
    dev = devbuf.zeros(pad + host.size + 256)
    dev[pad:pad + host.size] = devbuf.to_dev(host.reshape(-1))
    devbuf.sync()

    d = Demodulator(n_streams=S, buf_samples=BUF, max_buffers_per_run=NB)
    d.run_device(dev.data_ptr() + pad, 2 * NB * BUF, NB, BUF, continues=False, first_sample_timestamp=0)
    frames = [d.frames(s) for s in range(S)]
    bufres = [d.buffer_results(s) for s in range(S)]
    allf = np.concatenate(frames)
    assert len(allf) == d.total_frames() and len(allf) > S

    # (1) checksum of checksums: every accepted frame is a code word after correction
    long = allf[allf["msgbits"] == 112]; short = allf[allf["msgbits"] == 56]
    syn_l = _crc24_numpy(long["msg"], 14) if len(long) else np.zeros(0, np.uint32)
    syn_s = _crc24_numpy(short["msg"], 7) if len(short) else np.zeros(0, np.uint32)
    es = np.isin(long["msgtype"], (17, 18))
    assert np.all(syn_l[es] == 0)
    df11 = short["msgtype"] == 11
    assert np.all((syn_s[df11] & 0xFFFF80) == 0)
    ap_l = ~es
    assert np.array_equal(syn_l[ap_l], long["addr"][ap_l] & 0xFFFFFF)      # address/parity: syndrome is the address
    # (2) converter sums are exact: compare with a numpy gather through the same 65536-entry table
    lut = Oracle.lut().astype(np.uint64)
    idx = host.reshape(S, NB, BUF, 2)
    mags = lut[idx[..., 0].astype(np.uint32) * 256 + idx[..., 1]]
    want_level = mags.sum(axis=2); want_power = (mags * mags).sum(axis=2)
    got_level = np.stack([b["sum_level"] for b in bufres]); got_power = np.stack([b["sum_power"] for b in bufres])
    assert np.array_equal(got_level, want_level) and np.array_equal(got_power, want_power)
    # (3) order and skip-ahead: per receiver and buffer, frames ascend and never overlap the skipped region
    for s in range(S):
        f = frames[s]
        assert np.all(np.diff(f["timestamp"]) > 0)
        same = f["buffer_seq"][1:] == f["buffer_seq"][:-1]
        gap = f["j"][1:].astype(np.int64) - f["j"][:-1].astype(np.int64)
        need = np.where(f["signal_len"][:-1] == 268, 224, 112) + 1
        assert np.all(gap[same] >= need[same])
        assert np.array_equal(np.bincount(f["buffer_seq"], minlength=NB)[:NB], bufres[s]["n_frames"])
    # (4) idempotence / batching invariance: host path, one buffer per run, fresh context -> identical frames
    d2 = Demodulator(n_streams=S, buf_samples=BUF, max_buffers_per_run=1)
    out2 = [[] for _ in range(S)]
    for b in range(NB):
        d2.submit_iq_strided(0, S, host.ctypes.data + b * BUF * 2, host.strides[0], 1, BUF, b * BUF * 5)
        d2.run()
        for s in range(S):
            out2[s].append(d2.frames(s))
    for s in range(S):
        assert not diff_frames(np.concatenate(out2[s]), frames[s]), f"stream {s}"
    # (5) every receiver against the oracle: frames, per-buffer results and counters, cumulative statistics
    from concurrent.futures import ThreadPoolExecutor
    stats = [d.stats(s) for s in range(S)]

    def check(s):
        o = Oracle()
        fo, bo = o.run_stream(host[s], BUF)
        return diff_frames(frames[s], fo) + diff_bufres(bufres[s], bo) + diff_stats(stats[s], o.stats())
    with ThreadPoolExecutor(max_workers=8) as ex:
        for s, problems in enumerate(ex.map(check, range(S))):
            assert not problems, f"stream {s}: " + "\n".join(problems)
    d.close(); d2.close()


def test_dense_tile_takes_slow_path_and_stays_exact(cuda):
    """Inputs denser than the shared-memory candidate queues (a sawtooth on which half of all positions pass the
    pre-check; a saturated 40k frames/s capture at --preamble-threshold 40) must take the kernel's global-memory
    queues and stay bit-exact — never a dropped candidate."""
    from readsb_b200.demod import Demodulator
    n = 40000
    t = np.arange(n)
    ramp = (250 - (t % 120) * 2).astype(np.uint8)          # magnitude falls, then rises: ~50% of positions pass the pre-check
    saw = np.stack([ramp, np.full(n, 128, np.uint8)], axis=1).reshape(-1).copy()
    mag, _, _ = Oracle.convert(saw)
    m = mag.astype(np.int64); k = len(m) - 20
    pre = (m[1:k + 1] > m[7:k + 7]) & (m[12:k + 12] > m[14:k + 14]) & (m[12:k + 12] > m[15:k + 15])
    assert pre.mean() > 0.3                                  # > SCAN_Q1_CAP / SCAN_TILE
    storm = synth.generate(60000, seed=8, frames_per_sec=40000, df_mask=synth.DF17 | synth.DF11 | synth.AP, n_icao=4,
                           amp=(0.3, 0.9), p_bit_error=0.3)
    for iq, thr in ((saw, 58), (storm, 40)):
        o = Oracle(thr); fo, bo = o.run_stream(iq, 32768)
        d = Demodulator(n_streams=1, buf_samples=32768, max_buffers_per_run=2, preamble_threshold=thr)
        fg, bg = d.replay(iq)
        problems = diff_frames(fg, fo) + diff_bufres(bg, bo) + diff_stats(d.stats(0), o.stats())
        assert not problems, "\n".join(problems)
        d.close()


CONFIG1_REFERENCE_FIELDS = ("timestamp", "crc", "score", "msgtype", "msgbits", "correctedbits", "fix_bit", "msg")


def config1_capture():
    return synth.generate(24_000_000, seed=2024, frames_per_sec=180.0, df_mask=synth.DF17 | synth.DF11 | synth.AP, n_icao=64,
                          p_bit_error=0.1)


def test_config1_ten_second_replay(cuda):
    """BASELINE configs[0]: a 10 s, 2.4 MSPS uc8 capture replayed `--device-type ifile` style (183 full buffers of 131072
    samples + 1 partial at the default --sdr-buffer-size): CUDA path vs the oracle and vs the reference library's frames
    (stored in tests/golden/reference_runs.json)."""
    from readsb_b200.demod import Demodulator
    iq = config1_capture()
    o = Oracle(); fo, bo = o.run_stream(iq, 131072)
    assert len(bo) == 184 and len(fo) > 800
    d = Demodulator(n_streams=1, buf_samples=131072, max_buffers_per_run=8)
    fg, bg = d.replay(iq)
    problems = diff_frames(fg, fo) + diff_bufres(bg, bo) + diff_stats(d.stats(0), o.stats())
    assert not problems, "\n".join(problems)
    problems = diff_digests(record_digests(fg, CONFIG1_REFERENCE_FIELDS), reference_runs()["config1_ten_second_replay"])
    assert not problems, "\n".join(problems)
    d.close()
