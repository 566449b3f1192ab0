"""Writes tests/golden/reference_runs.json: what the REFERENCE ITSELF (oracle/_ref/libreadsb_ref.so, built by oracle/Makefile
where the reference tree is present) returns for the inputs of the reference comparisons in tests/test_oracle.py and
tests/test_gpu_fullsize.py.  Those tests take their inputs and field lists from the same functions and constants used here,
and compare the oracle / the CUDA path with this file, so the comparison holds on machines without the reference tree.
Arrays are stored as digests (tests/paritylib.py digest: dtype, shape, SHA-256), counts and statistics as they are.

    python tests/golden/make_reference_runs.py
"""
import ctypes as C
import json
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

import test_gpu_fullsize as F  # noqa: E402
import test_oracle as T  # noqa: E402
from oraclelib import Reference, have_ref  # noqa: E402
from paritylib import REFERENCE_RUNS, digest, record_digests  # noqa: E402
from readsb_b200 import synth  # noqa: E402


def main():
    assert have_ref(), "oracle/_ref/libreadsb_ref.so is not built: make -C oracle REF=<reference tree>"
    runs = {}
    ref = Reference()
    runs["tables"] = {"lut": digest(ref.lut()), "probes": T.table_probes(ref.crc24, ref.diagnose1)}
    for kind, seed in T.LIVE_INPUTS:
        for buf in T.LIVE_BUFS:
            ref = Reference()
            fr, levels, br, ml, _ = ref.run_stream(T.LIVE_GEN[kind](seed, 1_500_000), buf)
            runs[f"live/{kind}/{seed}/{buf}"] = {
                "frames": record_digests(fr, T.FRAME_FIELDS), "levels": {"signal_level": digest(levels), "mean_level": digest(ml)},
                "bufres": record_digests(br, T.LIVE_BUFRES_FIELDS), "stats": ref.stats()[0]}
    for thr, nfix, fixdf in T.OPTION_CASES:
        fr = Reference(thr, nfix, fixdf).run_stream(T.options_input(), 65536)[0]
        runs[f"options/{thr}/{nfix}/{fixdf}"] = {"frames": record_digests(fr, T.OPTION_FIELDS), "n_frames": len(fr)}
    for seed, buf in T.MODEAC_CASES:
        ref = Reference()
        ar = ref.run_stream_ac(synth.modeac_stream(seed, 1_500_000), buf)
        runs[f"modeac/{seed}/{buf}"] = {"replies": record_digests(ar, ("timestamp", "modeac")), "n": len(ar),
                                        "modeac_count": ref.modeac_count()}
    fr = Reference(icao_ttl_ms=T.ICAO_TTL_MS).run_stream(T.icao_ttl_input(), 131072)[0]
    runs["icao_ttl_two_flips"] = record_digests(fr, ("timestamp", "msg", "score"))
    runs["icao_filter_probes"] = T.icao_filter_probes(Reference())
    T.older_generation_is_forgotten(Reference())
    for n_icao, fps in T.BUSY_CASES:
        ref = Reference(icao_ttl_ms=T.BUSY_TTL_MS)
        fr = ref.run_stream(T.busy_input(n_icao, fps), 65536)[0]
        runs[f"busy/{n_icao}/{fps}"] = {"frames": record_digests(fr, T.BUSY_FIELDS), "n_frames": len(fr), "stats": ref.stats()[0]}
    for q11 in (False, True):
        mag, ml, mp = Reference().convert_sc16(T.sc16_input(q11), q11)
        runs[f"sc16/{int(q11)}"] = {"mag": digest(mag), "mean_level": ml, "mean_power": mp}
    for q11, buf in T.MODEAC_SC16_CASES:
        ar = Reference().run_stream_ac_sc16(T.modeac_sc16_input(q11), buf, q11)
        runs[f"modeac_sc16/{int(q11)}/{buf}"] = {"replies": record_digests(ar, ("timestamp", "modeac", "buffer_idx")), "n": len(ar)}
    ref = Reference(preamble_threshold=58)
    ref.set_samples_dropped(3)
    fr = ref.run_stream(T.dropped_input(), 65536)[0]
    runs["dropped_samples"] = {"frames": record_digests(fr, ("timestamp", "msg", "score")), "n_frames": len(fr),
                               "demod_preambles": ref.stats()[0]["demod_preambles"]}
    iq, thr = T.syndrome_ffffff_input()
    ref = Reference(preamble_threshold=thr)
    fr = ref.run_stream(iq, 65536)[0]
    runs["syndrome_ffffff"] = {"n_frames": len(fr), "demod_preambles": ref.stats()[0]["demod_preambles"]}
    ref = Reference()
    ref.L.ref_crc_table2_digest.argtypes = [C.c_int, C.POINTER(C.c_uint64)]
    runs["crc_table2_digest"] = {}
    for bits in (56, 112):
        d = C.c_uint64()
        runs["crc_table2_digest"][str(bits)] = [ref.L.ref_crc_table2_digest(bits, C.byref(d)), d.value]
    fr = Reference().run_stream(F.config1_capture(), 131072)[0]
    runs["config1_ten_second_replay"] = record_digests(fr, F.CONFIG1_REFERENCE_FIELDS)
    REFERENCE_RUNS.write_text(json.dumps(runs, indent=1, sort_keys=True) + "\n")
    print(REFERENCE_RUNS, len(runs), "entries")


if __name__ == "__main__":
    main()
