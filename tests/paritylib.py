"""Shared comparison helpers for the parity tests (CUDA path vs oracle / reference)."""
from __future__ import annotations

import functools
import hashlib
import json
from pathlib import Path

import numpy as np

from readsb_b200.abi import FRAME_PARITY_FIELDS, frame_hex

REFERENCE_RUNS = Path(__file__).resolve().parent / "golden" / "reference_runs.json"

BUFRES_FIELDS = ("sample_timestamp", "sum_level", "sum_power", "sum_signal_power", "length", "n_frames",
                 "buffer_seq", "icao_flipped", "demod_preambles", "demod_rejected_bad", "demod_rejected_unknown_icao",
                 "demod_accepted", "demod_preamblePhase", "demod_bestPhase")
STATS_INT_FIELDS = ("samples_processed", "demod_preambles", "demod_rejected_bad", "demod_rejected_unknown_icao",
                    "demod_accepted", "demod_preamblePhase", "demod_bestPhase", "signal_power_count",
                    "sum_signal_power", "strong_signal_count", "buffers", "icao_flips")


def diff_frames(a: np.ndarray, b: np.ndarray, fields=FRAME_PARITY_FIELDS, limit=3) -> list[str]:
    """Bit-exact comparison of two frame lists; returns human-readable differences (empty = equal)."""
    msgs = []
    if len(a) != len(b):
        msgs.append(f"frame count {len(a)} vs {len(b)}")
    n = min(len(a), len(b))
    if n == 0:
        return msgs
    for f in fields:
        x, y = a[f][:n], b[f][:n]
        if f == "addr":   # DF18 decoding may set non-ICAO flag bits above bit 23 (out of this path's scope)
            x, y = x & 0xFFFFFF, y & 0xFFFFFF
        ne = np.nonzero((x != y).reshape(n, -1).any(axis=1))[0]
        for i in ne[:limit]:
            msgs.append(f"{f}[{i}]: {a[f][i]} vs {b[f][i]}  (ts {a['timestamp'][i]}/{b['timestamp'][i]} "
                        f"{frame_hex(a[i])}/{frame_hex(b[i])})")
        if len(ne) > limit:
            msgs.append(f"{f}: {len(ne)} mismatches in total")
    return msgs


def diff_bufres(a: np.ndarray, b: np.ndarray, fields=BUFRES_FIELDS) -> list[str]:
    msgs = []
    if len(a) != len(b):
        return [f"buffer count {len(a)} vs {len(b)}"]
    if len(a) == 0:
        return msgs
    for f in fields:
        ne = np.nonzero((a[f] != b[f]).reshape(len(a), -1).any(axis=1))[0]
        if len(ne):
            i = ne[0]
            msgs.append(f"bufres {f}[{i}]: {a[f][i]} vs {b[f][i]} ({len(ne)} differ)")
    return msgs


def diff_stats(a: dict, b: dict, fields=STATS_INT_FIELDS) -> list[str]:
    msgs = [f"stats {k}: {a[k]} vs {b[k]}" for k in fields if a[k] != b[k]]
    if a["peak_signal_power"] != b["peak_signal_power"]:
        msgs.append(f"stats peak_signal_power: {a['peak_signal_power']!r} vs {b['peak_signal_power']!r}")
    return msgs


def digest(a) -> str:
    """dtype, shape and SHA-256 of an array's bytes: how tests/golden/reference_runs.json stores a reference output too large
    to keep whole; equal digests mean bit-identical arrays."""
    a = np.ascontiguousarray(a)
    return f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()[:32]}"


def record_digests(rec: np.ndarray, fields) -> dict:
    """One digest per field of a frame / buffer-result array (addr masked as in diff_frames)."""
    return {f: digest(rec[f] & np.uint32(0xFFFFFF) if f == "addr" else rec[f]) for f in fields}


def diff_digests(got: dict, want: dict, what: str = "") -> list[str]:
    return [f"{what}{k}: {got[k]} vs reference {v}" for k, v in want.items() if got[k] != v]


@functools.cache
def reference_runs() -> dict:
    """The reference's outputs on the inputs of the reference comparisons (tests/golden/make_reference_runs.py)."""
    return json.loads(REFERENCE_RUNS.read_text())


def crc_ok(frames: np.ndarray) -> np.ndarray:
    """Mode-S parity check of corrected frames in numpy: syndrome must be 0 for DF17/18 and DF11 (mod IID)."""
    from oraclelib import Oracle
    return np.array([Oracle.crc24(bytes(f["msg"][: int(f["msgbits"]) // 8])) for f in frames], dtype=np.uint32)
