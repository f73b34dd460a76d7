"""numpy twin of the simulator's message generator (dnaldpc_simulate, include/dnaldpc.h): word w of frame f's message is
the low 32 bits of rng_u64(seed, f, w, 1) (RNG stream 1, DESIGN.md §9), bits at and beyond K cleared; and the per-frame
counters of a decoded batch, as the simulator defines them."""
import numpy as np

import oraclelib as ol

MESSAGE_STREAM = 1


def messages(seed, f0, F, K):
    """uint32 [F][ceil(K/32)]: the messages of frames f0 .. f0+F-1."""
    kw = (K + 31) // 32
    f = np.arange(f0, f0 + F, dtype=np.uint64)[:, None]
    w = np.arange(kw, dtype=np.uint64)[None, :]
    words = (ol.rng_u64(seed, f, w, MESSAGE_STREAM) & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    if K % 32:
        words[:, kw - 1] &= np.uint32((1 << (K % 32)) - 1)
    return words


def popcount_rows(words):
    """Set bits per row of a uint32 [F][W] array."""
    words = np.ascontiguousarray(words, dtype=np.uint32)
    return np.unpackbits(words.view(np.uint8), axis=1).sum(axis=1, dtype=np.int64)


def frame_counters(sent, decoded, ok, iters, raw_hard, info_cols, N):
    """Per-frame records of a batch. sent / decoded / raw_hard: uint32 [F][ceil(N/32)] (bits beyond N ignored), ok / iters
    [F]. Returns a dict of int64 arrays [F] named like the fields of dnaldpc_sim_result."""
    wpf = (N + 31) // 32
    last = np.uint32(0xFFFFFFFF if N % 32 == 0 else (1 << (N % 32)) - 1)
    info = np.zeros(wpf * 32, np.uint8)
    info[np.asarray(info_cols)] = 1
    info_mask = np.packbits(info, bitorder="little").view(np.uint32)
    x = np.bitwise_xor(sent, decoded)
    x[:, -1] &= last
    r = np.bitwise_xor(sent, raw_hard)
    r[:, -1] &= last
    bit = popcount_rows(x)
    msg = popcount_rows(x & info_mask[None, :])
    raw = popcount_rows(r)
    ok = np.asarray(ok) != 0
    return dict(iterations=np.asarray(iters, np.int64), frame_errors=(bit > 0).astype(np.int64), bit_errors=bit,
                msg_frame_errors=(msg > 0).astype(np.int64), msg_bit_errors=msg, detected=(~ok).astype(np.int64),
                undetected=(ok & (bit > 0)).astype(np.int64), raw_frame_errors=(raw > 0).astype(np.int64), raw_bit_errors=raw)


def totals(per_frame, n):
    """dnaldpc_sim_result over the first n frames."""
    out = {k: int(v[:n].sum()) for k, v in per_frame.items()}
    out["frames"] = int(n)
    return out
