#!/usr/bin/env python3
"""Regenerate reference_digests.npz from the UNMODIFIED reference (oracle/_ref, built by `make -C oracle`).

    python tests/golden/make_reference_digests.py

The parity tests that compare the product with the reference row by row (tests/test_gpu_parity.py, test_gpu_hetero.py,
test_gpu_features.py, test_hostsim_parity.py) run only the product; what the reference produced on the same inputs is
stored here as md5 digests (tests/util.RowDigests: one per packet and one per stream, each folded over the per-row
digests).  Every case drives one FIX encoder and one FLP decoder per stream the way the test drives the product: the same
inputs and loss flags from the same helpers, the receiver's trimming, concealment where DTX sent nothing.
"""
import ctypes as C
import os
import struct
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from tests import test_gpu_features as F, test_gpu_hetero as H, test_gpu_parity as P, test_hostsim_parity as S  # noqa: E402
from tests.util import REFERENCE_DIGESTS, RowDigests, enc_row, load_clip, speech_replay, trim_payload  # noqa: E402


def Enc(**kw):
    return ref.RefEncoder("fix", **kw)


def Dec(**kw):
    return ref.RefDecoder("flp", **kw)


def per_stream(x, flags=None, enc_kw=None, dec_kw=None):
    """x: [T, S, samples]; flags: [S, T] lost flags, or None for encode only.  One reference encoder (+ decoder) per
    stream, streams in parallel (ctypes releases the GIL)."""
    T, n = x.shape[:2]
    enc, pcm = RowDigests(T, n), RowDigests(T, n)

    def run(s):
        e = Enc(**(enc_kw or {}))
        d = Dec(**(dec_kw or {})) if flags is not None else None
        for p in range(T):
            b, nb, _ = e.encode(x[p, s])
            assert len(b) == max(nb[0], 0), (p, s)
            enc.add(p, s, enc_row(b, nb))
            if d is None:
                continue
            f = int(flags[s, p])
            if nb[0] <= 0:               # DTX packet: nothing is sent, the receiver conceals
                pb, pnb, f = bytes(16), (16, 8), 1
            else:
                pb, pnb = trim_payload(b, nb, f)
            y, r = d.decode(pb, pnb, f)
            assert r == 0, (p, s)
            pcm.add(p, s, y.tobytes())
        e.close()
        if d is not None:
            d.close()

    with ThreadPoolExecutor(os.cpu_count() or 4) as pool:
        list(pool.map(run, range(n)))
    return dict(enc=enc, pcm=pcm)


def sampled_speech_replay(clip, N, T, sample):
    return np.stack([speech_replay(clip, N, 1, first_packet=p)[0][sample] for p in range(T)])


def single_stream(x, **kw):
    """The drop-in encoder on consecutive packets of one signal: [len(x), 1] digests."""
    e = Enc(**kw)
    d = RowDigests(len(x), 1)
    for p, xp in enumerate(x):
        b, nb, n = e.encode(xp)
        assert n == len(b)
        d.add(p, 0, enc_row(b, nb))
    e.close()
    return d


def small_output_buffer():
    """Encoder output buffer smaller than the packet: n = min(cap, total), bytes past the cap left alone."""
    clip = load_clip()
    enc = RowDigests(12, len(S.SMALL_CAPS))
    for i, cap in enumerate(S.SMALL_CAPS):
        e = Enc(rate=24000)
        for p in range(12):
            pcm = np.ascontiguousarray(clip[p * 640:(p + 1) * 640])
            bits = (C.c_uint8 * 1024)()
            C.memset(bits, 0xAA, 1024)
            nb = (C.c_int16 * 6)()
            n = e.L.AGR_Sate_Encoder_Encode(e.h, pcm.ctypes.data, bits, cap, nb)
            assert n == min(cap, nb[0]) and bytes(bits[cap:cap + 8]) == b"\xaa" * 8
            enc.add(p, i, enc_row(bytes(bits[:n]), (nb[0], nb[1])) + struct.pack("<i", n))
        e.close()
    return dict(enc=enc)


def cases():
    clip = load_clip()
    c = P.BATCH_ENCODE
    yield "parity_batch_encode", {"enc": per_stream(speech_replay(clip, c["N"], c["T"]))["enc"]}
    c = P.BATCH_ROUNDTRIP
    yield "parity_batch_roundtrip", {"pcm": per_stream(speech_replay(clip, c["N"], c["T"]), P.roundtrip_flags(c["N"], c["T"]))["pcm"]}

    yield "hetero_classes", per_stream(H.signal_classes(clip, 256, 40), H.hetero_flags(256, 40))
    for rate in (6000, 24000, 100000):
        yield "hetero_rate%d" % rate, per_stream(H.signal_classes(clip, 64, 20, seed=rate), H.hetero_flags(64, 20),
                                                 enc_kw=dict(rate=rate))
    c = H.FULL_BATCH
    sample, flags = H.full_batch_sample_and_flags(c["N"], c["T"])
    yield "hetero_full_batch", per_stream(sampled_speech_replay(clip, c["N"], c["T"], sample), flags[sample])

    c = F.CONFIG2
    yield "features_config2", {"enc": per_stream(sampled_speech_replay(clip, c["N"], c["T"], F.config2_sample(c["N"])))["enc"]}
    c = F.CONFIG5
    sample, flags = F.config5_sample_and_flags(c["N"], c["T"])
    yield "features_config5", {"pcm": per_stream(sampled_speech_replay(clip, c["N"], c["T"], sample), flags[sample])["pcm"]}
    c = F.PACKETS_20MS
    x, flags = F.packets_20ms_inputs(clip, c["N"], c["T"])
    d = per_stream(x[:, c["sample"]], flags[c["sample"]], enc_kw=dict(framesize_ms=20), dec_kw=dict(framesize_ms=20))
    d["single"] = single_stream([clip[p * 320:(p + 1) * 320] for p in range(10)], framesize_ms=20)
    yield "features_20ms", d
    c = F.JOINT
    x = speech_replay(clip, c["N"], c["T"])
    d = per_stream(x[:, c["sample"]], F.joint_flags(c["N"], c["T"])[c["sample"]], enc_kw=dict(joint_hb=1), dec_kw=dict(joint_hb=1))
    d["single"] = single_stream([x[0, 0]], joint_hb=1)
    yield "features_joint_mode1", d

    yield "hostsim_speech_replay", S.run_speech_replay_streams(Enc, Dec)
    yield "hostsim_random_rates", S.run_random_rates_and_signals(Enc, Dec)
    yield "hostsim_small_output_buffer", small_output_buffer()
    yield "hostsim_20ms", S.run_20ms_packets(Enc, Dec)
    yield "hostsim_joint_mode1", S.run_joint_mode1(Enc, Dec)
    yield "hostsim_long_run", S.run_long_run(Enc, Dec)


def main():
    out = {}
    for case, digests in cases():
        for kind, d in digests.items():
            packets, streams = d.folded()
            out["%s:%s:packets" % (case, kind)] = packets
            out["%s:%s:streams" % (case, kind)] = streams
            print(case, kind, d.rows.shape[:2], flush=True)
    np.savez_compressed(REFERENCE_DIGESTS, **out)


if __name__ == "__main__":
    main()
