"""Shared helpers of the test-suite (input synthesis, the reference driver's loss process, payload trimming, digests of
the reference's outputs)."""
import hashlib
import os
import struct

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
REFERENCE_DIGESTS = os.path.join(GOLDEN, "reference_digests.npz")


def load_clip():
    return np.load(os.path.join(GOLDEN, "speech_clip.npz"))["pcm"]


def load_golden():
    return np.load(os.path.join(GOLDEN, "golden.npz"))


def enc_row(payload, nb):
    """What an encoder call hands back for one stream: both length fields and the payload bytes."""
    return struct.pack("<hh", int(nb[0]), int(nb[1])) + bytes(payload)


class RowDigests:
    """md5 of every (packet, stream) row of a run, folded into one digest per packet and one per stream.

    tests/golden/make_reference_digests.py ran the unmodified reference on the inputs of the parity tests and stored the
    folded digests in reference_digests.npz, so the tests compare byte for byte with the reference without needing it,
    and a mismatch still names the packets and streams that differ."""

    def __init__(self, n_packets, n_streams):
        self.rows = np.zeros((n_packets, n_streams, 16), np.uint8)

    def add(self, p, s, row):
        self.rows[p, s] = np.frombuffer(hashlib.md5(row).digest(), np.uint8)

    def folded(self):
        fold = lambda rows: np.frombuffer(hashlib.md5(np.ascontiguousarray(rows).tobytes()).digest(), np.uint8)
        return (np.stack([fold(self.rows[p]) for p in range(self.rows.shape[0])]),
                np.stack([fold(self.rows[:, s]) for s in range(self.rows.shape[1])]))


def assert_matches_reference(case, **digests):
    """digests: kind ('enc', 'pcm', ...) -> RowDigests of this run; compared with the reference's digests of `case`."""
    g = np.load(REFERENCE_DIGESTS)
    for kind, d in sorted(digests.items()):
        packets, streams = d.folded()
        key = "%s:%s" % (case, kind)
        want_p, want_s = g[key + ":packets"], g[key + ":streams"]
        assert packets.shape == want_p.shape and streams.shape == want_s.shape, (key, packets.shape, want_p.shape)
        bad_p = np.nonzero((packets != want_p).any(axis=1))[0]
        bad_s = np.nonzero((streams != want_s).any(axis=1))[0]
        assert len(bad_p) == 0 and len(bad_s) == 0, "%s differs from the reference in packets %s and streams %s" % (
            key, bad_p[:20].tolist(), bad_s[:20].tolist())


def _lcg(s):
    return (907633515 + s * 196314165) & 0xFFFFFFFF


def _s32(x):
    return x - (1 << 32) if x >= (1 << 31) else x


def loss_flags(n_packets, loss_perc, seed=1):
    """lostflag sequence of the reference decoder driver (JC1_SDK_SRC_FLP/test/dec_main.c:24,227-307):
    per packet two LCG draws (one per description), float32 compare against loss/100; both kept -> 4,
    MD2 lost -> 2, MD1 lost -> 3, both lost -> 1."""
    rs = seed
    out = []
    thr = np.float32(loss_perc) / np.float32(100.0)
    for _ in range(n_packets):
        lost = []
        for _j in range(2):
            rs = _lcg(rs)
            v = np.float32(np.float32((_s32(rs) >> 16) + (1 << 15)) / np.float32(65535.0))
            lost.append(0 if v >= thr else 1)
        out.append({(0, 0): 4, (0, 1): 2, (1, 0): 3, (1, 1): 1}[tuple(lost)])
    return out


def trim_payload(b, nb, flag):
    """What the caller hands to AGR_Sate_Decoder_Decode for a given lostflag (dec_main.c:245-307)."""
    n0, n1 = int(nb[0]), int(nb[1])
    if flag == 2:
        return b[:n0 - n1], (n0 - n1, 0)
    if flag == 3:
        return b[n0 - n1:n0], (n1, 0)
    return b[:n0], (n0, n1)


def speech_replay(clip, n_streams, n_packets, first_packet=0):
    """SURVEY.md 8(d) synthetic batch (i): stream s reads the clip circularly from sample offset
    (s*7919*640) mod len(clip), scaled by 2^-(s mod 4).  Returns int16 [n_packets, n_streams, 640]."""
    n = len(clip)
    s = np.arange(n_streams, dtype=np.int64)
    off = (s * 7919 * 640) % n
    out = np.empty((n_packets, n_streams, 640), np.int16)
    idx = np.arange(640, dtype=np.int64)
    sh = (s & 3).astype(np.int16)
    for p in range(n_packets):
        ii = (off[:, None] + (first_packet + p) * 640 + idx[None, :]) % n
        out[p] = clip[ii] >> sh[:, None]
    return out


def synth_inputs(clip):
    """(name, int16 signal, encoder kwargs): parity cases beyond the plain clip (SURVEY.md 8(d) ii/iii + rates)."""
    rng = np.random.Generator(np.random.PCG64(1234))
    t = np.arange(640 * 60)
    cases = [
        ("rate6000", clip, dict(rate=6000)),
        ("rate15600", clip, dict(rate=15600)),
        ("rate24000", clip, dict(rate=24000)),
        ("rate100000", clip[:640 * 60], dict(rate=100000)),
        ("rate_default", clip[:640 * 60], dict(rate=0)),
        ("shift2", clip >> 2, {}),
        ("clip4x", np.clip(clip.astype(np.int32) * 4, -32768, 32767).astype(np.int16), {}),
        ("noise2000", np.clip(rng.normal(0, 2000, 640 * 80), -32768, 32767).astype(np.int16), {}),
        ("noise20000", np.clip(rng.normal(0, 20000, 640 * 40), -32768, 32767).astype(np.int16), {}),
        ("zeros", np.zeros(640 * 40, np.int16), {}),
        ("dc1000", np.full(640 * 40, 1000, np.int16), {}),
        ("square100", np.where((t // 80) % 2 == 0, 32767, -32767).astype(np.int16), {}),
        ("sine200", (8000 * np.sin(2 * np.pi * 200 * t / 16000)).astype(np.int16), {}),
        ("dtx", np.concatenate([clip[:640 * 60], np.zeros(640 * 60, np.int16), clip[:640 * 40]]), dict(dtx=1)),
        ("mdi", clip[:640 * 80], dict(mdi=1)),
    ]
    return cases
