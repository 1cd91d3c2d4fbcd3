"""Kernel arithmetic on the CPU: solo_b200/csrc/*.cuh compiled by g++ (tests/hostsim) against the golden fixtures and
against the unmodified reference's outputs on inputs the fixtures do not cover (digests in
tests/golden/reference_digests.npz).

The headers are written once as __host__ __device__ code, so what passes here is the same source nvcc compiles into
libsolo_b200.so (the warp-per-stream quantiser sb_nsq_warp.cuh is device-only; its scalar model sb_nsq.cuh runs here and
the `-m gpu` suite pins the device version).  Bar: payloads and length fields byte-identical to the FIX build, PCM
identical to the FLP build (north star allows +-1 LSB)."""
import hashlib
import struct

import numpy as np
import pytest

from tests.util import (RowDigests, assert_matches_reference, enc_row, load_clip, load_golden, loss_flags, speech_replay,
                        synth_inputs, trim_payload)

PCM_TOL = 0


@pytest.fixture(scope="module")
def sim():
    from tests.hostsim import sim as s
    s.lib()
    return s


def bitfile(pk):
    return b"".join(struct.pack("<hh", *nb) + (b if nb[0] else b"") for b, nb, n in pk)


def encode(mod_enc, pcm, **kw):
    e = mod_enc(**kw)
    pk = [e.encode(pcm[i * 640:(i + 1) * 640]) for i in range(len(pcm) // 640)]
    e.close()
    return pk


def test_encoder_matches_golden_bitstream(sim):
    g = load_golden()
    pk = encode(sim.SimEncoder, load_clip(), rate=13600)
    assert hashlib.md5(bitfile(pk)).hexdigest() == str(g["fix_bitfile_md5"])
    for i, (b, nb, n) in enumerate(pk):
        assert nb == tuple(g["fix_nbytes"][i]) and n == nb[0]
        assert b == bytes(g["fix_bits"][i, :n])


@pytest.mark.parametrize("mode", [4, 2, 3, "loss50"])
def test_decoder_matches_golden_pcm(sim, mode):
    g = load_golden()
    n = g["fix_nbytes"].shape[0]
    flags = list(g["loss50_flags"]) if mode == "loss50" else [mode] * n
    key = "flp_pcm_loss50" if mode == "loss50" else "flp_pcm_mode%d" % mode
    d = sim.SimDecoder()
    out = []
    for i in range(n):
        nb = tuple(int(v) for v in g["fix_nbytes"][i])
        pb, pnb = trim_payload(bytes(g["fix_bits"][i, :nb[0]]), nb, int(flags[i]))
        x, r = d.decode(pb, pnb, int(flags[i]))
        assert r == 0
        out.append(x)
    d.close()
    pcm = np.concatenate(out)
    assert np.abs(pcm.astype(np.int32) - g[key].astype(np.int32)).max() <= PCM_TOL


def test_encoder_matches_synthetic_hashes(sim):
    """Other rates, scaled / clipped speech, noise, silence, DC, full-scale square, sine, DTX, MD index flag."""
    g = load_golden()
    for name, x, kw in synth_inputs(load_clip()):
        kw = dict(kw)
        if "mdi" in kw:
            kw["use_md_index"] = kw.pop("mdi")
        assert hashlib.md5(bitfile(encode(sim.SimEncoder, x, **kw))).hexdigest() == str(g["synth_" + name]), name


def test_empty_and_error_inputs(sim):
    """Reference behaviour at the edges of the decode contract (AGR_BWE_SDK_API.c:268-270, decode_frame.c:303-324):
    nBytes[0] <= 0 is an error (-1) whatever the flag; a lost packet (flag 1) never reads its payload, and concealment
    from the initial state is silence."""
    d = sim.SimDecoder()
    for flag in (1, 2, 3, 4):
        x, r = d.decode(b"", (0, 0), flag)
        assert r == -1
    x, r = d.decode(bytes(16), (16, 8), 1)
    assert r == 0 and not x.any()
    d.close()


def run_speech_replay_streams(Enc, Dec):
    """SURVEY.md 8(d) batch (i), 12 streams x 30 packets, each stream with its own loss pattern (seed 1 + s, 50 %).
    Enc / Dec: encoder and decoder classes with the call shapes of tests/hostsim/sim.py (the reference's too)."""
    S, P = 12, 30
    x = speech_replay(load_clip(), S, P)
    enc, pcm = RowDigests(P, S), RowDigests(P, S)
    for s in range(S):
        e, d = Enc(rate=13600), Dec()
        flags = loss_flags(P, 50, seed=1 + s)
        for p in range(P):
            b, nb, n = e.encode(x[p, s])
            enc.add(p, s, enc_row(b[:max(n, 0)], nb) + struct.pack("<i", n))
            pb, pnb = trim_payload(b, nb, flags[p])
            y, r = d.decode(pb, pnb, flags[p])
            assert r == 0, (s, p)
            pcm.add(p, s, y.tobytes())
        e.close(); d.close()
    return dict(enc=enc, pcm=pcm)


def test_speech_replay_streams_match_reference(sim):
    """Encoder bytes vs FIX, decoder PCM vs FLP fed the same payloads and flags."""
    assert_matches_reference("hostsim_speech_replay", **run_speech_replay_streams(sim.SimEncoder, sim.SimDecoder))


def run_random_rates_and_signals(Enc, Dec):
    """Seeded sweep over target rates and signal classes that the fixtures do not hold: 5 configurations x 4 signals
    (one digest column each) x 25 packets."""
    rng = np.random.Generator(np.random.PCG64(99))
    clip = load_clip()
    t = np.arange(640 * 25)
    enc, pcm = RowDigests(25, 20), RowDigests(25, 20)
    col = 0
    for rate, mdi, dtx in ((8000, 0, 0), (11000, 1, 0), (13600, 0, 1), (20000, 0, 0), (40000, 1, 1)):
        off = int(rng.integers(0, len(clip) - 640 * 25))
        sigs = [clip[off:off + 640 * 25],
                (clip[off:off + 640 * 25].astype(np.int32) * 3 // 2).clip(-32768, 32767).astype(np.int16),
                (6000 * np.sin(2 * np.pi * (80 + 3e-3 * t) * t / 16000)).astype(np.int16),
                np.clip(rng.normal(0, 500, 640 * 25), -32768, 32767).astype(np.int16)]
        for x in sigs:
            e, d = Enc(rate=rate, dtx=dtx, use_md_index=mdi), Dec(use_md_index=mdi)
            for p in range(25):
                b, nb, n = e.encode(x[p * 640:(p + 1) * 640])
                enc.add(p, col, enc_row(b[:max(n, 0)], nb) + struct.pack("<i", n))
                if nb[0] <= 0:        # DTX: nothing was sent, the receiver conceals
                    y, _ = d.decode(bytes(16), (16, 8), 1)
                else:
                    y, _ = d.decode(b[:n], nb, 4)
                pcm.add(p, col, y.tobytes())
            e.close(); d.close()
            col += 1
    return dict(enc=enc, pcm=pcm)


def test_random_rates_and_signals_match_reference(sim):
    assert_matches_reference("hostsim_random_rates", **run_random_rates_and_signals(sim.SimEncoder, sim.SimDecoder))


SMALL_CAPS = (100, 64, 16, 9, 4)


def test_small_output_buffer_matches_reference(sim):
    """AGR_Sate_Buf_Size smaller than the packet (AGR_BWE_bits.c:166-168): the return value is min(cap, total), the length
    fields still describe the whole packet, and the first min(cap, total) bytes are the reference's."""
    clip = load_clip()
    enc = RowDigests(12, len(SMALL_CAPS))
    for i, cap in enumerate(SMALL_CAPS):
        s = sim.SimEncoder(rate=24000, cap=cap)
        for p in range(12):
            s.out[:] = 0xAA
            b, nb, n = s.encode(clip[p * 640:(p + 1) * 640])
            assert n == min(cap, nb[0]), (cap, p)
            enc.add(p, i, enc_row(b, nb) + struct.pack("<i", n))
        s.close()
    assert_matches_reference("hostsim_small_output_buffer", enc=enc)


def run_20ms_packets(Enc, Dec):
    clip = load_clip()
    enc, pcm = RowDigests(240, 3), RowDigests(240, 3)
    for i, (rate, dtx, mdi) in enumerate(((13600, 0, 0), (8000, 0, 1), (24000, 1, 0))):
        e = Enc(rate=rate, dtx=dtx, use_md_index=mdi, framesize_ms=20)
        d = Dec(use_md_index=mdi, framesize_ms=20)
        flags = loss_flags(240, 30, seed=5)
        for p in range(240):
            b, nb, n = e.encode(clip[p * 320:(p + 1) * 320])
            enc.add(p, i, enc_row(b[:max(n, 0)], nb) + struct.pack("<i", n))
            if nb[0] > 0:
                assert nb[1] >= 4 and n == nb[0], (rate, p)
                pb, pnb, f = trim_payload(b, nb, flags[p]) + (flags[p],)
            else:                                   # DTX: nothing was sent
                pb, pnb, f = bytes(16), (16, 8), 1
            y, r = d.decode(pb, pnb, f)
            assert r == 0 and y.size == 320, (rate, p, f)
            pcm.add(p, i, y.tobytes())
        e.close(); d.close()
    return dict(enc=enc, pcm=pcm)


def test_20ms_packets_match_reference(sim):
    """The reference's other packet size (framesize_ms = 20: one SILK frame + one high-band frame per packet, 4 high-band
    bytes, AGR_BWE_SDK_API.c:78-81,106-110): payloads vs FIX, PCM vs FLP, with loss, DTX and the MD index flag."""
    assert_matches_reference("hostsim_20ms", **run_20ms_packets(sim.SimEncoder, sim.SimDecoder))


def run_joint_mode1(Enc, Dec):
    clip = load_clip()
    enc, pcm = RowDigests(120, 3), RowDigests(120, 3)
    for i, (rate, dtx, mdi) in enumerate(((13600, 0, 0), (8000, 0, 1), (24000, 1, 0))):
        e = Enc(rate=rate, dtx=dtx, use_md_index=mdi, joint_hb=1)
        d = Dec(use_md_index=mdi, joint_hb=1)
        flags = loss_flags(120, 30, seed=9)
        for p in range(120):
            b, nb, n = e.encode(clip[p * 640:(p + 1) * 640])
            enc.add(p, i, enc_row(b[:max(n, 0)], nb) + struct.pack("<i", n))
            if nb[0] > 0:
                pb, pnb, f = trim_payload(b, nb, flags[p]) + (flags[p],)
            else:
                pb, pnb, f = bytes(16), (16, 8), 1
            y, r = d.decode(pb, pnb, f)
            assert r == 0, (rate, p, f)
            pcm.add(p, i, y.tobytes())
        e.close(); d.close()
    return dict(enc=enc, pcm=pcm)


def test_joint_mode1_matches_reference(sim):
    """joint_enable = 1, joint_mode = 1 (AGR_BWE_SDK_API.c:63-66): one 40 ms high-band frame (4 bytes, 80-sample
    sub-frames) per packet, core rate = target - 800."""
    assert_matches_reference("hostsim_joint_mode1", **run_joint_mode1(sim.SimEncoder, sim.SimDecoder))


def run_long_run(Enc, Dec):
    clip = load_clip()
    rng = np.random.Generator(np.random.PCG64(5))
    P = 1000
    enc, pcm = RowDigests(P, 3), RowDigests(P, 3)
    for i, (rate, dtx, mdi, fs, j) in enumerate(((13600, 1, 0, 40, 0), (9000, 0, 1, 20, 0), (20000, 1, 0, 40, 1))):
        spp = 16 * fs
        e = Enc(rate=rate, dtx=dtx, use_md_index=mdi, framesize_ms=fs, joint_hb=j)
        d = Dec(use_md_index=mdi, framesize_ms=fs, joint_hb=j)
        flags = loss_flags(P, 25, seed=77)
        pos, gain = 0, 1.0
        for p in range(P):
            if p % 97 == 0:
                gain = [1.0, 0.5, 0.1, 2.5, 0.0][int(rng.integers(0, 5))]
            seg = clip[pos:pos + spp]
            pos = (pos + spp) % (len(clip) - spp)
            x = np.clip(seg.astype(np.float64) * gain, -32768, 32767).astype(np.int16)
            b, nb, n = e.encode(x)
            enc.add(p, i, enc_row(b[:max(n, 0)], nb) + struct.pack("<i", n))
            f = flags[p] if (p // 200) % 2 == 0 else (1 if rng.random() < 0.6 else 4)
            if nb[0] <= 0:
                pb, pnb, f = bytes(16), (16, 8), 1
            else:
                pb, pnb = trim_payload(b, nb, f)
            y, r = d.decode(pb, pnb, f)
            assert r == 0, (rate, p, f)
            pcm.add(p, i, y.tobytes())
        e.close(); d.close()
    return dict(enc=enc, pcm=pcm)


def test_long_run_with_level_changes_dtx_and_loss_bursts(sim):
    """Soak: 1 000 packets per configuration (40 ms, 20 ms, joint mode 1) of programme material that changes level, goes
    silent (DTX on) and suffers loss bursts -- counters, hysteresis, CNG and concealment state must track the reference
    packet after packet."""
    assert_matches_reference("hostsim_long_run", **run_long_run(sim.SimEncoder, sim.SimDecoder))


def test_cooperative_analysis_under_32_lane_emulation(sim):
    """The warp-per-stream analysis code of the device kernels (sb_coop.cuh: lanes over outputs, wavefronts, shuffles, ballots)
    executed by 32 fibres per stream (sb_par.cuh SB_EMU: round-robin between barriers, divergent collectives abort) reproduces
    the golden bitstream of the whole clip, and equals the scalar model on the other input classes, packet modes and rates."""
    g = load_golden()
    clip = load_clip()
    e = sim.SimEncoder(rate=13600, emu=True)
    assert e.L.hs_is_emu() == 1
    for p in range(len(clip) // 640):
        b, nb, n = e.encode(clip[p * 640:(p + 1) * 640])
        assert nb == tuple(g["fix_nbytes"][p]) and b[:n] == bytes(g["fix_bits"][p, :n]), p
    e.close()
    cases = [(name, x, dict(kw)) for name, x, kw in synth_inputs(clip)]
    cases += [("20ms", clip[:320 * 80], dict(framesize_ms=20)), ("joint1", clip[:640 * 60], dict(joint_hb=1)),
              ("20ms_rate8000", clip[:320 * 60], dict(framesize_ms=20, rate=8000))]
    for name, x, kw in cases:
        if "mdi" in kw:
            kw["use_md_index"] = kw.pop("mdi")
        e0, e1 = sim.SimEncoder(emu=False, **kw), sim.SimEncoder(emu=True, **kw)
        spp = e0.samples
        for p in range(min(len(x) // spp, 50)):
            assert e0.encode(x[p * spp:(p + 1) * spp]) == e1.encode(x[p * spp:(p + 1) * spp]), (name, p)
        e0.close(); e1.close()


def test_quantiser_kernel_code_under_32_lane_emulation(sim):
    """The device code of the quantiser kernel (sb_nsq_warp.cuh: lane = (quantiser, decision state), shuffles for the joint
    rate-distortion decisions, 64-bit path words, history tables, output ring and random-generator history outside the
    shared-memory block) compiled for the host and run on 32 emulated lanes per stream behind the emulated analysis stage:
    golden bitstream on the first 48 packets of the clip (both signal types, rewhitening, decision-window resets), and the
    scalar model on the other input classes / modes / rates; then the kernel's two-streams-per-warp packing: the second lane group
    shadowing the first one's stream, and two different streams (speech beside noise / silence / a sine / other speech)."""
    g = load_golden()
    clip = load_clip()
    e = sim.SimEncoder(rate=13600, emu=True, emu_nsq=True)
    for p in range(48):
        b, nb, n = e.encode(clip[p * 640:(p + 1) * 640])
        assert nb == tuple(g["fix_nbytes"][p]) and b[:n] == bytes(g["fix_bits"][p, :n]), p
    e.close()
    cases = [(name, x, dict(kw)) for name, x, kw in synth_inputs(clip) if name not in ("rate15600", "rate_default", "shift2", "dtx")]
    cases += [("20ms", clip[320 * 30:], dict(framesize_ms=20)), ("joint1", clip[640 * 15:], dict(joint_hb=1))]
    for name, x, kw in cases:
        if "mdi" in kw:
            kw["use_md_index"] = kw.pop("mdi")
        e0, e1 = sim.SimEncoder(emu=False, **kw), sim.SimEncoder(emu=True, emu_nsq=True, **kw)
        spp = e0.samples
        first = 12 if name.startswith("rate") or name in ("clip4x", "mdi") else 0     # start inside the speech
        for p in range(first, first + 6):
            assert e0.encode(x[p * spp:(p + 1) * spp]) == e1.encode(x[p * spp:(p + 1) * spp]), (name, p)
        e0.close(); e1.close()
    # the kernel's packing -- two 16-lane groups per warp, group masks, segmented shuffles, ballot halves.  (a) the second
    # group shadows the first one's stream, which is what the kernel does with the last stream of an odd batch;
    e = sim.SimEncoder(rate=13600, emu="gw16", emu_nsq=True)
    for p in range(16):
        b, nb, n = e.encode(clip[p * 640:(p + 1) * 640])
        assert nb == tuple(g["fix_nbytes"][p]) and b[:n] == bytes(g["fix_bits"][p, :n]), ("gw16", p)
    e.close()
    # (b) two DIFFERENT streams in one warp: the groups go their own ways between the full-warp sample loops (rewhitening of
    # voiced frames, decision-window flushes, rescaling), every collective names its lanes, and the emulation's barriers wait
    # for exactly those
    rng = np.random.Generator(np.random.PCG64(3))
    t = np.arange(640 * 12)
    others = {"noise3000": np.clip(rng.normal(0, 3000, 640 * 12), -32768, 32767).astype(np.int16),
              "zeros": np.zeros(640 * 12, np.int16),
              "sine200": (8000 * np.sin(2 * np.pi * 200 * t / 16000)).astype(np.int16),
              "speech_later": clip[640 * 60:640 * 72]}
    for name, xo in others.items():
        ea, eb = sim.SimEncoder(emu="gw16"), sim.SimEncoder(emu="gw16")
        ra, rb = sim.SimEncoder(emu=False), sim.SimEncoder(emu=False)
        for p in range(8):
            xa, xb = clip[(p + 14) * 640:(p + 15) * 640], xo[p * 640:(p + 1) * 640]
            a, b = sim.encode_pair(ea, eb, xa, xb)
            assert a == ra.encode(xa) and b == rb.encode(xb), (name, p)
        for o in (ea, eb, ra, rb):
            o.close()


def test_fast_reciprocal_division_is_exact():
    """div_q29 (sb_common.cuh): (INT32_MAX >> 2) / d through a float reciprocal + one correction equals C integer division for
    every divisor the approximate-division helpers can produce (16384 <= |d| <= 32768) -- same float operations as the device."""
    N = np.int64(0x7FFFFFFF >> 2)
    d = np.concatenate([np.arange(-32768, -16383), np.arange(16384, 32768)]).astype(np.int64)
    r = (np.float32(1.0) / d.astype(np.float32)).astype(np.float32)
    q = (np.float32(N) * r).astype(np.float32).astype(np.int64)      # truncation toward zero
    rem = N - q * d
    pos = d > 0
    q = np.where(pos & (rem < 0), q - 1, np.where(pos & (rem >= d), q + 1, q))
    q = np.where(~pos & (rem < 0), q + 1, np.where(~pos & (rem >= -d), q - 1, q))
    want = np.trunc(N.astype(np.float64) / d.astype(np.float64)).astype(np.int64)
    assert np.array_equal(q, want)
