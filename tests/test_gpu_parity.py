"""On-device parity: the sm_100a kernels, called through the C ABI of libsolo_b200.so, against
 (a) the committed golden vectors and (b) the unmodified reference's outputs on the same inputs (digests in
 tests/golden/reference_digests.npz).
Bar: encoder payloads + length fields byte-identical to the reference FIX build; decoded PCM identical (tolerance
stated by the north star is +-1 LSB; we require 0) to the reference FLP build."""
import hashlib
import struct

import numpy as np
import pytest

from tests.util import (RowDigests, assert_matches_reference, enc_row, load_clip, load_golden, loss_flags, speech_replay,
                        synth_inputs, trim_payload)

pytestmark = pytest.mark.gpu

PCM_TOL = 0  # LSB; north star allows 1


@pytest.fixture(scope="module")
def sb():
    import solo_b200
    solo_b200.lib()
    return solo_b200


def bitfile(pk):
    return b"".join(struct.pack("<hh", *nb) + (b if nb[0] else b"") for b, nb, n in pk)


def encode_single(sb, pcm, **kw):
    e = sb.SoloEncoder(**kw)
    pk = [e.encode(pcm[i * 640:(i + 1) * 640]) for i in range(len(pcm) // 640)]
    e.close()
    return pk


def test_single_stream_golden_bitstream(sb):
    """Config 1/2 plumbing: the six-function ABI reproduces the reference FIX bit file of the shipped clip."""
    g = load_golden()
    pk = encode_single(sb, load_clip(), rate=13600)
    assert hashlib.md5(bitfile(pk)).hexdigest() == str(g["fix_bitfile_md5"])
    for i, (b, nb, n) in enumerate(pk):
        assert n == len(b) == g["fix_nbytes"][i, 0]
        assert nb == tuple(g["fix_nbytes"][i])
        assert b == bytes(g["fix_bits"][i, :n])


@pytest.mark.parametrize("mode", [4, 2, 3, "loss50"])
def test_single_stream_golden_decode(sb, mode):
    g = load_golden()
    n = g["fix_nbytes"].shape[0]
    flags = list(g["loss50_flags"]) if mode == "loss50" else [mode] * n
    d = sb.SoloDecoder()
    out = []
    for i in range(n):
        b = bytes(g["fix_bits"][i, :g["fix_nbytes"][i, 0]])
        pb, pnb = trim_payload(b, g["fix_nbytes"][i], flags[i])
        x, r = d.decode(pb, pnb, flags[i])
        assert r == 0 and d.last_nsamples == 640
        out.append(x)
    d.close()
    want = g["flp_pcm_loss50" if mode == "loss50" else "flp_pcm_mode%d" % mode]
    got = np.concatenate(out)
    assert np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= PCM_TOL


def test_synthetic_inputs_golden(sb):
    g = load_golden()
    for name, x, kw in synth_inputs(load_clip()):
        kw2 = dict(kw)
        if "mdi" in kw2:
            kw2["use_md_index"] = kw2.pop("mdi")
        pk = encode_single(sb, x, **kw2)
        assert hashlib.md5(bitfile(pk)).hexdigest() == str(g["synth_" + name]), name


BATCH_ENCODE = dict(N=256, T=12, cap=256)


def test_batch_encode_matches_reference(sb):
    """Config 2 (reduced for test time): N streams x T packets of the speech-replay batch, every payload byte and both
    length fields equal to libjc1_fix.so run per stream."""
    N, T, cap = BATCH_ENCODE["N"], BATCH_ENCODE["T"], BATCH_ENCODE["cap"]
    x = speech_replay(load_clip(), N, T)
    eb = sb.EncoderBatch(N, rate=13600)
    enc = RowDigests(T, N)
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        for s in range(N):
            enc.add(p, s, enc_row(bits[s, :nb[s, 0]], nb[s]))
    eb.close()
    assert_matches_reference("parity_batch_encode", enc=enc)


def roundtrip_flags(N, T):
    flags = np.array([loss_flags(T, 50, seed=1 + s) for s in range(N)], np.int32)  # [N, T]
    flags[:N // 4] = 4  # a quarter of the streams loss-free
    return flags


BATCH_ROUNDTRIP = dict(N=96, T=14, cap=256)


def test_batch_roundtrip_with_loss_matches_reference(sb):
    """Config 3 + 5 (reduced): encode -> decode with a per-stream loss process (seed 1 + stream id, 50 %), PCM against
    libjc1_flp.so driven with identical flags."""
    N, T, cap = BATCH_ROUNDTRIP["N"], BATCH_ROUNDTRIP["T"], BATCH_ROUNDTRIP["cap"]
    x = speech_replay(load_clip(), N, T)
    eb = sb.EncoderBatch(N)
    db = sb.DecoderBatch(N)
    flags = roundtrip_flags(N, T)
    pcm_d = RowDigests(T, N)
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        dbits = np.zeros((N, cap), np.uint8)
        dnb = np.zeros((N, 2), np.int16)
        for s in range(N):
            b = bytes(bits[s, :nb[s, 0]])
            pb, pnb = trim_payload(b, nb[s], flags[s, p])
            dbits[s, :len(pb)] = np.frombuffer(pb, np.uint8)
            dnb[s] = pnb
        pcm, ret = db.decode(dbits, dnb, flags[:, p].copy())
        assert (ret == 0).all()
        for s in range(N):
            pcm_d.add(p, s, pcm[s].tobytes())
    eb.close()
    db.close()
    assert_matches_reference("parity_batch_roundtrip", pcm=pcm_d)


def test_full_size_properties(sb):
    """BASELINE config 3 size (65 536 streams): size-independent properties instead of a CPU replay --
    (1) streams fed identical input produce identical payloads (replicas), (2) decode(encode(x)) of replicas is identical,
    (3) a sampled subset matches the golden single-stream payload for packet 0 of the clip."""
    N, cap = 65536, 128
    clip = load_clip()
    g = load_golden()
    x = np.broadcast_to(clip[:640], (N, 640)).copy()
    eb = sb.EncoderBatch(N)
    db = sb.DecoderBatch(N)
    bits, nb = eb.encode(x, cap=cap)
    assert (nb == nb[0]).all()
    assert (bits == bits[0]).all()
    n0 = int(g["fix_nbytes"][0, 0])
    assert tuple(nb[0]) == tuple(g["fix_nbytes"][0])
    assert bytes(bits[0, :n0]) == bytes(g["fix_bits"][0, :n0])
    pcm, ret = db.decode(bits, nb, np.full(N, 4, np.int32))
    assert (ret == 0).all()
    assert (pcm == pcm[0]).all()
    assert np.abs(pcm[0].astype(np.int32) - g["flp_pcm_mode4"][:640].astype(np.int32)).max() <= PCM_TOL
    eb.close()
    db.close()


def test_abi_error_conventions(sb):
    import ctypes as C
    L = sb.lib()
    assert L.AGR_Sate_Encoder_Encode(None, None, None, 0, None) == -1
    assert L.AGR_Sate_Decoder_Decode(None, None, None, None, None, 4) == -1
    assert L.AGR_Sate_Encoder_Uninit(None) == -1
    assert L.AGR_Sate_Decoder_Uninit(None) == -1
    c = sb.api.EncCtrl(2, 0, 16000, 0, 40, 0, 0, 0)
    h = L.AGR_Sate_Encoder_Init(C.byref(c))
    assert h and c.targetRate_bps == 15600  # written back like the reference
    L.AGR_Sate_Encoder_Uninit(h)
    c = sb.api.EncCtrl(2, 13600, 16000, 0, 40, 1, 7, 0)
    assert not L.AGR_Sate_Encoder_Init(C.byref(c))  # invalid joint mode -> NULL
    d = sb.SoloDecoder()
    x, r = d.decode(b"", (0, 0), 4)
    assert r == -1  # nBytes[0] <= 0
    d.close()
