"""On-device checks of the pieces around the hot path: pipelining invariance, ragged batch sizes, stream state hand-over
(SURVEY.md 8(f) rank 3) and receiver-side loss trimming for a whole batch on the GPU (rank 1)."""
import numpy as np
import pytest

from tests.util import (RowDigests, assert_matches_reference, enc_row, load_clip, load_golden, loss_flags, speech_replay,
                        trim_payload)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import solo_b200
    solo_b200.lib()
    return solo_b200


def run_streams(sb, N, T, cap=128, flags=None, rate=13600):
    x = speech_replay(load_clip(), N, T)
    eb, db = sb.EncoderBatch(N, rate=rate), sb.DecoderBatch(N)
    out = []
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        f = np.full(N, 4, np.int32) if flags is None else flags[:, p].copy()
        pcm, ret = db.decode(bits, nb, f)
        out.append((bits.copy(), nb.copy(), pcm.copy(), ret.copy()))
    eb.close(); db.close()
    return out


def test_results_do_not_depend_on_the_number_of_pipeline_chunks(sb):
    N, T = 8192 + 64 + 5, 3          # ragged: not a multiple of the chunk granularity, odd (a shadowed lane group in the NSQ kernel)
    ref = None
    for chunks in (1, 2, 3, 8):
        sb.set_chunks(chunks)
        got = run_streams(sb, N, T)
        if ref is None:
            ref = got
            g = load_golden()            # stream 0 of the speech-replay batch reads the clip from offset 0 at gain 1
            for p in range(T):
                n0 = int(g["fix_nbytes"][p, 0])
                assert tuple(got[p][1][0]) == tuple(g["fix_nbytes"][p])
                assert bytes(got[p][0][0, :n0]) == bytes(g["fix_bits"][p, :n0])
        else:
            for a, b in zip(ref, got):
                for u, v in zip(a, b):
                    assert np.array_equal(u, v), chunks
    sb.set_chunks(0)           # back to the defaults


@pytest.mark.parametrize("N", [1, 2, 3, 63, 65])
def test_small_and_odd_batches_match_the_single_stream_result(sb, N):
    T = 4
    got = run_streams(sb, N, T, cap=256)
    x = speech_replay(load_clip(), N, T)
    for s in sorted({0, N // 2, N - 1}):
        e, d = sb.SoloEncoder(rate=13600), sb.SoloDecoder()
        for p in range(T):
            b, nb, n = e.encode(x[p, s])
            assert nb == tuple(got[p][1][s]) and b == bytes(got[p][0][s, :n])
            pcm, r = d.decode(b, nb, 4)
            assert np.array_equal(pcm, got[p][2][s])
        e.close(); d.close()


def test_state_export_import_continues_bit_exactly(sb):
    """A stream leaves one batch (slot 5 of 16) after 6 packets and joins another one (slot 2 of 4, other streams at a
    different point of their lives): its payloads and decoded PCM continue as if nothing had happened."""
    T0, T1, cap = 6, 6, 256
    x = speech_replay(load_clip(), 16, T0 + T1)
    eb, db = sb.EncoderBatch(16), sb.DecoderBatch(16)
    want = []
    for p in range(T0 + T1):
        bits, nb = eb.encode(x[p], cap=cap)
        pcm, ret = db.decode(bits, nb, np.full(16, 4, np.int32))
        want.append((bytes(bits[5, :nb[5, 0]]), tuple(nb[5]), pcm[5].copy()))
        if p == T0 - 1:
            enc_blob, dec_blob = eb.export_state(5), db.export_state(5)
    eb.close(); db.close()
    assert enc_blob.size == sb.lib().solo_b200_enc_state_bytes() and dec_blob.size == sb.lib().solo_b200_dec_state_bytes()
    eb2, db2 = sb.EncoderBatch(4), sb.DecoderBatch(4)
    y = speech_replay(load_clip(), 4, 3, first_packet=40)
    for p in range(3):                                   # the new batch already has a history
        bits, nb = eb2.encode(y[p], cap=cap)
        db2.decode(bits, nb, np.full(4, 4, np.int32))
    eb2.import_state(2, enc_blob); db2.import_state(2, dec_blob)
    for p in range(T0, T0 + T1):
        xin = speech_replay(load_clip(), 4, 1, first_packet=50 + p)[0]
        xin[2] = x[p, 5]
        bits, nb = eb2.encode(xin, cap=cap)
        pcm, ret = db2.decode(bits, nb, np.full(4, 4, np.int32))
        assert (bytes(bits[2, :nb[2, 0]]), tuple(nb[2])) == want[p][:2], p
        assert np.array_equal(pcm[2], want[p][2]), p
    with pytest.raises(sb.SoloError):
        eb2.import_state(7, enc_blob)                    # no such slot
    eb2.close(); db2.close()


def test_loss_trimming_on_device_matches_the_receiver_restatement(sb):
    import torch
    N, cap, T = 4096, 128, 3
    x = speech_replay(load_clip(), N, T)
    eb, db, db_ref = sb.EncoderBatch(N), sb.DecoderBatch(N), sb.DecoderBatch(N)
    flags = np.array([loss_flags(T, 50, seed=1 + s) for s in range(N)], np.int32)
    dev = torch.device("cuda", 0)
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        f = flags[:, p].copy()
        # host restatement of dec_main.c:245-307, row by row
        hb, hn = np.zeros((N, cap), np.uint8), np.zeros((N, 2), np.int16)
        for s in range(N):
            pb, pnb = trim_payload(bytes(bits[s, :nb[s, 0]]), nb[s], f[s])
            hb[s, :len(pb)] = np.frombuffer(pb, np.uint8)
            hn[s] = pnb
        want, wret = db_ref.decode(hb, hn, f)
        # the same on the device, feeding the device decode entry point
        d_in, d_nb, d_f = torch.from_numpy(bits).to(dev), torch.from_numpy(nb).to(dev), torch.from_numpy(f).to(dev)
        d_out, d_onb = torch.zeros_like(d_in), torch.zeros_like(d_nb)
        d_pcm, d_ret = torch.zeros((N, 640), dtype=torch.int16, device=dev), torch.zeros(N, dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        sb.apply_loss_device(d_in.data_ptr(), d_nb.data_ptr(), d_f.data_ptr(), d_out.data_ptr(), d_onb.data_ptr(), cap, N, st)
        db.decode_device(d_pcm.data_ptr(), d_out.data_ptr(), cap, d_onb.data_ptr(), d_f.data_ptr(), d_ret.data_ptr(), st)
        torch.cuda.synchronize()
        assert np.array_equal(d_onb.cpu().numpy(), hn)
        keep = f != 1
        got_rows, want_rows = d_out.cpu().numpy(), hb
        for s in np.nonzero(keep)[0][:512]:
            assert bytes(got_rows[s, :hn[s, 0]]) == bytes(want_rows[s, :hn[s, 0]])
        assert np.array_equal(d_pcm.cpu().numpy(), want) and np.array_equal(d_ret.cpu().numpy(), wret)
    eb.close(); db.close(); db_ref.close()


CONFIG2 = dict(N=4096, T=50, cap=160)


def config2_sample(N):
    return sorted(set(list(range(0, N, 67)) + [1, 2, 3, N - 1]))[:64]


def test_config2_batch_4096_streams_50_packets_sampled_against_reference(sb):
    """BASELINE config 2: 4 096 concurrent streams, encode only, 50 packets (2 s).  Every stream runs on the GPU; 64 of
    them (spread over the batch, all four input gains) must match libjc1_fix.so byte for byte."""
    N, T, cap = CONFIG2["N"], CONFIG2["T"], CONFIG2["cap"]
    clip = load_clip()
    sample = config2_sample(N)
    eb = sb.EncoderBatch(N, rate=13600)
    enc = RowDigests(T, len(sample))
    for p in range(T):
        x = speech_replay(clip, N, 1, first_packet=p)[0]
        bits, nb = eb.encode(x, cap=cap)
        assert (nb[:, 0] <= cap).all()
        for i, s in enumerate(sample):
            enc.add(p, i, enc_row(bits[s, :nb[s, 0]], nb[s]))
    eb.close()
    assert_matches_reference("features_config2", enc=enc)


CONFIG5 = dict(N=65536, T=8, cap=128)


def config5_sample_and_flags(N, T):
    """48 sampled streams with a 50 % loss process each (seed 1 + stream id, dec_main.c:229-241); arbitrary flags for
    everybody else."""
    sample = [0, 1, 2, 3] + list(range(997, N, 1489))[:44]
    flags = np.full((N, T), 4, np.int32)
    for s in sample:
        flags[s] = loss_flags(T, 50, seed=1 + s)
    rng = np.random.Generator(np.random.PCG64(7))
    other = rng.integers(1, 5, size=(N, T)).astype(np.int32)
    mask = np.ones(N, bool); mask[sample] = False
    flags[mask] = other[mask]
    return sample, flags


def test_config5_full_batch_with_per_stream_loss_sampled_against_reference(sb):
    """BASELINE configs 3 + 5 at full size: 65 536 streams, encode -> receiver-side trimming on the device -> decode with
    a 50 % loss process per stream; 48 sampled streams against libjc1_flp.so fed the same payloads and flags (PCM
    identical; the north star allows +-1 LSB)."""
    import torch
    N, T, cap = CONFIG5["N"], CONFIG5["T"], CONFIG5["cap"]
    clip = load_clip()
    sample, flags = config5_sample_and_flags(N, T)
    dev = torch.device("cuda", 0)
    eb, db = sb.EncoderBatch(N), sb.DecoderBatch(N)
    d_bits, d_nb = torch.zeros((N, cap), dtype=torch.uint8, device=dev), torch.zeros((N, 2), dtype=torch.int16, device=dev)
    d_tb, d_tnb = torch.zeros_like(d_bits), torch.zeros_like(d_nb)
    d_pcm, d_ret = torch.zeros((N, 640), dtype=torch.int16, device=dev), torch.zeros(N, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    pcm_d = RowDigests(T, len(sample))
    for p in range(T):
        x = torch.from_numpy(speech_replay(clip, N, 1, first_packet=p)[0]).to(dev)
        f = torch.from_numpy(flags[:, p].copy()).to(dev)
        eb.encode_device(x.data_ptr(), d_bits.data_ptr(), cap, d_nb.data_ptr(), st)
        sb.apply_loss_device(d_bits.data_ptr(), d_nb.data_ptr(), f.data_ptr(), d_tb.data_ptr(), d_tnb.data_ptr(), cap, N, st)
        db.decode_device(d_pcm.data_ptr(), d_tb.data_ptr(), cap, d_tnb.data_ptr(), f.data_ptr(), d_ret.data_ptr(), st)
        torch.cuda.synchronize()
        assert int((d_ret != 0).sum().item()) == 0
        idx = torch.tensor(sample, device=dev)
        pcm = d_pcm[idx].cpu().numpy()
        for i in range(len(sample)):
            pcm_d.add(p, i, pcm[i].tobytes())
    eb.close(); db.close()
    assert_matches_reference("features_config5", pcm=pcm_d)


def test_single_stream_small_output_buffer(sb):
    """Same contract through the drop-in ABI on the GPU (the caller's buffer may be smaller than the packet)."""
    g = load_golden()
    clip = load_clip()
    for cap in (64, 9):
        e = sb.SoloEncoder(rate=13600)
        for p in range(6):
            b, nb, n = e.encode(clip[p * 640:(p + 1) * 640], bufsize=cap)
            n0 = int(g["fix_nbytes"][p, 0])
            assert nb == tuple(g["fix_nbytes"][p]) and n == min(cap, n0) and b == bytes(g["fix_bits"][p, :n])
        e.close()


PACKETS_20MS = dict(N=130, T=40, cap=128, sample=[0, 1, 64, 65, 129])


def packets_20ms_inputs(clip, N, T):
    """[T, N, 320] windows of the clip at per-stream offsets, and a 40 % loss process per stream (seed 3 + stream id)."""
    off = (np.arange(N) * 7919 * 320) % (len(clip) - 320 * (T + 1))
    x = np.stack([np.stack([clip[o + p * 320:o + (p + 1) * 320] for o in off]) for p in range(T)]).astype(np.int16)
    flags = np.array([loss_flags(T, 40, seed=3 + s) for s in range(N)], np.int32)
    return x, flags


def test_20ms_packets_on_device(sb):
    """framesize_ms = 20 through the batched ABI and the drop-in ABI against the reference (FIX bytes, FLP PCM)."""
    N, T, cap, sample = PACKETS_20MS["N"], PACKETS_20MS["T"], PACKETS_20MS["cap"], PACKETS_20MS["sample"]
    clip = load_clip()
    eb, db = sb.EncoderBatch(N, rate=13600, framesize_ms=20), sb.DecoderBatch(N, framesize_ms=20)
    x, flags = packets_20ms_inputs(clip, N, T)
    enc, pcm_d = RowDigests(T, len(sample)), RowDigests(T, len(sample))
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        tb, tnb = np.zeros_like(bits), np.zeros_like(nb)
        for s in range(N):
            pb, pnb = trim_payload(bytes(bits[s, :nb[s, 0]]), nb[s], flags[s, p])
            tb[s, :len(pb)] = np.frombuffer(pb, np.uint8); tnb[s] = pnb
        pcm, ret = db.decode(tb, tnb, flags[:, p].copy())
        assert pcm.shape == (N, 320) and (ret == 0).all()
        for i, s in enumerate(sample):
            enc.add(p, i, enc_row(bits[s, :nb[s, 0]], nb[s]))
            pcm_d.add(p, i, pcm[s].tobytes())
    eb.close(); db.close()
    e, d = sb.SoloEncoder(rate=13600, framesize_ms=20), sb.SoloDecoder(framesize_ms=20)
    single = RowDigests(10, 1)
    for p in range(10):
        b, nb2, n = e.encode(clip[p * 320:(p + 1) * 320])
        assert n == len(b)
        single.add(p, 0, enc_row(b, nb2))
        y, r = d.decode(b, nb2, 4)
        assert r == 0 and y.size == 320 and d.last_nsamples == 320
    e.close(); d.close()
    assert_matches_reference("features_20ms", enc=enc, pcm=pcm_d, single=single)


def test_example_file_codec_reproduces_the_reference_cli_files(sb, tmp_path):
    """examples/jc1_file_codec.c (plain C on the six-function API + framing helpers) writes the same .bit file and the
    same decoded PCM files as the reference's enc_main / dec_main: both descriptions, 50 % loss (seed 1), MD1 only, MD2 only."""
    import hashlib
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "jc1_file_codec"
    subprocess.check_call(["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(root, "include"), os.path.join(root, "examples", "jc1_file_codec.c"),
                           "-L", os.path.join(root, "solo_b200"), "-lsolo_b200", "-Wl,-rpath," + os.path.join(root, "solo_b200"), "-o", str(exe)])
    g = load_golden()
    pcm, bit = tmp_path / "in.pcm", tmp_path / "out.bit"
    load_clip().tofile(pcm)
    subprocess.check_call([str(exe), "enc", str(pcm), str(bit), "13600"])
    assert hashlib.md5(bit.read_bytes()).hexdigest() == str(g["fix_bitfile_md5"])
    for args, key in ((["0", "0"], "flp_pcm_mode4_md5"), (["50", "0"], "flp_pcm_loss50_md5"), (["0", "1"], "flp_pcm_mode2_md5"), (["0", "2"], "flp_pcm_mode3_md5")):
        out = tmp_path / ("out_%s_%s.pcm" % tuple(args))
        subprocess.check_call([str(exe), "dec", str(bit), str(out)] + args)
        assert hashlib.md5(out.read_bytes()).hexdigest() == str(g[key]), key


JOINT = dict(N=67, T=20, cap=192, sample=[0, 1, 33, 66])


def joint_flags(N, T):
    return np.array([loss_flags(T, 40, seed=11 + s) for s in range(N)], np.int32)


def test_joint_mode1_on_device(sb):
    """The reference's joint mode 1 through the batched ABI and the drop-in ABI (unsupported modes are refused)."""
    N, T, cap, sample = JOINT["N"], JOINT["T"], JOINT["cap"], JOINT["sample"]
    x = speech_replay(load_clip(), N, T)
    eb, db = sb.EncoderBatch(N, rate=13600, joint_hb=1), sb.DecoderBatch(N, joint_hb=1)
    flags = joint_flags(N, T)
    enc, pcm_d = RowDigests(T, len(sample)), RowDigests(T, len(sample))
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        tb, tnb = np.zeros_like(bits), np.zeros_like(nb)
        for s in range(N):
            pb, pnb = trim_payload(bytes(bits[s, :nb[s, 0]]), nb[s], flags[s, p])
            tb[s, :len(pb)] = np.frombuffer(pb, np.uint8); tnb[s] = pnb
        pcm, ret = db.decode(tb, tnb, flags[:, p].copy())
        assert (ret == 0).all()
        for i, s in enumerate(sample):
            enc.add(p, i, enc_row(bits[s, :nb[s, 0]], nb[s]))
            pcm_d.add(p, i, pcm[s].tobytes())
    eb.close(); db.close()
    e = sb.SoloEncoder(rate=13600, joint_enable=1, joint_mode=1)
    b, nb2, n = e.encode(x[0, 0])
    assert n == len(b)
    single = RowDigests(1, 1)
    single.add(0, 0, enc_row(b, nb2))
    e.close()
    assert_matches_reference("features_joint_mode1", enc=enc, pcm=pcm_d, single=single)
    for bad in (dict(joint_enable=1, joint_mode=0), dict(joint_enable=1, joint_mode=2), dict(samplerate=32000), dict(framesize_ms=60)):
        with pytest.raises(sb.SoloError):
            sb.SoloEncoder(**bad)


def test_malformed_payloads_do_not_fault_and_match_the_host_build(sb):
    """Bit-flipped / random / mislabelled payloads on the device: the kernel must survive (a fault would kill the whole
    batch) and, the arithmetic being deterministic, produce exactly what the host build of the same source produces --
    including the reference's 'stale payload' continuation after a corrupted frame terminator."""
    from tests.hostsim import sim
    N, T, cap = 96, 24, 128
    rng = np.random.Generator(np.random.PCG64(21))
    x = speech_replay(load_clip(), N, T)
    eb, db = sb.EncoderBatch(N), sb.DecoderBatch(N)
    hdec = [sim.SimDecoder() for _ in range(N)]
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        bits, nb = bits.copy(), nb.copy()
        flags = rng.integers(1, 5, size=N).astype(np.int32)
        for s in range(N):
            kind = int(rng.integers(0, 6))
            n0 = int(nb[s, 0])
            if kind == 1:
                for _ in range(int(rng.integers(1, 4))):
                    bits[s, int(rng.integers(0, n0))] ^= np.uint8(1 << int(rng.integers(0, 8)))
            elif kind == 2:
                bits[s] = rng.integers(0, 256, size=cap).astype(np.uint8)
            elif kind == 3:
                nb[s] = (int(rng.integers(1, cap + 1)), 0)
                nb[s, 1] = int(rng.integers(0, int(nb[s, 0]) + 1))
            elif kind == 4:
                flags[s] = int(rng.integers(-2, 8))
        pcm, ret = db.decode(bits, nb, flags)
        for s in range(N):
            want, r = hdec[s].decode(bytes(bits[s]), (int(nb[s, 0]), int(nb[s, 1])), int(flags[s]))
            assert r == ret[s], (p, s, r, ret[s])
            if r == 0:
                assert np.array_equal(want, pcm[s]), (p, s)
    eb.close(); db.close()


def test_ten_thousand_drop_in_handles_share_the_arena(sb):
    """AGR_Sate_Encoder_Init / Decoder_Init hand out slots of the process-wide arena (segments of 256 streams): 10 000 encoder
    handles come up in well under a second each thousand, occupy 40 segments (not 10 000 batches / 50 000 CUDA streams), still
    produce the golden bitstream, and a released slot is reused."""
    import ctypes as C
    import time
    L = sb.lib()
    L.solo_b200_arena_stats.argtypes = [C.POINTER(C.c_int)]
    st = (C.c_int * 4)()
    L.solo_b200_arena_stats(st)
    seg0, used0 = st[0], st[1]
    g, clip = load_golden(), load_clip()
    t0 = time.perf_counter()
    hs = [sb.SoloEncoder(rate=13600) for _ in range(10000)]
    dt = time.perf_counter() - t0
    L.solo_b200_arena_stats(st)
    assert st[1] - used0 == 10000 and st[0] - seg0 <= 40, list(st)
    assert dt < 10.0, dt                     # ~0.1 ms per handle including the Python wrapper; round 1 needed ~1 ms and 5 CUDA streams each
    for k in (0, 255, 256, 5000, 9999):      # slots of different segments, first packets of the clip
        for p in range(3):
            b, nb, n = hs[k].encode(clip[p * 640:(p + 1) * 640])
            assert nb == tuple(g["fix_nbytes"][p]) and b[:n] == bytes(g["fix_bits"][p, :n]), (k, p)
    for h in hs[:3000]:
        h.close()
    L.solo_b200_arena_stats(st)
    assert st[1] - used0 == 7000
    again = [sb.SoloEncoder(rate=13600) for _ in range(3000)]      # reuses the released slots: no new segment
    L.solo_b200_arena_stats(st)
    assert st[1] - used0 == 10000 and st[0] - seg0 <= 40
    b, nb, n = again[0].encode(clip[:640])                          # a recycled slot starts from a fresh state
    assert nb == tuple(g["fix_nbytes"][0]) and b[:n] == bytes(g["fix_bits"][0, :n])
    for h in hs[3000:] + again:
        h.close()
    d = [sb.SoloDecoder() for _ in range(1000)]
    L.solo_b200_arena_stats(st)
    assert st[3] >= 1000 and st[2] <= 8
    for h in d:
        h.close()
    print("10000 encoder handles in %.3f s" % dt)
