"""Batched parity with *different* signal classes in neighbouring streams (SURVEY.md 8(d) ii/iii): the warps of a block, the
two lane groups of a quantiser warp and the 64 threads of an entropy-coding / decoder block then take different paths
(voiced / unvoiced, different decision delays, rewhitening, DTX-like silence, clipping) at the same time.
Every row is compared with the unmodified reference run per stream (digests in tests/golden/reference_digests.npz): payload
bytes + length fields against libjc1_fix.so, decoded PCM under a per-stream 50 % loss process against libjc1_flp.so fed
the same payloads and flags.
Tolerances: payloads bit-exact; PCM 0 LSB (the north star allows +-1)."""
import numpy as np
import pytest

from tests.util import RowDigests, assert_matches_reference, enc_row, load_clip, loss_flags, speech_replay, trim_payload

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import solo_b200
    solo_b200.lib()
    return solo_b200


def signal_classes(clip, n_rows, n_packets, seed=5):
    """int16 [n_packets, n_rows, 640]; row s belongs to class s % 8:
    0 speech, 1 noise sigma 2000, 2 noise sigma 20000, 3 zeros, 4 DC 1000, 5 +-32767 square, 6 200 Hz sine, 7 4x clipped speech."""
    rng = np.random.Generator(np.random.PCG64(seed))
    L = n_packets * 640
    t = np.arange(L)
    out = np.zeros((n_rows, L), np.int16)
    for s in range(n_rows):
        k = s % 8
        off = (s * 7919 * 640) % (len(clip) - 1)
        sp = np.take(clip, (off + t) % len(clip))
        if k == 0:
            out[s] = sp
        elif k == 1:
            out[s] = np.clip(rng.normal(0, 2000, L), -32768, 32767).astype(np.int16)
        elif k == 2:
            out[s] = np.clip(rng.normal(0, 20000, L), -32768, 32767).astype(np.int16)
        elif k == 3:
            out[s] = 0
        elif k == 4:
            out[s] = 1000
        elif k == 5:
            out[s] = np.where(((t + 13 * s) // 80) % 2 == 0, 32767, -32767).astype(np.int16)
        elif k == 6:
            out[s] = (8000 * np.sin(2 * np.pi * 200 * (t + 7 * s) / 16000)).astype(np.int16)
        else:
            out[s] = np.clip(sp.astype(np.int32) * 4, -32768, 32767).astype(np.int16)
    return np.ascontiguousarray(out.reshape(n_rows, n_packets, 640).transpose(1, 0, 2))


def hetero_flags(N, T, loss_perc=50):
    flags = np.array([loss_flags(T, loss_perc, seed=1 + s) for s in range(N)], np.int32)
    flags[::5] = 4           # every fifth row loss-free
    return flags


def run_against_reference(sb, case, x, rate):
    """x: [T, N, 640].  GPU batch vs the reference run per row (one encoder + decoder per row, digests of its outputs
    under `case`)."""
    T, N, _ = x.shape
    cap = 1024 if rate > 40000 else 256
    eb, db = sb.EncoderBatch(N, rate=rate), sb.DecoderBatch(N)
    flags = hetero_flags(N, T)
    enc, pcm_d = RowDigests(T, N), RowDigests(T, N)
    for p in range(T):
        bits, nb = eb.encode(x[p], cap=cap)
        dbits = np.zeros((N, cap), np.uint8)
        dnb = np.zeros((N, 2), np.int16)
        f_eff = np.zeros(N, np.int32)
        for s in range(N):
            b = bytes(bits[s, :max(int(nb[s, 0]), 0)])
            enc.add(p, s, enc_row(b, nb[s]))
            f = int(flags[s, p])
            if nb[s, 0] <= 0:    # DTX packet: nothing is sent, the receiver conceals
                pb, pnb, f = bytes(16), (16, 8), 1
            else:
                pb, pnb = trim_payload(b, nb[s], f)
            dbits[s, :len(pb)] = np.frombuffer(pb, np.uint8)
            dnb[s] = pnb
            f_eff[s] = f
        pcm, ret = db.decode(dbits, dnb, f_eff)
        assert (ret == 0).all()
        for s in range(N):
            pcm_d.add(p, s, pcm[s].tobytes())
    eb.close(); db.close()
    assert_matches_reference(case, enc=enc, pcm=pcm_d)


def test_neighbouring_streams_of_eight_signal_classes_match_the_reference(sb):
    x = signal_classes(load_clip(), 256, 40)
    run_against_reference(sb, "hetero_classes", x, rate=13600)


@pytest.mark.parametrize("rate", [6000, 24000, 100000])
def test_signal_classes_at_other_rates(sb, rate):
    x = signal_classes(load_clip(), 64, 20, seed=rate)
    run_against_reference(sb, "hetero_rate%d" % rate, x, rate=rate)


FULL_BATCH = dict(N=65536, T=25, cap=128)


def full_batch_sample_and_flags(N, T):
    """1 024 sampled streams spread over the batch (per-stream loss process, seed 1 + stream id) and arbitrary flags for
    every other stream."""
    sample = sorted(set(list(range(0, N, 64))))[:1024]
    flags = np.full((N, T), 4, np.int32)
    for s in sample:
        flags[s] = loss_flags(T, 50, seed=1 + s)
    rng = np.random.Generator(np.random.PCG64(11))
    other = rng.integers(1, 5, size=(N, T)).astype(np.int32)
    mask = np.ones(N, bool); mask[sample] = False
    flags[mask] = other[mask]
    return sample, flags


def test_full_batch_sample_of_1024_streams_25_packets(sb):
    """BASELINE configs 3 + 5 at full size (65 536 streams, per-stream loss process, trimming on the device): 1 024 streams
    spread over the batch x 25 packets against the reference (SURVEY.md 8(d) config 4 wording)."""
    import torch
    N, T, cap = FULL_BATCH["N"], FULL_BATCH["T"], FULL_BATCH["cap"]
    clip = load_clip()
    sample, flags = full_batch_sample_and_flags(N, T)
    dev = torch.device("cuda", 0)
    eb, db = sb.EncoderBatch(N), sb.DecoderBatch(N)
    d_bits, d_nb = torch.zeros((N, cap), dtype=torch.uint8, device=dev), torch.zeros((N, 2), dtype=torch.int16, device=dev)
    d_tb, d_tnb = torch.zeros_like(d_bits), torch.zeros_like(d_nb)
    d_pcm, d_ret = torch.zeros((N, 640), dtype=torch.int16, device=dev), torch.zeros(N, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    idx = torch.tensor(sample, device=dev)
    enc, pcm_d = RowDigests(T, len(sample)), RowDigests(T, len(sample))
    for p in range(T):
        xh = speech_replay(clip, N, 1, first_packet=p)[0]
        x = torch.from_numpy(xh).to(dev)
        f = torch.from_numpy(flags[:, p].copy()).to(dev)
        eb.encode_device(x.data_ptr(), d_bits.data_ptr(), cap, d_nb.data_ptr(), st)
        sb.apply_loss_device(d_bits.data_ptr(), d_nb.data_ptr(), f.data_ptr(), d_tb.data_ptr(), d_tnb.data_ptr(), cap, N, st)
        db.decode_device(d_pcm.data_ptr(), d_tb.data_ptr(), cap, d_tnb.data_ptr(), f.data_ptr(), d_ret.data_ptr(), st)
        torch.cuda.synchronize()
        assert int((d_ret != 0).sum().item()) == 0
        bits, nb, pcm = d_bits[idx].cpu().numpy(), d_nb[idx].cpu().numpy(), d_pcm[idx].cpu().numpy()
        for i in range(len(sample)):
            enc.add(p, i, enc_row(bits[i, :nb[i, 0]], nb[i]))
            pcm_d.add(p, i, pcm[i].tobytes())
    eb.close(); db.close()
    assert_matches_reference("hetero_full_batch", enc=enc, pcm=pcm_d)
