"""GPU tier (B200): parity tests proper, through the C ABI of the nvcc-built library, against the oracle on the
same seeded inputs; plus size-independent properties at BASELINE.json's full sizes."""
import json
import os

import numpy as np
import pytest

import parity_cases as pc
from conftest import GOLDEN_DIR
from lyra_b200 import _capi

pytestmark = pytest.mark.gpu


def test_codec_parity_speech_with_loss(gpu_api, oracle, sample1):
    pc.run_codec_parity(_capi.Context, gpu_api, oracle, max_streams=100, stream_ids=[0, 5, 17, 31, 32, 64, 99],
                        frames=60, bits=64, wav=sample1, loss_every=6)


@pytest.mark.parametrize("bits", [64, 120, 184])
def test_codec_parity_noise_all_bitrates(gpu_api, oracle, bits):
    pc.run_codec_parity(_capi.Context, gpu_api, oracle, max_streams=48, stream_ids=list(range(48)), frames=25, bits=bits,
                        seed=bits, check=[0, 1, 15, 16, 33, 47])


@pytest.mark.parametrize("kind", ["loud", "silence"])
def test_codec_parity_extreme_inputs(gpu_api, oracle, kind):
    pc.run_codec_parity(_capi.Context, gpu_api, oracle, max_streams=16, stream_ids=[3, 4, 9], frames=12, bits=120, kind=kind)


@pytest.mark.parametrize("kind", ["speech", "noise", "loud"])
def test_tensor_decoder_mode_within_tolerance(gpu_api, oracle, sample1, kind):
    # opt-in split-precision TF32 decoder: packets stay bit-exact, PCM within TENSOR_PCM_TOL_LSB of the oracle
    worst = pc.run_codec_parity(_capi.Context, gpu_api, oracle, max_streams=40, stream_ids=[0, 7, 8, 21, 39], frames=60,
                                bits=64 if kind != "loud" else 184, wav=sample1 if kind == "speech" else None,
                                kind="noise" if kind == "speech" else kind, loss_every=9, decoder_mode="tensor", seed=5)
    print("tensor-mode decoder, %s: worst |PCM - oracle| = %d LSB" % (kind, worst))
    assert worst <= pc.TENSOR_PCM_TOL_LSB


def test_tensor_decoder_mode_full_size_matches_exact_mode(gpu_api):
    # 4096 streams x 20 frames: the tensor-mode PCM stays within the tolerance of the exact-mode PCM on every stream
    n = 4096
    rng = np.random.default_rng(11)
    a = _capi.Context(n, capi=gpu_api)
    b = _capi.Context(n, capi=gpu_api)
    b.set_decoder_mode("tensor")
    worst = 0
    for f in range(20):
        pcm = pc.synth_pcm(rng, n, "noise")
        pk = a.encode(pcm, 64)
        assert np.array_equal(pk, b.encode(pcm, 64))
        worst = max(worst, int(np.abs(a.decode(pk, 64).astype(int) - b.decode(pk, 64).astype(int)).max()))
    a.close()
    b.close()
    print("tensor vs exact decoder, 4096 streams: worst |dPCM| = %d LSB" % worst)
    assert worst <= pc.TENSOR_PCM_TOL_LSB


def test_priority_switch(gpu_api, oracle):
    # lyra_b200_set_priority re-creates the context's streams between hops; state and results are unaffected
    pc.run_priority_switch(_capi.Context, gpu_api, oracle, n=20, frames=8)


@pytest.mark.parametrize("mode", ["exact", "tensor"])
def test_sixteen_stream_tiles(gpu_api, oracle, sample1, monkeypatch, mode):
    # the alternative tile size (LYRA_B200_TILE_STREAMS=16, one block per SM) runs the same kernels with other tile shapes
    monkeypatch.setenv("LYRA_B200_TILE_STREAMS", "16")
    ctx = _capi.Context(16, capi=gpu_api)
    assert ctx.tile_streams == 16
    ctx.close()
    pc.run_codec_parity(_capi.Context, gpu_api, oracle, max_streams=40, stream_ids=[0, 15, 16, 33, 39], frames=24, bits=120,
                        wav=sample1, loss_every=5, decoder_mode=mode)


def test_bitrate_switch_mid_stream(gpu_api, oracle):
    # LyraEncoder::set_bitrate (lyra/lyra_encoder.cc:158-167): the number of quantized bits may change from hop to hop
    n, ids = 3, np.array([1, 8, 9], dtype=np.int32)
    ctx = _capi.Context(16, capi=gpu_api)
    from conftest import MODEL_DIR
    codecs = [oracle.Codec(MODEL_DIR) for _ in range(n)]
    rng = np.random.default_rng(3)
    for f, bits in enumerate([64, 184, 120, 64, 120, 184, 64, 64]):
        pcm = pc.synth_pcm(rng, n)
        pk = ctx.encode(pcm, bits, stream_ids=ids)
        out = ctx.decode(pk, bits, stream_ids=ids)
        for k in range(n):
            opkt, _, _ = codecs[k].encode(pcm[k], bits)
            opcm, _, _ = codecs[k].decode(opkt, bits)
            assert bytes(pk[k]) == opkt and np.array_equal(out[k], opcm), (f, bits, k)
    ctx.close()


def test_non_standard_bit_counts(gpu_api, oracle):
    # any multiple of 4 up to 184 is accepted by Quantize (residual_vector_quantizer.cc:79-89)
    for bits in (4, 60, 100, 180):
        pc.run_codec_parity(_capi.Context, gpu_api, oracle, max_streams=4, stream_ids=[2], frames=2, bits=bits, seed=bits)


def test_plugin_surface(gpu_api, oracle):
    pc.run_plugin_surface_parity(_capi.Context, gpu_api, oracle, n=9, frames=4)


def test_reset_and_isolation(gpu_api, oracle):
    pc.run_reset_and_isolation(_capi.Context, gpu_api, oracle)


def test_error_paths(gpu_api):
    pc.run_error_paths(_capi.Context, gpu_api, _capi.LyraB200Error)


def test_logmel(gpu_api, oracle, sample1):
    pc.run_logmel_parity(_capi.Context, gpu_api, oracle, sample1, n=6, frames=8)


def test_noise_estimator(gpu_api, oracle, sample1):
    pc.run_noise_estimator_parity(_capi.Context, gpu_api, oracle, sample1, n=9, frames=120)


def test_decode_track_noise_sparse_and_dense(gpu_api, oracle, sample1):
    pc.run_decode_track_noise_parity(_capi.Context, gpu_api, oracle, sample1, stream_ids=[0, 3, 8, 30], max_streams=32, frames=40)
    # dense call over 1024 streams: cut into two concurrent sub-batches, each followed by its own estimator update
    pc.run_decode_track_noise_parity(_capi.Context, gpu_api, oracle, sample1, n=1024, frames=8, check=[0, 7, 511, 512, 777, 1023])


def test_role_contexts(gpu_api, oracle):
    pc.run_role_contexts(_capi.Context, gpu_api, oracle, _capi.LyraB200Error, frames=20)


@pytest.mark.parametrize("mode", ["exact", "tensor"])
def test_schedule_independence_full_size(gpu_api, mode):
    # 4096 streams x 24 frames: the result may not depend on how the call is cut into concurrent sub-batches, on the number
    # of resident blocks the scheduler mixes, or on encoder and decoder living in separate contexts
    n = 4096
    rng = np.random.default_rng(21)
    ref = _capi.Context(n, capi=gpu_api)
    ref.set_split(1)
    ref.set_decoder_mode(mode)
    alt = _capi.Context(n, capi=gpu_api)
    alt.set_split(3)
    alt.set_decoder_mode(mode)
    enc = _capi.Context(n, capi=gpu_api, roles="encoder")
    dec = _capi.Context(n, capi=gpu_api, roles="decoder")
    dec.set_decoder_mode(mode)
    enc.set_split(2)
    dec.set_split(4)
    for f in range(24):
        pcm = pc.synth_pcm(rng, n, "noise" if f % 5 else "loud")
        bits = (64, 120, 184)[f % 3]
        received = (rng.random(n) < 0.9).astype(np.uint8)
        pk = ref.encode(pcm, bits)
        out = ref.decode(pk, bits, received=received)
        assert np.array_equal(pk, alt.encode(pcm, bits)) and np.array_equal(pk, enc.encode(pcm, bits)), f
        assert np.array_equal(out, alt.decode(pk, bits, received=received)), f
        assert np.array_equal(out, dec.decode(pk, bits, received=received)), f
    for c in (ref, alt, enc, dec):
        c.close()


@pytest.mark.parametrize("n", [64, 1024])
def test_cuda_graphs_replay_matches_direct_calls(gpu_api, n):
    # lyra_b200_set_graphs: dense host-buffer calls on page-locked buffers replay a captured graph; the streaming state must
    # advance exactly as with directly issued calls (30 hops, two rotating buffer pairs, loss masks, a change of bit rate)
    import ctypes as C

    import torch
    rng = np.random.default_rng(5)
    ref = _capi.Context(n, capi=gpu_api)
    gr = _capi.Context(n, capi=gpu_api)
    gr.set_graphs(True)
    lib = gpu_api.lib
    pin_pcm = [torch.zeros((n, 320), dtype=torch.int16).pin_memory() for _ in range(2)]
    pin_pk = [torch.zeros((n, 23), dtype=torch.uint8).pin_memory() for _ in range(2)]
    pin_rec = [torch.zeros(n, dtype=torch.uint8).pin_memory() for _ in range(2)]
    pin_out = torch.zeros((n, 320), dtype=torch.int16).pin_memory()

    def p(t):
        return C.c_void_p(t.data_ptr())
    for f in range(30):
        b = f % 2
        bits = 64 if f < 20 else 120
        pb = _capi.packet_bytes(bits)
        pcm = pc.synth_pcm(rng, n, "noise" if f % 4 else "loud")
        received = (rng.random(n) < 0.85).astype(np.uint8)
        pk = ref.encode(pcm, bits)
        out = ref.decode(pk, bits, received=received)
        pin_pcm[b].numpy()[:] = pcm
        pin_rec[b].numpy()[:] = received
        assert lib.lyra_b200_encode(gr.h, None, n, p(pin_pcm[b]), bits, p(pin_pk[b])) == 0
        got_pk = pin_pk[b].numpy().reshape(-1)[: n * pb].reshape(n, pb)
        assert np.array_equal(pk, got_pk), f
        assert lib.lyra_b200_decode(gr.h, None, n, p(pin_pk[b]), p(pin_rec[b]), bits, p(pin_out)) == 0
        assert np.array_equal(out, pin_out.numpy()), f
    # 30 encode + 30 decode calls over 2 buffer pairs and 2 bit rates: 4 + 4 captures, every other call is a replay
    assert gr.graph_replays() >= 40, gr.graph_replays()
    assert ref.graph_replays() == 0
    # pageable host buffers (the ctypes wrappers allocate with numpy) cannot be captured: the call must run directly, same results
    replays = gr.graph_replays()
    pcm = pc.synth_pcm(rng, n, "noise")
    pk = ref.encode(pcm, 64)
    assert np.array_equal(pk, gr.encode(pcm, 64)) and np.array_equal(ref.decode(pk, 64), gr.decode(pk, 64))
    assert gr.graph_replays() == replays
    gr.set_graphs(False)
    pcm = pc.synth_pcm(rng, n, "noise")
    assert np.array_equal(ref.encode(pcm, 64), gr.encode(pcm, 64))
    ref.close()
    gr.close()


def test_golden_fixture_packets(gpu_api, sample1):
    """Committed fixtures (tests/golden/oracle_sample1.json): the GPU path reproduces them without the oracle present."""
    with open(os.path.join(GOLDEN_DIR, "oracle_sample1.json")) as f:
        g = json.load(f)
    ctx = _capi.Context(3, capi=gpu_api)
    for h in range(g["hops"]):
        x = np.tile(sample1[320 * h:320 * h + 320], (3, 1))
        for k, bits in enumerate((64, 120, 184)):
            pkt = ctx.encode(x[k:k + 1], bits, stream_ids=np.array([k], dtype=np.int32))
            assert bytes(pkt[0]).hex() == g["packets_%d" % bits][h], (bits, h)
            pcm = ctx.decode(pkt, bits, stream_ids=np.array([k], dtype=np.int32))
            assert int((pcm[0].astype(np.int64) * np.arange(1, 321)).sum()) == g["pcm_checksum_%d" % bits][h]
    ctx.close()


def test_integration_criterion_on_gpu(gpu_api, oracle, sample1):
    """lyra/lyra_integration_test.cc:132-142 on the GPU path: every hop's log-spectral distance < 2.0."""
    ctx = _capi.Context(3, capi=gpu_api)
    hops = 150
    worst = [0.0, 0.0, 0.0]
    for h in range(hops):
        x = sample1[320 * h:320 * h + 320]
        for k, bits in enumerate((64, 120, 184)):
            ids = np.array([k], dtype=np.int32)
            y = ctx.decode(ctx.encode(x[None], bits, stream_ids=ids), bits, stream_ids=ids)[0]
            a = ctx.logmel(x[None], num_mel_bins=64, bank=0, stream_ids=ids)[0]
            b = ctx.logmel(y[None], num_mel_bins=64, bank=1, stream_ids=ids)[0]
            worst[k] = max(worst[k], oracle.log_spectral_distance(a, b))
    assert max(worst) < 2.0, worst
    ctx.close()


@pytest.mark.parametrize("n,bits", [(1024, 64), (4096, 64), (4096, 120), (4096, 184)])
def test_full_size_properties(gpu_api, oracle, n, bits):
    """BASELINE configs 2/3 sizes.  Properties that need no per-stream oracle:
    (1) batch independence: streams fed the same audio produce identical packets/PCM wherever they sit in the batch;
    (2) a sample of streams with distinct audio matches the oracle bit for bit;
    (3) packet -> dequantize -> quantize is idempotent on the decoded features' indices."""
    ctx = _capi.Context(n, capi=gpu_api)
    rng = np.random.default_rng(n + bits)
    base = rng.integers(-8192, 8192, size=(6, 320), dtype=np.int16)
    distinct = sorted(set([7, 100, n // 2 + 1, n - 2]))
    refs = {k: oracle.Codec(_capi.MODEL_DIR) for k in distinct}
    same_ref = oracle.Codec(_capi.MODEL_DIR)
    for f in range(6):
        pcm = np.tile(base[f], (n, 1))
        other = rng.integers(-8192, 8192, size=(len(distinct), 320), dtype=np.int16)
        for j, k in enumerate(distinct):
            pcm[k] = other[j]
        pk = ctx.encode(pcm, bits)
        out = ctx.decode(pk, bits)
        same = np.array([k for k in range(n) if k not in distinct])
        assert (pk[same] == pk[same[0]]).all()
        assert (out[same] == out[same[0]]).all()
        opkt, _, _ = same_ref.encode(base[f], bits)
        opcm, _, _ = same_ref.decode(opkt, bits)
        assert bytes(pk[same[0]]) == opkt and np.array_equal(out[same[-1]], opcm)
        for j, k in enumerate(distinct):
            opkt, _, _ = refs[k].encode(pcm[k], bits)
            opcm, _, _ = refs[k].decode(opkt, bits)
            assert bytes(pk[k]) == opkt and np.array_equal(out[k], opcm)
        feats = ctx.dequantize(pk[:64], bits)
        assert (ctx.quantize(feats, 4)[:, 0] >> 4 == pk[:64, 0] >> 4).all()     # first-stage index is a fixed point
    ctx.close()


def test_decoder_only_concealment_4096(gpu_api, oracle):
    """BASELINE config 4 (decoder-only PLC path): no packets at all, then Bernoulli(0.9) reception."""
    n, bits = 4096, 64
    ctx = _capi.Context(n, capi=gpu_api)
    rng = np.random.default_rng(1234)
    check = [0, 77, 2048, 4095]
    refs = {k: oracle.Codec(_capi.MODEL_DIR) for k in check}
    mels = {k: oracle.LogMel(16000, 320, 640, 160) for k in check}
    pk = rng.integers(0, 256, size=(n, 8), dtype=np.uint8)
    for f in range(5):
        rec = np.zeros(n, np.uint8) if f < 2 else (rng.random(n) < 0.9).astype(np.uint8)
        out = ctx.decode(pk, bits, received=rec)
        mel = ctx.logmel(out, num_mel_bins=160)                 # NoiseEstimator's extractor runs on every decoded hop
        assert np.isfinite(mel).all() and mel.shape == (n, 160)
        for k in check:
            assert np.array_equal(mel[k], mels[k].extract(out[k])), "log-mel mismatch frame %d stream %d" % (f, k)
        for k in check:
            opcm, _, _ = refs[k].decode(bytes(pk[k]) if rec[k] else None, bits)
            assert np.array_equal(out[k], opcm)
    ctx.close()


def test_cpp_components_against_oracle(gpu_api, oracle, tmp_path):
    """include/lyra_b200/lyra_b200_components.h: the reference's plugin classes re-hosted on the C ABI (C++)."""
    import subprocess
    from conftest import ROOT
    exe = str(tmp_path / "test_components")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle"),
                           os.path.join(ROOT, "tests", "cpp", "test_components.cc"), "-o", exe,
                           "-L" + os.path.join(ROOT, "lyra_b200"), "-llyra_b200", "-L" + os.path.join(ROOT, "oracle", "_build"), "-llyra_oracle",
                           "-Wl,-rpath," + os.path.join(ROOT, "lyra_b200"), "-Wl,-rpath," + os.path.join(ROOT, "oracle", "_build"), "-lpthread"])
    env = dict(os.environ, LYRA_B200_MAX_STREAMS="64")
    out = subprocess.run([exe, _capi.MODEL_DIR], capture_output=True, text=True, env=env)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout + out.stderr


def test_cpp_duplex_server_example(gpu_api, oracle, tmp_path):
    """examples/duplex_server.cc on the GPU: checksum of the decoded audio against the oracle (small), then a full-size run."""
    import subprocess
    from conftest import MODEL_DIR, ROOT
    exe = str(tmp_path / "duplex_server")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "duplex_server.cc"),
                           "-o", exe, "-L" + os.path.join(ROOT, "lyra_b200"), "-llyra_b200", "-Wl,-rpath," + os.path.join(ROOT, "lyra_b200"), "-lpthread"])
    streams, steps = 16, 5

    def hop(stream, step):          # FillHop of the example
        x = (2463534242 ^ (stream * 7919 + step * 104729)) & 0xFFFFFFFF
        out = np.empty(320, dtype=np.int16)
        for i in range(320):
            x = (x * 1664525 + 1013904223) & 0xFFFFFFFF
            out[i] = ((x >> 16) & 16383) - 8192
        return out

    want = 0
    for s in range(streams):
        c = oracle.Codec(MODEL_DIR)
        for i in range(steps):
            pkt, _, _ = c.encode(hop(s, i), 120)
            pcm, _, _ = c.decode(pkt, 120)
        want += int(pcm.astype(np.int64).sum())
    out = subprocess.run([exe, MODEL_DIR, str(streams), str(steps), "2", "120"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert int(out.stdout.strip().rsplit("checksum", 1)[1]) == want, out.stdout
    big = subprocess.run([exe, MODEL_DIR, "4096", "60", "2", "64"], capture_output=True, text=True, timeout=300)
    assert big.returncode == 0, big.stdout + big.stderr
    print(big.stdout.strip())


@pytest.mark.parametrize("probe,cases", [("umma_probe", 2), ("umma_probe2", 7)])
def test_umma_probes_on_hardware(tmp_path, probe, cases):
    """tests/cpp/umma_probe{,2}.cu built with nvcc: the tcgen05 / TMEM instruction sequences of device_compat.h that the product's
    UMMA kernel (DecoderKernelDU) is made of - shared-memory descriptors, split-precision TF32 MMAs, A operands in tensor memory,
    tcgen05.st / wide tcgen05.ld, kind::i8, N = 160 / 16 shapes, bulk stores.  The product depends on them: a mismatch is a failure."""
    import subprocess

    import __graft_entry__ as g
    from conftest import ROOT
    exe = str(tmp_path / probe)
    subprocess.check_call([g.NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I" + os.path.join(ROOT, "lyra_b200", "csrc"),
                           "-o", exe, os.path.join(ROOT, "tests", "cpp", probe + ".cu")])
    out = subprocess.run(["timeout", "60", exe], capture_output=True, text=True, timeout=120)
    print(out.stdout.strip())
    assert out.returncode == 0 and out.stdout.count("MATCH") == cases and "MISMATCH" not in out.stdout, out.stdout + out.stderr


# ---- packet-loss concealment, comfort noise, DTX (SURVEY.md section 8 rows f2, f4) ----

def test_comfort_noise_generator_parity(gpu_api, oracle):
    pc.run_cng_parity(_capi.Context, gpu_api, oracle, stream_ids=(0, 5, 63, 64), hops=12)


def test_comfort_noise_reference_criterion_on_gpu(gpu_api, oracle):
    """comfort_noise_generator_test.cc:100-138 on the GPU path: log-mel of the generated noise within LSD 0.7 of its conditioning."""
    ctx = _capi.Context(8, capi=gpu_api)
    ctx.set_cng_seed(1)
    rng = np.random.default_rng(1)
    x = rng.integers(-10000, 10001, size=(8, 320)).astype(np.int16)
    for _ in range(10):
        fi = ctx.logmel(x, 160, bank=0)
        fo = ctx.logmel(ctx.cng_generate(fi), 160, bank=1)
    lsd = [oracle.log_spectral_distance(fi[k], fo[k]) for k in range(8)]
    print("CNG log-spectral distance per stream:", ["%.3f" % v for v in lsd])
    assert max(lsd) < 0.7
    ctx.close()


@pytest.mark.parametrize("mode", ["exact", "tensor"])
def test_plc_state_machine_parity(gpu_api, oracle, sample1, mode):
    pc.run_plc_parity(_capi.Context, gpu_api, oracle, max_streams=64, stream_ids=(1, 6, 9, 40, 63), frames=40, wav=sample1,
                      outages=((3, 12), (5, 3), (0, 0), (10, 25), (20, 7)), decoder_mode=mode)
    if mode == "exact":
        pc.run_plc_state_peer(_capi.Context, gpu_api, oracle)


def test_plc_full_size_bernoulli_loss(gpu_api, oracle):
    """BASELINE configs[3] with the reference's real state machine: 4096 streams, burst losses; a few streams are checked against
    the oracle, all of them against the invariants of the state machine."""
    n, bits = 4096, 64
    ctx = _capi.Context(n, capi=gpu_api)
    ctx.set_cng_seed(21)
    rng = np.random.default_rng(1234)
    check = [0, 77, 2048, 4095]
    decs = {k: oracle.Decoder(_capi.MODEL_DIR, cng_seed=21 + k) for k in check}
    pk = rng.integers(0, 256, size=(n, 8), dtype=np.uint8)
    burst = np.zeros(n, dtype=np.int32)
    cn_hops = 0
    for f in range(24):
        start = (rng.random(n) < 0.08) & (burst == 0)
        burst[start] = rng.integers(1, 12, size=int(start.sum()))
        rec = (burst == 0).astype(np.uint8)
        burst = np.maximum(burst - 1, 0)
        out, cn = ctx.decode_plc(pk, bits, received=rec)
        st = ctx.plc_state(n)
        assert ((st[:, 0] % 320 == 0) & (st[:, 0] >= 0) & (st[:, 0] <= 1280)).all()
        assert np.isin(st[:, 1], [0, 320, 640]).all() and np.isin(st[:, 2], [-1, 1]).all()
        assert (st[rec == 1, 0] == 0).all()                      # a received packet always ends concealment
        assert (cn == (st[:, 1] == 640)).all()
        cn_hops += int(cn.sum())
        for k in check:
            if rec[k]:
                assert decs[k].set_encoded_packet(bytes(pk[k]))
            assert np.array_equal(out[k], decs[k].decode_samples(320)), (f, k)
    assert cn_hops > 0
    ctx.close()


def test_dtx_encoder_parity(gpu_api, oracle, sample1):
    pc.run_dtx_parity(_capi.Context, gpu_api, oracle, wav=sample1, frames=40)


def test_resampler_parity(gpu_api, oracle):
    pc.run_resampler_parity(_capi.Context, gpu_api, oracle)


@pytest.mark.parametrize("rate", [8000, 32000, 48000])
def test_integration_criterion_other_sample_rates(gpu_api, oracle, rate):
    from conftest import read_wav_any
    wav = read_wav_any("sample1_%dkHz.wav" % (rate // 1000), rate)
    worst = pc.run_integration_other_rates(_capi.Context, gpu_api, oracle, rate=rate, wav=wav)
    print("integration LSD at %d Hz: worst hop %.3f" % (rate, worst))
    assert worst < 2.0
