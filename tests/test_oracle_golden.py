"""CPU: the oracle against golden vectors produced by the REFERENCE's own modules (tests/golden/make_golden.py) and the
reference's own fixtures (infer/modules/vc/lgdsng.npz, logs/mute/2a_f0, 2b-f0nsf)."""
import contextlib
import math
import os

import numpy as np
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@contextlib.contextmanager
def one_thread():
    """As tests/golden/make_golden.py::one_thread made the glue goldens: the oracle's float32 sums depend on the thread count."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        yield
    finally:
        torch.set_num_threads(threads)


def test_synth_oracle_matches_reference_golden():
    from oracle import synth as OS, weights as OW
    z = np.load(os.path.join(G, "synth_v2_48k_T24.npz"))
    w, cfg = OW.synth_weights(1234), OW.V2_48K_CONFIG
    phone = torch.from_numpy(z["phone"].astype(np.float32))
    pitch, pitchf = torch.from_numpy(z["pitch"]), torch.from_numpy(z["pitchf"])
    T = phone.shape[1]
    torch.manual_seed(int(z["seed"]))
    n1 = torch.randn(1, 192, T); torch.rand(1, 1, 1); n2 = torch.randn(1, T * 480, 1)
    with torch.no_grad():
        out = OS.synth_infer(w, cfg, phone, torch.tensor([T]), torch.tensor([int(z["sid"])]), pitch, pitchf, n1, n2)[0, 0]
    assert np.abs(out.numpy() - z["out"]).max() < 5e-6
    torch.manual_seed(int(z["seed_rt"]))
    n1 = torch.randn(1, 192, T); torch.rand(1, 1, 1); n2 = torch.randn(1, 6 * 480, 1)   # flow_head = max(16-24, 0) = 0
    with torch.no_grad():
        out = OS.synth_infer(w, cfg, phone, torch.tensor([T]), torch.tensor([int(z["sid"])]), pitch, pitchf, n1, n2, 16, 6, 6)[0, 0]
    assert np.abs(out.numpy() - z["out_rt"]).max() < 5e-6


def test_rmvpe_oracle_matches_reference_golden():
    from oracle import rmvpe as ORM, weights as OW
    z = np.load(os.path.join(G, "rmvpe_e2e_64.npz"))
    with torch.no_grad():
        hid = ORM.e2e_forward(OW.rmvpe_weights(4321), torch.from_numpy(z["mel"]))[0].numpy()
    assert np.abs(hid - z["hidden"]).max() < 1e-5
    assert np.abs(ORM.decode(z["hidden"].copy(), 0.03) - z["f0"]).max() == 0
    for x, r in zip(z["tracks"], z["resized"]):
        assert np.array_equal(ORM.interpolate_f0(ORM.resize_f0(x.copy(), 37)), r)


def test_post_process_against_reference_fixtures():
    """lgdsng.npz: the reference stores (pitch, pitchf) produced by its own post_process (hash.py:51-54);
    logs/mute: unvoiced input -> coarse 1, f0 0 (gen.py:34-40)."""
    from oracle import rmvpe as ORM
    from rvc_b200 import f0post
    z = np.load(os.path.join(G, "ref_fixtures_f0.npz"))
    for fn in (ORM.post_process, lambda f, k: f0post.post_process(f, k)):
        c, f = fn(z["lgdsng_pitchf"].copy(), 0)
        assert np.array_equal(c, z["lgdsng_pitch"])
        c, f = fn(z["mute_2b_f0nsf"].copy(), 0)
        assert np.array_equal(c, z["mute_2a_f0"]) and (f == 0).all()


def test_hubert_oracle_matches_transformers_golden():
    from oracle import hubert as OH, weights as OW
    z = np.load(os.path.join(G, "hubert_hf_0p5s.npz"))
    w = OW.hubert_weights(777)
    wav = OW.synth_voice(0.5, seed=6)[None]
    with torch.no_grad():
        assert np.abs(OH.extract_features(w, wav, 9)[0].numpy() - z["layer9"]).max() < 5e-5
        assert np.abs(OH.extract_features(w, wav, 12)[0].numpy() - z["layer12"]).max() < 5e-5


def test_ivf_oracle_against_an_independent_knn():
    """faiss is absent (un-vendored, un-pinned), so the IVF-Flat oracle *defines* the expected arithmetic; its SEMANTICS
    (squared-L2 nearest centroid, exact top-8 inside that list, ascending order, ids) are cross-checked here against an
    independent implementation: scikit-learn's brute-force neighbours in float64 restricted to the probed list.  Index sets
    must agree wherever the 8th/9th distance gap exceeds float32 resolution; distances to 1e-5 relative."""
    from sklearn.neighbors import NearestNeighbors
    from oracle import ivf as OI, weights as OW
    vec = OW.index_vectors(4000, 768, 3).numpy()
    idx = OI.build_ivf(vec, None, seed=1, exact_assign=True)
    rng = np.random.default_rng(0)
    q = (vec[rng.integers(0, 4000, 60)] + 0.05 * rng.standard_normal((60, 768))).astype(np.float32)
    D, I = idx.search(q, 8)
    cen = NearestNeighbors(n_neighbors=1, algorithm="brute", metric="sqeuclidean").fit(idx.centroids.astype(np.float64))
    lists = cen.kneighbors(q.astype(np.float64), return_distance=False)[:, 0]
    checked = 0
    for qi in range(q.shape[0]):
        a, b = idx.list_off[lists[qi]], idx.list_off[lists[qi] + 1]
        ids = idx.list_ids[a:b]
        if len(ids) == 0:
            assert (I[qi] == -1).all()
            continue
        k = min(8, len(ids))
        nn = NearestNeighbors(n_neighbors=min(k + 1, len(ids)), algorithm="brute", metric="sqeuclidean").fit(vec[ids].astype(np.float64))
        d64, j = nn.kneighbors(q[qi:qi + 1].astype(np.float64))
        d64, j = d64[0], ids[j[0]]
        assert np.all(np.diff(D[qi, :k]) >= 0) and (I[qi, k:] == -1).all()
        assert np.allclose(D[qi, :k], d64[:k], rtol=1e-5, atol=1e-5)
        if len(d64) > k and (d64[k] - d64[k - 1]) < 1e-4 * d64[k - 1]:
            continue                                   # near-tie at the cut: set membership is arithmetic-dependent
        assert set(I[qi, :k].tolist()) == set(j[:k].tolist()), qi
        checked += 1
    assert checked >= 50


def test_torchgate_oracle_matches_reference_golden():
    """oracle/torchgate.py vs the outputs of the reference's own TorchGate class (both on CPU torch.stft: bit-equal)."""
    import math
    from oracle import torchgate as OT
    z = np.load(os.path.join(G, "torchgate.npz"))

    def inputs(seed, n, n_noise, sr):
        g = torch.Generator().manual_seed(seed)
        t = torch.arange(n_noise) / sr
        tone = sum(torch.sin(2 * math.pi * (180.0 + 40.0 * t) * h * t) / h for h in (1, 2, 3, 5))
        env = ((t * 3.0) % 1.0 < 0.6).float()
        xn = 0.3 * tone * env + 0.02 * torch.randn(n_noise, generator=g)
        return xn[-n:].clone()[None], xn[None]
    x, xn = inputs(21, 9600, 48000, 48000)
    assert np.abs(OT.torchgate(x, xn, 48000, 1920, prop_decrease=0.9)[0].numpy() - z["rt_y"]).max() <= 1e-7
    assert np.abs(OT.torchgate(x, None, 48000, 1920, prop_decrease=0.9)[0].numpy() - z["rt_y_self"]).max() <= 1e-7
    x, xn = inputs(22, 8192, 32000, 16000)
    assert np.abs(OT.torchgate(x, xn, 16000)[0].numpy() - z["d16_y"]).max() <= 1e-7
    assert np.abs(OT.torchgate(x, None, 16000, nonstationary=True, prop_decrease=0.8)[0].numpy() - z["d16_ns_y"]).max() <= 1e-7


def test_resample_table_equals_torchaudio():
    """The product's windowed-sinc table (engine.sinc_resample_kernel) is torchaudio's, entry for entry."""
    import torchaudio.transforms as tat
    from rvc_b200 import engine
    for o, n in ((48000, 16000), (16000, 48000), (40000, 48000), (44100, 16000), (32000, 48000)):
        k, w, up, down = engine.sinc_resample_kernel(o, n)
        r = tat.Resample(o, n, dtype=torch.float32)
        assert torch.equal(k, r.kernel[:, 0]) and w == r.width and (up, down) == (n // math.gcd(o, n), o // math.gcd(o, n))


def test_phase_vocoder_oracle_matches_reference_golden():
    """oracle.rtrvc.phase_vocoder vs the outputs of the reference's own function (gui.py:27-48, executed from its source by
    tests/golden/make_golden.py): same torch ops in the same order -> bit-equal."""
    from oracle import rtrvc as ORT
    z = np.load(os.path.join(G, "phase_vocoder.npz"))
    for n in (1920, 1600, 441):
        fi, fo = ORT.fade_windows(n)
        y = ORT.phase_vocoder(torch.from_numpy(z[f"a{n}"]), torch.from_numpy(z[f"b{n}"]), fo, fi).numpy()
        assert np.array_equal(y, z[f"y{n}"]), n


def test_callback_oracle_matches_the_reference_statements():
    """oracle.rtrvc.OracleCallback / SolaTail vs outputs of the reference's OWN callback statements (gui.py GUI.audio_infer: the input
    rings + input noise gate + cross-fade + 16 kHz resampling, and the SOLA step with both cross-fades), executed from the reference's
    source by tests/golden/make_golden.py::callback_pieces on a stand-in ``self``.  Inputs are re-drawn from the same seeds."""
    from oracle import rtrvc as ORT
    z = np.load(os.path.join(G, "callback_pieces.npz"))
    sr, zc = 24000, 240

    class _Silent:                                    # OracleCallback needs an engine: the pre-processing under test runs before it
        tgt_sr = sr

        def infer(self, wav, block_frame_16k, skip_head, return_length):
            return np.zeros(return_length * zc, dtype=np.float32)
    orc = ORT.OracleCallback(_Silent(), samplerate=sr, block_time=0.16, crossfade_time=0.05, extra_time=0.5, I_noise_reduce=True)
    assert (orc.block_frame, orc.block_frame_16k, orc.sola_buffer_frame) == (3840, 2560, 960)
    g = torch.Generator().manual_seed(91)
    for b in range(3):
        indata = (torch.randn(orc.block_frame, generator=g) * (0.3 if b != 1 else 0.02)).numpy()
        orc.block(indata)
        assert np.array_equal(orc.input_wav_res[-orc.block_frame_16k - 160:].numpy(), z[f"pre_res{b}"]), b
        assert np.array_equal(orc.input_wav_denoise[-orc.block_frame:].numpy(), z[f"pre_den{b}"]), b
        assert np.array_equal(orc.nr_buffer.numpy(), z[f"pre_nr{b}"]), b
    for use_pv in (False, True):
        tail = ORT.SolaTail(3840, 960, 240, use_pv=use_pv)
        g = torch.Generator().manual_seed(92)
        offs = []
        for b in range(3):
            y = torch.randn(3840 + 960 + 240, generator=g) * 0.2
            out, off = tail.step(y)
            offs.append(off)
            assert off == int(z[f"sola{int(use_pv)}_off{b}"]) and np.array_equal(out.numpy(), z[f"sola{int(use_pv)}_{b}"]), (use_pv, b)
        assert len(set(offs)) > 1


@one_thread()
def test_pipeline_vc_glue_oracle_matches_the_reference_method():
    """oracle.pipeline.OraclePipeline.vc vs what the reference's OWN ``Pipeline.vc`` (pipeline.py:76-184, executed from its source on
    duck-typed components by tests/golden/make_golden.py::vc_glue) hands to the synthesizer: retrieval weights + blend, x2 nearest
    up-sampling, p_len truncation, protect mix, final_proj (v1) -- bit-equal on the stored channel subset."""
    from oracle import ivf as OI, pipeline as OP, weights as OW
    z = np.load(os.path.join(G, "vc_glue.npz"))
    hw = OW.hubert_weights(777)
    audio0 = OW.synth_voice(0.62, seed=12).numpy().astype(np.float32)
    idx = OI.build_ivf(OW.index_vectors(500, 768, 3).numpy(), 8, seed=0, exact_assign=True)
    big = idx.reconstruct_n(0, idx.ntotal)
    p_len = audio0.shape[0] // 160
    pitchf = torch.zeros(1, p_len); pitchf[0, 10:40] = 180.0 + torch.arange(30)
    pitch = torch.where(pitchf > 0, torch.full_like(pitchf, 60), torch.ones_like(pitchf)).long()
    seen = {}
    real_synth = OP.OS.synth_infer
    try:
        OP.OS.synth_infer = lambda w, cfg, feats, lens, sid, p, pf, n1, n2, **kw: (seen.update(phone=feats.clone(), plen=int(lens[0]), pf=pf) or
                                                                                   torch.zeros(1, 1, 8))
        op = OP.OraclePipeline(48000, 1, 6, 38, 41, hw, None, None, OW.V2_48K_CONFIG, noise_seed=0)
        op.vc(torch.tensor([0]), audio0, pitch, pitchf, idx, big, 0.75, "v2", 0.33)
        assert seen["plen"] == int(z["v2_plen"]) == 60 and np.array_equal(seen["phone"][0, :, ::32].numpy(), z["v2_phone"])
        assert np.array_equal(seen["pf"].numpy(), z["v2_pitchf"])
        op = OP.OraclePipeline(40000, 1, 6, 38, 41, hw, None, None, OW.V1_40K_CONFIG, noise_seed=0)
        op.vc(torch.tensor([0]), audio0, pitch, pitchf, None, None, 0.0, "v1", 0.5)
        assert seen["plen"] == int(z["v1_plen"]) and seen["phone"].shape[2] == 256 and np.array_equal(seen["phone"][0, :, ::16].numpy(), z["v1_phone"])
    finally:
        OP.OS.synth_infer = real_synth


def _chunk_stub_vc(audio0, pitch, pitchf, window=160, upp=16):
    """Same stand-in as tests/golden/make_golden.py::chunk_stub_vc (kept in step by the golden itself)."""
    n = audio0.shape[0] // window
    fr = np.asarray(audio0[: n * window], dtype=np.float32).astype(np.float64).reshape(n, window)      # vc casts to float32 first (pipeline.py:91-95)
    v = fr.mean(1) + 0.25 * np.abs(fr).max(1)
    if pitchf is not None:
        m = min(n, pitchf.shape[1])
        v[:m] += 1e-3 * pitchf[0, :m].double().numpy() + 1e-4 * pitch[0, :m].double().numpy()
    return np.repeat(v, upp).astype(np.float32) * np.tile(np.linspace(0.5, 1.0, upp, dtype=np.float32), n)


def test_pipeline_control_flow_oracle_matches_the_reference_method():
    """oracle.pipeline.OraclePipeline.pipeline vs the reference's OWN ``Pipeline.pipeline`` (pipeline.py:186-366, executed from its source
    with a deterministic stand-in for ``vc``): high-pass filter, silence-point search over a 10.3 s input (three cut points at x_max = 4 s),
    per-chunk audio and pitch windows, x_pad trimming, concatenation, peak scaling; f0 and no-f0 models."""
    from oracle import pipeline as OP, weights as OW
    z = np.load(os.path.join(G, "pipeline_flow.npz"))
    audio = OW.synth_voice(10.3, seed=14).numpy().astype(np.float32)
    audio[40000:52000] *= 0.01; audio[90000:100000] *= 0.02
    p_len = (audio.shape[0] + 2 * 16000) // 160
    pitchf = (100.0 + np.arange(p_len) * 0.37).astype(np.float64)
    pitch = (1 + np.arange(p_len) % 250).astype(np.int64)
    cfg = list(OW.V2_48K_CONFIG); cfg[-1] = 1600
    op = OP.OraclePipeline(1600, 1, 1, 3, 4, None, None, None, cfg, noise_seed=0)
    op.vc = lambda sid, audio0, p, pf, *a, **k: _chunk_stub_vc(audio0, p, pf)
    out = op.pipeline(0, audio.copy(), 0, (pitch, pitchf), None, 0.0, 2, 1600, 0, 1.0, "v2", 0.33)
    assert out.shape[0] == int(z["n"]) and np.array_equal(out[::3].astype(np.float32), z["out"])
    assert abs(float(np.abs(out.astype(np.float64)).sum()) - float(z["total"])) <= 1e-6 * float(z["total"])
    out0 = op.pipeline(0, audio.copy(), 0, "rmvpe", None, 0.0, 0, 1600, 0, 1.0, "v2", 0.33)
    assert out0.shape[0] == int(z["n_nof0"]) and np.array_equal(out0[::3].astype(np.float32), z["out_nof0"])


@one_thread()
def test_rtrvc_oracle_matches_the_reference_method():
    """oracle.rtrvc.OracleRVC.infer vs the reference's OWN realtime ``RVC.infer`` (infer/lib/rtrvc.py:134-260, executed from its source
    on duck-typed components by tests/golden/make_golden.py::rtrvc_glue) over three consecutive rolling-window blocks: what reaches the
    synthesizer (features after last-frame duplication, tail-only retrieval, x2 up-sampling; the pitch-ring slices) and the ring itself."""
    from oracle import ivf as OI, rtrvc as ORT, weights as OW
    z = np.load(os.path.join(G, "rtrvc_glue.npz"))
    hw, rw, sw = OW.hubert_weights(777), OW.rmvpe_weights(4321), OW.synth_weights(1234)
    idx = OI.build_ivf(OW.index_vectors(2000, 768, 1).numpy(), None, seed=0, exact_assign=True)
    real = ORT.OS.synth_infer
    try:
        ORT.OS.synth_infer = lambda w, cfg, feats, lens, sid, p, pf, n1, n2, **kw: torch.zeros(1, 1, kw["return_length2"] * 480)
        orc = ORT.OracleRVC(hw, rw, sw, OW.V2_48K_CONFIG, idx, 0.5, key=0, noise_seed=0)
        WIN, BLK, SKIP, RET = 43520, 2560, 250, 21
        stream = OW.synth_voice(2.72 + 0.16 * 3 + 0.1, seed=9).numpy()
        for b in range(3):
            orc.infer(stream[b * BLK: b * BLK + WIN], BLK, SKIP, RET)
            tap = orc.taps[-1]
            assert list(z[f"meta{b}"]) == [tap["phone"].shape[1], SKIP, RET, RET]
            assert np.array_equal(tap["phone"][0, :, ::32].numpy(), z[f"phone{b}"]), b
            assert np.array_equal(tap["pitch"].numpy(), z[f"pitch{b}"]) and np.array_equal(tap["pitchf"].numpy(), z[f"pitchf{b}"]), b
        assert np.array_equal(orc.cache_pitch.numpy(), z["ring_pitch"]) and np.array_equal(orc.cache_pitchf.numpy(), z["ring_pitchf"])
    finally:
        ORT.OS.synth_infer = real


def test_rmvpe_compute_f0_oracle_matches_the_reference_methods():
    """oracle.rmvpe.compute_f0 vs the reference's OWN RMVPE.compute_f0 / _mel2hidden / _decode / _to_local_average_cents (rmvpe.py:96-164,
    executed from their source on the reference's own E2E network and F0Predictor base class; only the mel front end is the oracle's)."""
    from oracle import rmvpe as ORM, weights as OW
    z = np.load(os.path.join(G, "rmvpe_compute_f0.npz"))
    w = OW.rmvpe_weights(4321)
    for name, sec, seed in (("a", 1.0, 31), ("b", 0.73, 32)):
        wav = OW.synth_voice(sec, seed=seed).numpy()
        wav[int(0.4 * 16000): int(0.55 * 16000)] *= 1e-4
        with torch.no_grad():
            f0 = np.asarray(ORM.compute_f0(w, wav, None, 0.03), dtype=np.float64)
        ref = z[f"f0_{name}"]
        assert f0.shape == ref.shape and (ref > 0).any()
        assert np.array_equal(f0 > 0, ref > 0) and np.abs(f0 - ref).max() <= 1e-6 * np.abs(ref).max(), (name, np.abs(f0 - ref).max())
