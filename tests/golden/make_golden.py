"""Generates tests/golden/*.npz by running the REFERENCE's own modules (imported from a checkout of the reference) and, for
HuBERT (un-vendored fairseq), transformers.HubertModel.  Weights/inputs come from seeds, so only the small outputs are stored.
Run:  python tests/golden/make_golden.py <reference checkout> [golden ...]   (no golden names: all of them)"""
import contextlib
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)
OUT = os.path.dirname(os.path.abspath(__file__))
torch.set_grad_enabled(False)

# import the REFERENCE's packages first: the product package mirrors the same module names (rvc.*, infer.*)
from rvc.synthesizer import get_synthesizer  # noqa: E402
from rvc.f0.e2e import E2E  # noqa: E402
from rvc.f0.f0 import F0Predictor  # noqa: E402
assert get_synthesizer.__code__.co_filename.startswith(REF)

from oracle import weights as OW  # noqa: E402  (seeded generators only)


@contextlib.contextmanager
def one_thread():
    """For goldens compared bit for bit: the float32 sums of the oracle HuBERT / RMVPE under the glue change with torch's CPU
    thread count, so the golden and its test both run them on one thread."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        yield
    finally:
        torch.set_num_threads(threads)


def synth():
    cpt = OW.synth_cpt(1234, "v2")
    net_g, _ = get_synthesizer(cpt, "cpu")
    T = 24
    g = torch.Generator().manual_seed(11)
    phone = (torch.randn(1, T, 768, generator=g) * 0.5).half().float()     # stored as fp16, exactly representable
    pitchf = torch.full((1, T), 0.0)
    pitchf[:, 3:20] = 200 + 30 * torch.sin(torch.arange(17) / 3.0)
    mn, mx = 1127 * math.log(1 + 50 / 700), 1127 * math.log(1 + 1100 / 700)
    fm = 1127 * torch.log(1 + pitchf / 700)
    pitch = torch.round(torch.where(fm > 0, (fm - mn) * 254 / (mx - mn) + 1, fm).clamp(1, 255)).long()
    torch.manual_seed(2024)
    out = net_g.infer(phone, torch.tensor([T]), torch.tensor([5]), pitch, pitchf)
    torch.manual_seed(2025)
    out_rt = net_g.infer(phone, torch.tensor([T]), torch.tensor([5]), pitch, pitchf, skip_head=16, return_length=6, return_length2=6)
    np.savez_compressed(os.path.join(OUT, "synth_v2_48k_T24.npz"), phone=phone.numpy().astype(np.float16), pitch=pitch.numpy(),
                        pitchf=pitchf.numpy(), out=out[0, 0].numpy(), out_rt=out_rt[0, 0].numpy(), seed=2024, seed_rt=2025, sid=5)


def rmvpe():
    m = E2E(4, 1, (2, 2)).eval()
    m.load_state_dict(OW.rmvpe_weights(4321))
    g = torch.Generator().manual_seed(5)
    mel = torch.randn(1, 128, 64, generator=g) * 3 - 4.5
    hid = m(mel)[0].numpy()
    # decode with the reference's literal per-frame loop (rmvpe.py:119-137)
    cents_mapping = np.pad(20 * np.arange(360) + 1997.3794084376191, (4, 4))
    sal = hid.copy()
    center = np.argmax(sal, axis=1); salp = np.pad(sal, ((0, 0), (4, 4))); center += 4
    ts, tc = [], []
    for i in range(salp.shape[0]):
        ts.append(salp[:, center[i] - 4:center[i] + 5][i]); tc.append(cents_mapping[center[i] - 4:center[i] + 5])
    ts, tc = np.array(ts), np.array(tc)
    dev = np.sum(ts * tc, 1) / np.sum(ts, 1); dev[np.max(salp, axis=1) <= 0.03] = 0
    f0 = 10 * (2 ** (dev / 1200)); f0[f0 == 10] = 0
    fp = F0Predictor()
    rng = np.random.RandomState(3)
    tracks, outs = [], []
    for _ in range(6):
        x = np.abs(rng.randn(50)) * 120 * (rng.rand(50) > 0.45)
        tracks.append(x)
        outs.append(fp._interpolate_f0(fp._resize_f0(x.copy(), 37))[0])
    np.savez_compressed(os.path.join(OUT, "rmvpe_e2e_64.npz"), mel=mel.numpy().astype(np.float32), hidden=hid, f0=f0,
                        tracks=np.array(tracks), resized=np.array(outs))


def f0_fixtures():
    z = np.load(REF + "/infer/modules/vc/lgdsng.npz")
    np.savez_compressed(os.path.join(OUT, "ref_fixtures_f0.npz"), lgdsng_pitch=z["pitch"], lgdsng_pitchf=z["pitchf"],
                        mute_2a_f0=np.load(REF + "/logs/mute/2a_f0/mute.wav.npy"),
                        mute_2b_f0nsf=np.load(REF + "/logs/mute/2b-f0nsf/mute.wav.npy"))


def hubert():
    import re
    from transformers import HubertConfig, HubertModel
    w = OW.hubert_weights(777)
    m = HubertModel(HubertConfig()).eval()
    sd = m.state_dict()
    new = {}
    for k, v in w.items():
        if k.startswith("final_proj"):
            continue
        k = k.replace("feature_extractor.conv_layers.0.2.", "feature_extractor.conv_layers.0.layer_norm.")
        k = re.sub(r"feature_extractor\.conv_layers\.(\d)\.0\.weight", r"feature_extractor.conv_layers.\1.conv.weight", k)
        if k.startswith("layer_norm."):
            k = "feature_projection." + k
        k = k.replace("post_extract_proj.", "feature_projection.projection.")
        k = k.replace("encoder.pos_conv.0.weight_g", "encoder.pos_conv_embed.conv.parametrizations.weight.original0")
        k = k.replace("encoder.pos_conv.0.weight_v", "encoder.pos_conv_embed.conv.parametrizations.weight.original1")
        k = k.replace("encoder.pos_conv.0.bias", "encoder.pos_conv_embed.conv.bias")
        k = k.replace("self_attn.", "attention.").replace("self_attn_layer_norm", "layer_norm")
        k = k.replace("fc1.", "feed_forward.intermediate_dense.").replace("fc2.", "feed_forward.output_dense.")
        assert k in sd and sd[k].shape == v.shape, k
        new[k] = v
    m.load_state_dict(new, strict=False)
    wav = OW.synth_voice(0.5, seed=6)[None]
    hs = m(wav, output_hidden_states=True).hidden_states
    np.savez_compressed(os.path.join(OUT, "hubert_hf_0p5s.npz"), layer9=hs[9][0].numpy(), layer12=hs[12][0].numpy())


def torchgate_inputs(seed, n, n_noise, sr):
    """Seeded test signal shared by this script and tests/: a gliding harmonic tone with an onset + white noise floor."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n_noise) / sr
    tone = sum(torch.sin(2 * math.pi * (180.0 + 40.0 * t) * h * t) / h for h in (1, 2, 3, 5))
    env = ((t * 3.0) % 1.0 < 0.6).float()
    xn = 0.3 * tone * env + 0.02 * torch.randn(n_noise, generator=g)
    return xn[-n:].clone()[None], xn[None]


def torchgate():
    """The reference's OWN TorchGate (infer/modules/gui/torchgate.py) on seeded inputs.  Its module imports rvc.f0.stft, whose
    top-level `from librosa.util import pad_center` is only used by the DirectML STFT class the CPU branch never builds:
    librosa is absent here, so a stub module supplies that one name."""
    import types
    if "librosa" not in sys.modules:
        lib = types.ModuleType("librosa"); util = types.ModuleType("librosa.util")
        util.pad_center = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("stub"))
        lib.util = util
        sys.modules["librosa"] = lib; sys.modules["librosa.util"] = util
    # oracle.weights put the product package (which mirrors the `infer.*` names as a regular package) on sys.path: hide it
    saved_path, saved_mods = sys.path[:], {k: sys.modules.pop(k) for k in list(sys.modules) if k == "infer" or k.startswith("infer.")}
    sys.path[:] = [REF] + [p for p in sys.path if "webui_b200" not in p]
    try:
        from infer.modules.gui.torchgate import TorchGate
    finally:
        sys.path[:] = saved_path
        for k in [k for k in sys.modules if k == "infer" or k.startswith("infer.")]:
            del sys.modules[k]
        sys.modules.update(saved_mods)
    assert TorchGate.forward.__code__.co_filename.startswith(REF)
    out = {}
    # (a) the realtime GUI's instance (gui.py:869-871): sr = 48 kHz, n_fft = 4 * zc = 1920, prop_decrease 0.9, noise reference given
    x, xn = torchgate_inputs(21, 9600, 48000, 48000)
    out["rt_y"] = TorchGate(sr=48000, n_fft=1920, prop_decrease=0.9)(x, xn)[0].numpy()
    out["rt_y_self"] = TorchGate(sr=48000, n_fft=1920, prop_decrease=0.9)(x)[0].numpy()           # xn = None: own statistics
    # (b) class defaults at 16 kHz (n_fft 1024, hop 256), stationary and non-stationary
    x, xn = torchgate_inputs(22, 8192, 32000, 16000)
    out["d16_y"] = TorchGate(sr=16000)(x, xn)[0].numpy()
    out["d16_ns_y"] = TorchGate(sr=16000, nonstationary=True, prop_decrease=0.8)(x)[0].numpy()
    np.savez_compressed(os.path.join(OUT, "torchgate.npz"), **out)


def phase_vocoder():
    """The reference's OWN phase_vocoder (gui.py:27-48).  gui.py cannot be imported (FreeSimpleGUI, sounddevice, ...): the function's
    source is cut out of the file with ast and executed with torch / numpy in scope -- the code that runs is the reference's."""
    import ast
    src = open(REF + "/gui.py").read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "phase_vocoder")
    ns = {"torch": torch, "np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), REF + "/gui.py", "exec"), ns)
    ref_pv = ns["phase_vocoder"]
    g = torch.Generator().manual_seed(77)
    out = {}
    for n in (1920, 1600, 441):                                   # even (48 k / 40 k) and odd (44.1 k: zc = 441) frame lengths
        fade_in = torch.sin(0.5 * np.pi * torch.linspace(0.0, 1.0, steps=n, dtype=torch.float32)) ** 2
        fade_out = 1 - fade_in
        a, b = torch.randn(n, generator=g) * 0.2, torch.randn(n, generator=g) * 0.2
        out[f"a{n}"], out[f"b{n}"], out[f"y{n}"] = a.numpy(), b.numpy(), ref_pv(a, b, fade_out, fade_in).numpy()
    np.savez_compressed(os.path.join(OUT, "phase_vocoder.npz"), **out)


def callback_geometry(sr=24000, block_time=0.16, crossfade_time=0.05, extra_time=0.5):
    """gui.py:783-815 for a small configuration (24 kHz device rate: zc = 240, 3:2 resampler to 16 kHz)."""
    zc = sr // 100
    block = int(np.round(block_time * sr / zc)) * zc
    cross = int(np.round(crossfade_time * sr / zc)) * zc
    extra = int(np.round(extra_time * sr / zc)) * zc
    return dict(sr=sr, zc=zc, block_frame=block, block_frame_16k=160 * block // zc, crossfade_frame=cross,
                sola_buffer_frame=min(cross, 4 * zc), sola_search_frame=zc, extra_frame=extra)


def callback_pieces():
    """Statements of the reference's OWN realtime callback (gui.py GUI.audio_infer), cut out of the file with ast and executed on a
    stand-in ``self``: (a) the input rings + input noise gate + cross-fade + resampling to 16 kHz (gui.py:964-999), with the
    reference's own TorchGate and torchaudio's Resample as ``self.tg`` / ``self.resampler``; (b) the SOLA step (gui.py:1058-1090),
    sin^2 and phase-vocoder cross-fades.  Inputs come from seeds; only the per-block outputs are stored."""
    import ast
    import sys as _sys
    import types
    import torch.nn.functional as F_
    import torchaudio.transforms as tat
    tree = ast.parse(open(REF + "/gui.py").read())
    fn = next(n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name == "audio_infer")
    pv = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "phase_vocoder")
    first = next(i for i, st in enumerate(fn.body) if isinstance(st, ast.Assign) and "self.input_wav[:-self.block_frame]" in ast.unparse(st))
    gate_if = next(i for i, st in enumerate(fn.body) if isinstance(st, ast.If) and "I_noise_reduce" in ast.unparse(st.test))
    sola0 = next(i for i, st in enumerate(fn.body) if isinstance(st, ast.Assign) and ast.unparse(st).startswith("conv_input"))
    sola1 = next(i for i, st in enumerate(fn.body) if isinstance(st, ast.Assign) and ast.unparse(st).startswith("self.sola_buffer[:]"))

    def make(name, args, stmts, ret):
        f = ast.FunctionDef(name=name, args=ast.arguments(posonlyargs=[], args=[ast.arg(arg=a) for a in args], kwonlyargs=[], kw_defaults=[],
                                                          defaults=[]),
                            body=list(stmts) + [ast.parse("return " + ret).body[0]], decorator_list=[])
        return ast.fix_missing_locations(ast.Module(body=[pv, f], type_ignores=[]))
    ns = {"torch": torch, "np": np, "F": F_, "sys": _sys}
    exec(compile(make("ref_pre", ["self", "indata"], fn.body[first:gate_if + 1], "None"), REF + "/gui.py", "exec"), ns)
    exec(compile(make("ref_sola", ["self", "infer_wav"], fn.body[sola0:sola1 + 1], "infer_wav, sola_offset"), REF + "/gui.py", "exec"), ns)
    # the reference's TorchGate (same import trick as torchgate())
    if "librosa" not in sys.modules:
        lib = types.ModuleType("librosa"); util = types.ModuleType("librosa.util")
        util.pad_center = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("stub"))
        lib.util = util
        sys.modules["librosa"] = lib; sys.modules["librosa.util"] = util
    saved_path, saved_mods = sys.path[:], {k: sys.modules.pop(k) for k in list(sys.modules) if k == "infer" or k.startswith("infer.")}
    sys.path[:] = [REF] + [p for p in sys.path if "webui_b200" not in p]
    try:
        from infer.modules.gui.torchgate import TorchGate
    finally:
        sys.path[:] = saved_path
        for k in [k for k in sys.modules if k == "infer" or k.startswith("infer.")]:
            del sys.modules[k]
        sys.modules.update(saved_mods)
    geo = callback_geometry()
    zc, block, sbf = geo["zc"], geo["block_frame"], geo["sola_buffer_frame"]
    n_in = geo["extra_frame"] + geo["crossfade_frame"] + geo["sola_search_frame"] + block
    fade_in = torch.sin(0.5 * np.pi * torch.linspace(0.0, 1.0, steps=sbf, dtype=torch.float32)) ** 2
    out = {}
    me = types.SimpleNamespace(
        **{k: geo[k] for k in ("zc", "block_frame", "block_frame_16k", "sola_buffer_frame", "sola_search_frame")},
        input_wav=torch.zeros(n_in), input_wav_denoise=torch.zeros(n_in), input_wav_res=torch.zeros(160 * n_in // zc),
        nr_buffer=torch.zeros(sbf), fade_in_window=fade_in, fade_out_window=1 - fade_in,
        resampler=tat.Resample(orig_freq=geo["sr"], new_freq=16000, dtype=torch.float32),
        tg=TorchGate(sr=geo["sr"], n_fft=4 * zc, prop_decrease=0.9),
        gui_config=types.SimpleNamespace(I_noise_reduce=True), config=types.SimpleNamespace(device="cpu"))
    g = torch.Generator().manual_seed(91)
    for b in range(3):
        indata = (torch.randn(block, generator=g) * (0.3 if b != 1 else 0.02)).numpy()
        ns["ref_pre"](me, indata)
        out[f"pre_res{b}"] = me.input_wav_res[-geo["block_frame_16k"] - 160:].numpy().copy()
        out[f"pre_den{b}"] = me.input_wav_denoise[-block:].numpy().copy()
        out[f"pre_nr{b}"] = me.nr_buffer.numpy().copy()
    for use_pv in (False, True):
        me = types.SimpleNamespace(**{k: geo[k] for k in ("block_frame", "sola_buffer_frame", "sola_search_frame")},
                                   sola_buffer=torch.zeros(sbf), fade_in_window=fade_in, fade_out_window=1 - fade_in,
                                   gui_config=types.SimpleNamespace(use_pv=use_pv), config=types.SimpleNamespace(device="cpu"))
        g = torch.Generator().manual_seed(92)
        for b in range(3):
            y = torch.randn(block + sbf + geo["sola_search_frame"], generator=g) * 0.2
            w, off = ns["ref_sola"](me, y.clone())
            out[f"sola{int(use_pv)}_{b}"] = w[:block].numpy().copy()
            out[f"sola{int(use_pv)}_off{b}"] = np.int64(int(off))
    np.savez_compressed(os.path.join(OUT, "callback_pieces.npz"), **out)


@one_thread()
def vc_glue():
    """The reference's OWN ``Pipeline.vc`` (infer/modules/vc/pipeline.py:76-184), cut out of the file with ast (the module itself needs
    faiss / librosa to import) and executed with duck-typed components: ``model`` = the oracle HuBERT (so only the glue is under test),
    ``index`` = the oracle IVF-Flat object, ``net_g`` = a recorder that keeps what reaches the synthesizer.  Pins the glue arithmetic of
    rows a3 / a6: retrieval weights and blend, x2 nearest up-sampling, p_len truncation, protect mix, final_proj for v1."""
    import ast
    import types
    from time import time as _time
    import torch.nn.functional as F_
    from oracle import hubert as OH, ivf as OI
    tree = ast.parse(open(REF + "/infer/modules/vc/pipeline.py").read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "Pipeline")
    vc = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "vc")
    ns = {"torch": torch, "np": np, "F": F_, "time": _time}
    exec(compile(ast.fix_missing_locations(ast.Module(body=[vc], type_ignores=[])), REF + "/infer/modules/vc/pipeline.py", "exec"), ns)
    ref_vc = ns["vc"]
    hw = OW.hubert_weights(777)

    class Model:
        def extract_features(self, source, padding_mask, output_layer):
            assert not bool(padding_mask.any())
            return (OH.extract_features(hw, source.float(), output_layer),)

        def final_proj(self, x):
            return OH.final_proj(hw, x)

    class Recorder:
        def infer(self, feats, p_len, sid, pitch=None, pitchf=None):
            self.seen = (feats.clone(), int(p_len[0]), None if pitch is None else pitch.clone(), None if pitchf is None else pitchf.clone())
            return torch.zeros(1, 1, 8)
    me = types.SimpleNamespace(is_half=False, device="cpu", window=160)
    audio0 = OW.synth_voice(0.62, seed=12).numpy().astype(np.float32)            # 9920 samples: 30 HuBERT frames -> 60, p_len 62 -> 60
    idx = OI.build_ivf(OW.index_vectors(500, 768, 3).numpy(), 8, seed=0, exact_assign=True)
    big = idx.reconstruct_n(0, idx.ntotal)
    p_len = audio0.shape[0] // 160
    pitchf = torch.zeros(1, p_len); pitchf[0, 10:40] = 180.0 + torch.arange(30)
    pitch = torch.where(pitchf > 0, torch.full_like(pitchf, 60), torch.ones_like(pitchf)).long()
    out = {}
    rec = Recorder()
    ref_vc(me, Model(), rec, torch.tensor([0]), audio0, pitch, pitchf, [0, 0, 0], idx, big, 0.75, "v2", 0.33)
    out["v2_phone"], out["v2_plen"] = rec.seen[0][0, :, ::32].numpy(), np.int64(rec.seen[1])
    out["v2_pitchf"] = rec.seen[3].numpy()
    rec = Recorder()
    ref_vc(me, Model(), rec, torch.tensor([0]), audio0, pitch, pitchf, [0, 0, 0], None, None, 0.0, "v1", 0.5)
    out["v1_phone"], out["v1_plen"] = rec.seen[0][0, :, ::16].numpy(), np.int64(rec.seen[1])
    np.savez_compressed(os.path.join(OUT, "vc_glue.npz"), **out)


def chunk_stub_vc(audio0, pitch, pitchf, window=160, upp=16):
    """Deterministic stand-in for ``vc`` shared by this generator and the test: one output frame of ``upp`` samples per input frame,
    built from that frame's samples and its pitch values, so any mis-sliced chunk / pitch window / trim shows up in the output."""
    n = audio0.shape[0] // window
    fr = np.asarray(audio0[: n * window], dtype=np.float32).astype(np.float64).reshape(n, window)      # vc casts to float32 first (pipeline.py:91-95)
    v = fr.mean(1) + 0.25 * np.abs(fr).max(1)
    if pitchf is not None:
        m = min(n, pitchf.shape[1])
        v[:m] += 1e-3 * pitchf[0, :m].double().numpy() + 1e-4 * pitch[0, :m].double().numpy()
    return np.repeat(v, upp).astype(np.float32) * np.tile(np.linspace(0.5, 1.0, upp, dtype=np.float32), n)


def pipeline_flow():
    """The reference's OWN ``Pipeline.pipeline`` (pipeline.py:186-366), cut out with ast and run on a stand-in ``self`` whose ``vc`` is
    chunk_stub_vc: silence-point search, per-chunk audio / pitch windows, x_pad trimming, concatenation, peak scaling -- a 10.3 s input
    with x_max = 4 s gives three cut points.  (No index file, resample_sr = 0, rms_mix_rate = 1: those branches need faiss / librosa.)"""
    import ast
    import types
    from time import time as _time
    from scipy import signal
    tree = ast.parse(open(REF + "/infer/modules/vc/pipeline.py").read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "Pipeline")
    fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "pipeline")
    bh, ah = signal.butter(N=5, Wn=48, btype="high", fs=16000)                 # pipeline.py:23
    ns = {"torch": torch, "np": np, "os": os, "signal": signal, "time": _time, "bh": bh, "ah": ah,
          "traceback": __import__("traceback")}
    exec(compile(ast.fix_missing_locations(ast.Module(body=[fn], type_ignores=[])), REF + "/infer/modules/vc/pipeline.py", "exec"), ns)
    sr, tgt_sr, x_pad, x_query, x_center, x_max = 16000, 1600, 1, 1, 3, 4
    me = types.SimpleNamespace(window=160, sr=sr, device="cpu", t_pad=sr * x_pad, t_pad_tgt=tgt_sr * x_pad, t_pad2=sr * x_pad * 2,
                               t_query=sr * x_query, t_center=sr * x_center, t_max=sr * x_max)
    me.vc = lambda model, net_g, sid, audio0, pitch, pitchf, times, index, big_npy, index_rate, version, protect: chunk_stub_vc(audio0, pitch, pitchf)
    audio = OW.synth_voice(10.3, seed=14).numpy().astype(np.float32)
    audio[40000:52000] *= 0.01; audio[90000:100000] *= 0.02                   # quiet stretches for the cut-point search
    p_len = (audio.shape[0] + 2 * me.t_pad) // 160
    pitchf = (100.0 + np.arange(p_len) * 0.37).astype(np.float64)
    pitch = (1 + np.arange(p_len) % 250).astype(np.int64)
    out = ns["pipeline"](me, None, None, 0, audio.copy(), [0, 0, 0], 0, (pitch, pitchf), "", 0.0, 2, 3, tgt_sr, 0, 1.0, "v2", 0.33)
    out0 = ns["pipeline"](me, None, None, 0, audio.copy(), [0, 0, 0], 0, "rmvpe", "", 0.0, 0, 3, tgt_sr, 0, 1.0, "v2", 0.33)   # no-f0 model
    np.savez_compressed(os.path.join(OUT, "pipeline_flow.npz"), out=out[::3].astype(np.float32), n=np.int64(out.shape[0]),
                        total=np.float64(np.abs(out.astype(np.float64)).sum()), out_nof0=out0[::3].astype(np.float32), n_nof0=np.int64(out0.shape[0]))


@one_thread()
def rtrvc_glue():
    """The reference's OWN realtime ``RVC.infer`` (infer/lib/rtrvc.py:134-260), cut out with ast (the module needs fairseq / faiss to
    import) and run on a stand-in ``self``: hubert = the oracle HuBERT, index = the oracle IVF-Flat object, ``_get_f0`` = the oracle RMVPE
    through the reference's own ``_get_f0`` body, net_g = a recorder.  Three consecutive rolling-window blocks pin the glue of row a17:
    last-frame duplication, tail-only retrieval behind the ``(ix >= 0).all()`` guard, the pitch ring roll and ``pitch[3:-1]`` write, x2
    up-sampling, what reaches ``net_g.infer``."""
    import ast
    import types
    import torch.nn.functional as F_
    from typing import Union, Optional, Literal
    from torchaudio.transforms import Resample
    from oracle import hubert as OH, ivf as OI, rmvpe as ORM
    tree = ast.parse(open(REF + "/infer/lib/rtrvc.py").read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "RVC")
    fns = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in ("infer", "_get_f0")]
    ns = {"torch": torch, "np": np, "F": F_, "Union": Union, "Optional": Optional, "Literal": Literal, "Resample": Resample}
    exec(compile(ast.fix_missing_locations(ast.Module(body=fns, type_ignores=[])), REF + "/infer/lib/rtrvc.py", "exec"), ns)
    hw, rw = OW.hubert_weights(777), OW.rmvpe_weights(4321)

    class Model:
        def extract_features(self, source, padding_mask, output_layer):
            return (OH.extract_features(hw, source.float(), output_layer),)

    class Recorder:
        def infer(self, feats, p_len, sid, pitch=None, pitchf=None, skip_head=None, return_length=None, return_length2=None):
            self.seen = dict(phone=feats.clone(), p_len=int(p_len[0]), pitch=pitch.clone(), pitchf=pitchf.clone(),
                             args=(int(skip_head), int(return_length), int(return_length2)))
            return torch.zeros(1, 1, return_length2 * 480)

    class F0Gen:
        def calculate(self, x, p_len, f0_up_key, method, filter_radius):
            assert method == "rmvpe"
            return ORM.calculate(rw, x.numpy(), None, f0_up_key)
    idx = OI.build_ivf(OW.index_vectors(2000, 768, 1).numpy(), None, seed=0, exact_assign=True)
    me = types.SimpleNamespace(is_half=False, device="cpu", version="v2", if_f0=1, hubert=Model(), index=idx,
                               big_npy=idx.reconstruct_n(0, idx.ntotal), index_rate=0.5, window=160, formant_shift=0.0, f0_up_key=0,
                               cache_pitch=torch.zeros(1024, dtype=torch.long), cache_pitchf=torch.zeros(1024, dtype=torch.float32),
                               net_g=Recorder(), tgt_sr=48000, resample_kernel={}, f0_gen=F0Gen())
    me._get_f0 = types.MethodType(ns["_get_f0"], me)
    WIN, BLK, SKIP, RET = 43520, 2560, 250, 21
    stream = OW.synth_voice(2.72 + 0.16 * 3 + 0.1, seed=9)
    out = {}
    for b in range(3):
        ns["infer"](me, stream[b * BLK: b * BLK + WIN].clone(), BLK, SKIP, RET, "rmvpe")
        seen = me.net_g.seen
        out[f"phone{b}"] = seen["phone"][0, :, ::32].numpy()
        out[f"pitch{b}"], out[f"pitchf{b}"] = seen["pitch"].numpy(), seen["pitchf"].numpy()
        out[f"meta{b}"] = np.array([seen["p_len"], *seen["args"]], dtype=np.int64)
    out["ring_pitch"], out["ring_pitchf"] = me.cache_pitch.numpy(), me.cache_pitchf.numpy()
    np.savez_compressed(os.path.join(OUT, "rtrvc_glue.npz"), **out)


def rmvpe_compute_f0():
    """The reference's OWN ``RMVPE.compute_f0 / _mel2hidden / _decode / _to_local_average_cents`` (rvc/f0/rmvpe.py:96-164), cut out with
    ast (the module imports mel.py -> librosa) and attached to a stand-in that inherits the reference's importable ``F0Predictor``
    (``_resize_f0``, ``_interpolate_f0``) and holds the reference's own ``E2E`` network; only the mel front end is the oracle's
    (mel.py needs librosa.filters.mel).  Pins everything of row a8 downstream of the mel: padding to 32 frames, slicing, the
    local-average-cents decode, threshold, resize and gap interpolation."""
    import ast
    import torch.nn.functional as F_
    from typing import Optional, Union
    from oracle import rmvpe as ORM
    tree = ast.parse(open(REF + "/rvc/f0/rmvpe.py").read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "RMVPE")
    want = ("compute_f0", "_mel2hidden", "_decode", "_to_local_average_cents")
    fns = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in want]
    assert len(fns) == len(want)
    ns = {"torch": torch, "np": np, "F": F_, "Optional": Optional, "Union": Union}
    exec(compile(ast.fix_missing_locations(ast.Module(body=fns, type_ignores=[])), REF + "/rvc/f0/rmvpe.py", "exec"), ns)
    Stand = type("Stand", (F0Predictor,), {k: ns[k] for k in want})
    me = Stand(160, 30, 8000, 16000, "cpu")
    me.is_half = False
    me.cents_mapping = np.pad(20 * np.arange(360) + 1997.3794084376191, (4, 4))          # rmvpe.py:62-63
    net = E2E(4, 1, (2, 2)).eval()
    net.load_state_dict(OW.rmvpe_weights(4321))
    me.model = net
    me.mel_extractor = lambda wav, center=True: ORM.log_mel(wav)
    out = {}
    for name, sec, seed in (("a", 1.0, 31), ("b", 0.73, 32)):
        wav = OW.synth_voice(sec, seed=seed).numpy()
        wav[int(0.4 * 16000): int(0.55 * 16000)] *= 1e-4                                   # an unvoiced gap to interpolate across
        out[f"f0_{name}"] = np.asarray(me.compute_f0(wav, None, 0.03), dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "rmvpe_compute_f0.npz"), **out)


def reference_modules(stride=7):
    """The reference's OWN synthesizer classes (rvc/synthesizer.py: the v2/48k f0 model, its realtime skip_head / return_length
    path, the no-f0 family and the v1/48k, v1/32k, v2/32k decoder schedules) and RMVPE network (rvc/f0/e2e.py) on seeded weights,
    inputs and noise, with each model's state-dict key set.  Outputs are stored every ``stride``-th value (7 is coprime with the
    480 / 320 up-sampling and the 360 salience bins); tests/test_oracle_vs_reference.py draws the same inputs in the same order."""
    g = torch.Generator().manual_seed(1)
    T = 60
    phone = torch.randn(1, T, 768, generator=g) * 0.5
    pitchf = torch.zeros(1, T); pitchf[:, 5:50] = 150 + 50 * torch.rand(45, generator=g)
    fm = 1127 * torch.log(1 + pitchf / 700); mn, mx = 1127 * math.log(1 + 50 / 700), 1127 * math.log(1 + 1100 / 700)
    pitch = torch.round(torch.where(fm > 0, (fm - mn) * 254 / (mx - mn) + 1, fm).clamp(1, 255)).long()
    out = {"stride": np.int64(stride)}

    def model(name, cpt):
        net, _ = get_synthesizer({**cpt, "weight": dict(cpt["weight"]), "config": list(cpt["config"])}, "cpu")
        out[name + "_keys"] = np.array(sorted(net.state_dict()))
        return net

    def keep(name, y):
        out[name], out[name + "_shape"] = y.numpy().reshape(-1)[::stride].copy(), np.array(y.shape, dtype=np.int64)
    net_g = model("v2_48k", OW.synth_cpt(77, "v2"))
    torch.manual_seed(5); keep("v2_48k", net_g.infer(phone, torch.tensor([T]), torch.tensor([2]), pitch, pitchf))
    torch.manual_seed(6)
    keep("v2_48k_rt", net_g.infer(phone, torch.tensor([T]), torch.tensor([2]), pitch, pitchf, skip_head=40, return_length=12, return_length2=14))
    net0 = model("nof0", OW.synth_cpt(5, "v2", f0=0))
    torch.manual_seed(3); keep("nof0", net0.infer(phone, torch.tensor([T]), torch.tensor([1])))
    for name, cfgx, ver in (("v1_48k", OW.V1_48K_CONFIG, "v1"), ("v1_32k", OW.V1_32K_CONFIG, "v1"), ("v2_32k", OW.V2_32K_CONFIG, "v2")):
        netx = model(name, OW.synth_cpt(5, ver, config=cfgx))
        Tx = 24; phx = torch.randn(1, Tx, 256 if ver == "v1" else 768, generator=g) * 0.5
        torch.manual_seed(3); keep(name, netx.infer(phx, torch.tensor([Tx]), torch.tensor([1]), pitch[:, :Tx], pitchf[:, :Tx]))
    m = E2E(4, 1, (2, 2)).eval()
    out["e2e_keys"] = np.array(sorted(m.state_dict()))
    m.load_state_dict(OW.rmvpe_weights(9))
    keep("e2e", m(torch.randn(1, 128, 96, generator=g) * 3 - 4))
    np.savez_compressed(os.path.join(OUT, "reference_modules.npz"), **out)


GOLDENS = (synth, rmvpe, f0_fixtures, hubert, torchgate, phase_vocoder, callback_pieces, vc_glue, pipeline_flow, rtrvc_glue,
           rmvpe_compute_f0, reference_modules)

if __name__ == "__main__":
    names = sys.argv[2:] or [fn.__name__ for fn in GOLDENS]
    unknown = set(names) - {fn.__name__ for fn in GOLDENS}
    if unknown:
        sys.exit(f"unknown golden(s) {sorted(unknown)}; choose from {[fn.__name__ for fn in GOLDENS]}")
    for fn in GOLDENS:
        if fn.__name__ in names:
            fn()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
