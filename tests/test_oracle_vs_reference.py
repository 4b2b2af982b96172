"""CPU: the oracle against the outputs of the reference's own modules -- its synthesizer classes and RMVPE network -- stored in
tests/golden/reference_modules.npz by tests/golden/make_golden.py::reference_modules (every stride-th output value, the full
shapes and each model's state-dict key set).  Inputs and noise are re-drawn here from the same seeds in the same order."""
import math
import os

import numpy as np
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_oracle_matches_reference_modules():
    from oracle import rmvpe as ORM, synth as OS, weights as OW
    z = np.load(os.path.join(G, "reference_modules.npz"))
    stride = int(z["stride"])

    def same(name, out, tol):
        assert tuple(out.shape) == tuple(z[name + "_shape"]), name
        err = np.abs(out.numpy().reshape(-1)[::stride] - z[name]).max()
        assert err < tol, (name, err)

    with torch.no_grad():
        cpt = OW.synth_cpt(77, "v2")
        w = OW.synth_weights(77)
        assert set(w) == set(z["v2_48k_keys"].tolist())
        T = 60
        g = torch.Generator().manual_seed(1)
        phone = torch.randn(1, T, 768, generator=g) * 0.5
        pitchf = torch.zeros(1, T); pitchf[:, 5:50] = 150 + 50 * torch.rand(45, generator=g)
        fm = 1127 * torch.log(1 + pitchf / 700); mn, mx = 1127 * math.log(1 + 50 / 700), 1127 * math.log(1 + 1100 / 700)
        pitch = torch.round(torch.where(fm > 0, (fm - mn) * 254 / (mx - mn) + 1, fm).clamp(1, 255)).long()
        torch.manual_seed(5); n1 = torch.randn(1, 192, T); torch.rand(1, 1, 1); n2 = torch.randn(1, T * 480, 1)
        same("v2_48k", OS.synth_infer(w, cpt["config"], phone, torch.tensor([T]), torch.tensor([2]), pitch, pitchf, n1, n2), 5e-6)
        torch.manual_seed(6); n1 = torch.randn(1, 192, T - 16); torch.rand(1, 1, 1); n2 = torch.randn(1, 12 * 480, 1)
        same("v2_48k_rt", OS.synth_infer(w, cpt["config"], phone, torch.tensor([T]), torch.tensor([2]), pitch, pitchf, n1, n2, 40, 12, 14), 5e-6)
        # no-f0 family (SynthesizerTrnMs768NSFsid_nono: no emb_pitch, plain Generator decoder)
        cpt0 = OW.synth_cpt(5, "v2", f0=0)
        w0 = OW.synth_weights(5, use_f0=False)
        assert set(w0) == set(z["nof0_keys"].tolist())
        torch.manual_seed(3); n1 = torch.randn(1, 192, T)
        same("nof0", OS.synth_infer(w0, cpt0["config"], phone, torch.tensor([T]), torch.tensor([1]), None, None, n1, None), 5e-6)
        # the other decoder schedules of configs/{v1,v2}/*.json (5-stage decoders, kernel 16 at stride 4 / 6)
        for name, cfgx, ver in (("v1_48k", OW.V1_48K_CONFIG, "v1"), ("v1_32k", OW.V1_32K_CONFIG, "v1"), ("v2_32k", OW.V2_32K_CONFIG, "v2")):
            cptx = OW.synth_cpt(5, ver, config=cfgx)
            encx = 256 if ver == "v1" else 768
            wx = OW.synth_weights(5, cfgx, encx)
            assert set(wx) == set(z[name + "_keys"].tolist()), name
            Tx = 24; phx = torch.randn(1, Tx, encx, generator=g) * 0.5
            torch.manual_seed(3); n1 = torch.randn(1, 192, Tx); torch.rand(1, 1, 1); n2 = torch.randn(1, Tx * (cfgx[-1] // 100), 1)
            same(name, OS.synth_infer(wx, cptx["config"], phx, torch.tensor([Tx]), torch.tensor([1]), pitch[:, :Tx], pitchf[:, :Tx], n1, n2), 5e-6)
        rw = OW.rmvpe_weights(9)
        assert set(rw) == set(z["e2e_keys"].tolist())
        mel = torch.randn(1, 128, 96, generator=g) * 3 - 4
        same("e2e", ORM.e2e_forward(rw, mel), 1e-5)
