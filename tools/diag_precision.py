import os, sys, numpy as np, torch
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, "tests"))
from common import make_model, load_golden, si_sdr_db, rel_err
from oracle import synth
for tag in ("crn_small","crn_teacher","crn_student"):
    g = load_golden(tag)
    for prec in ("tf32","fp16"):
        m = make_model(tag, prec)
        out = m.forward(torch.from_numpy(g["spec_chunk1"]).cuda()); out = out[0] if isinstance(out, tuple) else out
        B, L = int(g["meta"][1]), int(g["meta"][2])
        mix,_ = synth.make_mixture(B, L)
        y = m.realtime_process(torch.from_numpy(mix).cuda()); y = (y[0] if isinstance(y, tuple) else y).cpu().numpy()
        print(tag, prec, "fwd rel", rel_err(out.cpu().numpy(), g["fwd_chunk1"]), "wave max_abs", float(np.abs(y-g["out"]).max()), "peak", float(np.abs(g["out"]).max()), "sisdr", si_sdr_db(y, g["out"]))
