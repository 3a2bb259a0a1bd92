"""One forward of a named workload inside a cudaProfilerStart/Stop range, for `ncu --profile-from-start off`:

    ncu --set full --clock-control none --import-source on --profile-from-start off -o gpurun_out/r02_melgan \
        python scripts/ncu_families.py melgan

Workloads (sizes of the bench's sub-records where ncu's ~40 replays per launch stay affordable):
  autovc   AutoVC(32,256,512,32) 512 x 128 frames, fp16x2 (BASELINE configs[1]; persistent LSTM kernels launched without
           the cooperative attribute, which ncu cannot replay -- AVC_LSTM_NO_COOP=1, same kernels)
  melgan   Generator(80,32,3) on B = 32 x 1000 frames (the vocoder of configs[3])
  lstmdv   LstmDV on B = 64 x 256 frames, fp16x2 (the weight-stationary small-batch recurrence)
  meta     MetaPool(44,256,512,22) on B = 128 x 176 frames, fp16x2 (every Meta / mixer kernel family)
"""
import os
import sys
import warnings

os.environ.setdefault("AVC_LSTM_NO_COOP", "1")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")
import torch

from oracle import templates
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker


def build(what):
    if what == "autovc":
        from autoformer_b200.factory.AutoVC import AutoVC
        args = (32, 256, 512, 32)
        m = AutoVC(*args)
        m.load_state_dict(seeded_state_dict(templates.autovc_template(*args), 0))
        m = m.cuda().eval()
        m.precision = os.environ.get("AVC_NCU_PRECISION", "fp16x2")
        B, T = 512, 128
        x, co, ct = synthetic_mel(B, T, 1).cuda(), synthetic_speaker(B, 1, "org").cuda(), synthetic_speaker(B, 1, "trg").cuda()
        return lambda: m(x, co, ct)
    if what == "melgan":
        from autoformer_b200.melgan.modules import Generator
        g = Generator(80, 32, 3)
        g.load_state_dict(seeded_state_dict(templates.melgan_template(), 4))
        g = g.cuda().eval()
        g.precision = os.environ.get("AVC_NCU_PRECISION", "fp32")
        B, T = int(os.environ.get("AVC_NCU_B", 32)), 1000
        mel = synthetic_mel(B, T, 2).transpose(1, 2).contiguous().cuda()
        return lambda: g(mel)
    if what == "lstmdv":
        from autoformer_b200.factory.LstmDV import LstmDV
        m = LstmDV()
        m.load_state_dict(seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5))
        m = m.cuda().eval()
        m.precision = os.environ.get("AVC_NCU_PRECISION", "fp16x2")
        x = synthetic_mel(64, 256, 3).cuda()
        return lambda: m(x)
    if what == "meta":
        from autoformer_b200.factory.MetaPool import MetaPool
        args = (44, 256, 512, 22)
        m = MetaPool(*args)
        m.load_state_dict(seeded_state_dict(templates.meta_template("pool", *args), 6))
        m = m.cuda().eval()
        m.precision = os.environ.get("AVC_NCU_PRECISION", "fp16x2")
        B = int(os.environ.get("AVC_NCU_B", 128))
        x, co, ct = synthetic_mel(B, 176, 4).cuda(), synthetic_speaker(B, 4, "org").cuda(), synthetic_speaker(B, 4, "trg").cuda()
        return lambda: m(x, co, ct)
    if what == "misc":
        # the small kernels no other workload launches: gn_apply (MetaConv), global_stats / adain (AdaIN "2" variants),
        # audio_frames / complex_mag (Audio2Mel), resblock_kernel (MelGAN in the split format), lstm_step_kernel
        # (un-fused input projection, one launch per frame: LstmLayer.use_fused picks it for the decoder's lstm2 at B = 8)
        from autoformer_b200.factory.AutoVC import AutoVC
        from autoformer_b200.factory.AutoVC2 import AutoVC2
        from autoformer_b200.factory.MetaConv import MetaConv
        from autoformer_b200.melgan.modules import Audio2Mel, Generator
        margs = (44, 256, 512, 22)
        mc = MetaConv(*margs)
        mc.load_state_dict(seeded_state_dict(templates.meta_template("conv", *margs), 7))
        mc = mc.cuda().eval()
        xm, com, ctm = synthetic_mel(8, 176, 4).cuda(), synthetic_speaker(8, 4, "org").cuda(), synthetic_speaker(8, 4, "trg").cuda()
        args = (32, 256, 512, 32)
        a2 = AutoVC2(*args)
        a2.load_state_dict(seeded_state_dict(templates.autovc2_template(*args), 16))
        a2 = a2.cuda().eval()
        av = AutoVC(*args)
        av.load_state_dict(seeded_state_dict(templates.autovc_template(*args), 0))
        av = av.cuda().eval()
        av.persistent_lstm = False
        xa, coa, cta = synthetic_mel(64, 64, 1).cuda(), synthetic_speaker(64, 1, "org").cuda(), synthetic_speaker(64, 1, "trg").cuda()
        fft = Audio2Mel().cuda()
        audio = torch.randn(8, 22050, device="cuda") * 0.1
        g = Generator(80, 32, 3)
        g.load_state_dict(seeded_state_dict(templates.melgan_template(), 4))
        g = g.cuda().eval()
        mel = synthetic_mel(4, 256, 2).transpose(1, 2).contiguous().cuda()

        def run():
            mc(xm, com, ctm)
            a2(xa, coa, cta)
            av(xa[:8, :32].contiguous(), coa[:8], cta[:8])       # per-frame lstm_step launches (un-fused projection)
            fft(audio)
            g(mel)
        run.models = (mc, a2, av, fft, g)
        return run
    raise SystemExit(f"unknown workload {what}")


if __name__ == "__main__":
    fn = build(sys.argv[1])
    fn()
    fn()
    # serving mode: no per-forward weight digest inside the profiled range
    for m in list(getattr(fn, "models", ())) + [c.cell_contents for c in (fn.__closure__ or [])]:
        if hasattr(m, "freeze_weights"):
            m.freeze_weights()
    fn()
    torch.cuda.synchronize()
    torch.cuda.profiler.start()
    fn()
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    print("done", sys.argv[1])
