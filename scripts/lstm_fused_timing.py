"""Per-frame clock64 breakdown of the fused (input projection + recurrence) persistent LSTM kernel (profiling aid).
Stamps per (frame, CTA): 0 barrier passed (h producer), 1 first recurrent stage landed, 2 all MMAs issued,
3 input-part MMAs issued, 4 accumulator ready (cell warps), 5 cell update done.
`python scripts/lstm_fused_timing.py pair`: the same for the two-layer launch (ops.lstm_seq2) at AutoVC's lstm2 shapes,
per tick, against the two one-layer launches it replaces."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from autoformer_b200 import ops, packing


def run(precision, B=512, T=128, H=1024, I=1024):
    torch.manual_seed(0)
    G = ops.choose_gate_group(B, H, True)
    w_hh, w_ih = torch.randn(4 * H, H) * 0.03, torch.randn(4 * H, I) * 0.03
    b = torch.zeros(4 * H)
    hh = packing.pack_lstm_hh(w_hh, precision, G).cuda()
    wih, bias = packing.pack_lstm_ih_fused(w_ih, b, b, precision, G)
    wih, bias = wih.cuda(), bias.cuda()
    x = packing.to_act(torch.randn(B, T, I), precision).cuda()
    m_tiles = (B + 127) // 128
    m_tiles = (m_tiles + 1) // 2 * 2 if m_tiles >= 2 else m_tiles
    grid = m_tiles * (H // G)
    kw = dict(xin=x, w_ih=wih, bias=bias, c_in=I, persistent=True)
    for _ in range(2):
        ops.lstm_seq(None, hh, B, T, H, precision, G, **kw)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); ops.lstm_seq(None, hh, B, T, H, precision, G, **kw); e1.record()
    torch.cuda.synchronize()
    plain = e0.elapsed_time(e1) * 1e3 / T
    dbg = torch.zeros(T * grid * 8, dtype=torch.int64, device="cuda")
    ops.lstm_seq(None, hh, B, T, H, precision, G, debug_clk=dbg, **kw)
    torch.cuda.synchronize()
    d = dbg.view(T, grid, 8).double().cpu()
    step = 2 if m_tiles >= 2 else 1
    lead = d[10:T - 1, 0::step]
    nxt = d[11:T, 0::step]
    f = lambda a: f"{a.mean():.0f}"
    print(f"fused {precision} B={B} H={H} I={I} G={G} grid={grid}: {plain:.2f} us/frame; cycles: "
          f"barrier->first h stage {f(lead[..., 1] - lead[..., 0])}, h mainloop issue {f(lead[..., 2] - lead[..., 1])}, "
          f"issue end->acc ready {f(lead[..., 4] - lead[..., 2])}, cell {f(lead[..., 5] - lead[..., 4])}, "
          f"cell end->next barrier passed {f(nxt[..., 0] - lead[..., 5])} "
          f"(epi_done seen +{f(nxt[..., 6] - lead[..., 5])}, arrival issued +{f(nxt[..., 7] - nxt[..., 6])}, "
          f"all arrived +{f(nxt[..., 0] - nxt[..., 7])}; slowest CTA's arrival {f((nxt[..., 7].max(dim=1).values.unsqueeze(1) - nxt[..., 7]))} after the mean), "
          f"x part issued relative to barrier {f(lead[..., 3] - lead[..., 0])} (negative = hidden), "
          f"frame {f(nxt[..., 0] - lead[..., 0])}")


if __name__ == "__main__" and len(sys.argv) == 1:
    for prec in ("fp32", "bf16", "tf32"):
        run(prec, I=1024)
    run("fp32", I=512)
    run("fp32", H=512, I=320)
    run("fp32", B=32, T=256, H=768, I=80)


def per_cta(precision="fp32", B=512, T=128, H=1024, I=1024):
    """Which CTAs are late at the barrier?  Per leader CTA, mean over frames of: wait at the barrier after its own
    arrival (small = this CTA is among the last), recurrent mainloop, input-part span, cell."""
    torch.manual_seed(0)
    G = ops.choose_gate_group(B, H, True)
    hh = packing.pack_lstm_hh(torch.randn(4 * H, H) * 0.03, precision, G).cuda()
    wih, bias = packing.pack_lstm_ih_fused(torch.randn(4 * H, I) * 0.03, torch.zeros(4 * H), torch.zeros(4 * H), precision, G)
    x = packing.to_act(torch.randn(B, T, I), precision).cuda()
    m_tiles = (B + 127) // 128
    m_tiles = (m_tiles + 1) // 2 * 2 if m_tiles >= 2 else m_tiles
    grid = m_tiles * (H // G)
    kw = dict(xin=x, w_ih=wih.cuda(), bias=bias.cuda(), c_in=I, persistent=True)
    ops.lstm_seq(None, hh, B, T, H, precision, G, **kw)
    dbg = torch.zeros(T * grid * 8, dtype=torch.int64, device="cuda")
    ops.lstm_seq(None, hh, B, T, H, precision, G, debug_clk=dbg, **kw)
    torch.cuda.synchronize()
    d = dbg.view(T, grid, 8).double().cpu()
    cur, nxt = d[10:T - 1], d[11:T]
    wait = (nxt[..., 0] - nxt[..., 7]).mean(0)              # every CTA has an h producer
    hmain = (cur[:, 0::2, 2] - cur[:, 0::2, 1]).mean(0)     # leaders only
    xspan = (nxt[:, 0::2, 3] - cur[:, 0::2, 2]).mean(0)
    cell = (cur[:, 0::2, 5] - cur[:, 0::2, 4]).mean(0)
    first = (cur[:, 0::2, 1] - cur[:, 0::2, 0]).mean(0)
    print(f"per-CTA {precision} H={H} I={I}: barrier wait after own arrival, all {grid} CTAs sorted:")
    print(" ", [int(v) for v in wait.sort().values.tolist()])
    order = wait[0::2].argsort()
    print("  leaders sorted by wait: (pair, wait, barrier->first h, h mainloop, x span, cell)")
    for i in order.tolist()[:6] + order.tolist()[-6:]:
        print(f"   pair {i:3d} wait {wait[2 * i]:6.0f} first {first[i]:6.0f} hmain {hmain[i]:6.0f} xspan {xspan[i]:6.0f} cell {cell[i]:6.0f}")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "cta":
    per_cta(I=1024)
    per_cta(I=512)


def run_pair(precision="fp16x2", B=512, T=128, H=1024, I=512):
    """Two-layer launch: time per tick against two one-layer launches, and the tick's stamps (avc_lstm_seq2: 0 barrier
    passed, 1 first rec0 stage landed, 2 / 3 rec0 / rec1 issued, 4 / 5 layer 0 accumulator ready / cell done, 6 / 7
    layer 1, 8 cell warps done seen, 9 arrival issued, 10 / 11 in0 / in1 issued)."""
    torch.manual_seed(0)
    G = ops.choose_gate_group(B, H, True)
    packs = []
    for k in (I, H):
        hh = packing.pack_lstm_hh(torch.randn(4 * H, H) * 0.03, precision, G).cuda()
        wih, bias = packing.pack_lstm_ih_fused(torch.randn(4 * H, k) * 0.03, torch.zeros(4 * H), torch.zeros(4 * H),
                                               precision, G)
        packs.append((hh, wih.cuda(), bias.cuda()))
    x = packing.to_act(torch.randn(B, T, I), precision).cuda()
    (hh0, wih0, b0), (hh1, wih1, b1) = packs
    m_tiles = (B + 127) // 128
    m_tiles = (m_tiles + 1) // 2 * 2 if m_tiles >= 2 else m_tiles
    grid = m_tiles * (H // G)

    def two():
        h = ops.lstm_seq(None, hh0, B, T, H, precision, G, persistent=True, xin=x, w_ih=wih0, bias=b0, c_in=I)
        ops.lstm_seq(None, hh1, B, T, H, precision, G, persistent=True, xin=h, w_ih=wih1, bias=b1, c_in=H)

    def pair(dbg=None):
        ops.lstm_seq2((hh0, hh1), B, T, H, precision, G, x, (wih0, wih1), (b0, b1), I, debug_clk=dbg)

    def timed(fn, n=5):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    t_two, t_pair = timed(two), timed(pair)
    dbg = torch.zeros((T + 2) * grid * 12, dtype=torch.int64, device="cuda")
    pair(dbg)
    torch.cuda.synchronize()
    d = dbg.view(T + 2, grid, 12).double().cpu()
    cur, nxt = d[10:T - 1, 0::2 if m_tiles >= 2 else 1], d[11:T, 0::2 if m_tiles >= 2 else 1]
    f = lambda a: f"{a.mean():.0f}"
    print(f"pair {precision} B={B} T={T} H={H} I={I} G={G} grid={grid}: two launches {t_two:.3f} ms, one launch "
          f"{t_pair:.3f} ms ({t_pair * 1e3 / (T + 2):.2f} us/tick); cycles from barrier passed: first h stage "
          f"{f(cur[..., 1] - cur[..., 0])}, rec0 issued {f(cur[..., 2] - cur[..., 0])}, rec1 issued "
          f"{f(cur[..., 3] - cur[..., 0])}, acc0 ready {f(cur[..., 4] - cur[..., 0])}, cell0 done "
          f"{f(cur[..., 5] - cur[..., 0])}, acc1 ready {f(cur[..., 6] - cur[..., 0])}, cell1 done "
          f"{f(cur[..., 7] - cur[..., 0])}, in0 issued {f(cur[..., 10] - cur[..., 0])}, in1 issued "
          f"{f(cur[..., 11] - cur[..., 0])}, cells done seen {f(nxt[..., 8] - cur[..., 0])}, arrival "
          f"{f(nxt[..., 9] - cur[..., 0])}, next barrier passed (tick) {f(nxt[..., 0] - cur[..., 0])}")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "pair":
    run_pair("fp16x2")
    run_pair("fp32")
