"""Development aid: runs each GPU check in its own process (a trapping kernel poisons its CUDA context) and prints
compact results.  Usage on the GPU box:  python scripts/gpu_diag.py [check ...]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def check_umma():
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    torch.manual_seed(0)
    a = (torch.randn(136, 64, device="cuda")).to(torch.bfloat16).contiguous()
    b = (torch.randn(64, 64, device="cuda")).to(torch.bfloat16).contiguous()
    for mode in (0, 2):
        for shift in (0, 1, 2, 3, 8):
            d = torch.zeros(128, 64, device="cuda")
            rc = lib.psgla_selftest_umma(a.data_ptr(), b.data_ptr(), d.data_ptr(), shift, mode, None)
            torch.cuda.synchronize()
            ref = a[shift:shift + 128].float() @ b.float().t()
            print("umma mode=%d shift=%d rc=%d maxerr=%.4g (ref max %.3g)" % (mode, shift, rc, (d - ref).abs().max().item(),
                                                                            ref.abs().max().item()), flush=True)


def _conv_case(B, H, W, layer, depth=20, seed=0):
    import torch
    import torch.nn.functional as F
    import psgla_b200 as P
    lib = P._lib.lib()
    sd = P.random_dncnn_state_dict(seed, depth, scale=3.0)
    den = P.DnCNN(depth=depth, pretrained=sd)
    names = ["in_conv"] + ["conv_list.%d" % i for i in range(depth - 2)] + ["out_conv"]
    w = sd[names[layer] + ".weight"].cuda()
    bias = sd[names[layer] + ".bias"].cuda()
    cin = w.shape[1]
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, cin, H, W, device="cuda", generator=g)
    xb = x.to(torch.bfloat16)
    cpad = 16 if layer == 0 else 64
    xin = torch.zeros(B, H, W, cpad, device="cuda", dtype=torch.bfloat16)
    xin[..., :cin] = xb.permute(0, 2, 3, 1)
    xin = xin.contiguous()
    shape = P._lib.ImgShape(B, 3, H, W)
    ref = F.conv2d(xb.float(), w.to(torch.bfloat16).float(), bias, padding=1)
    if layer == depth - 1:
        out = torch.full((B, 3, H, W), float("nan"), device="cuda")
        rc = lib.psgla_conv3x3_layer(den.packed.data_ptr(), depth, layer, shape, xin.data_ptr(), out.data_ptr(), 0, None)
        torch.cuda.synchronize()
        got = out
    else:
        out = torch.full((B, H, W, 64), float("nan"), device="cuda", dtype=torch.bfloat16)
        rc = lib.psgla_conv3x3_layer(den.packed.data_ptr(), depth, layer, shape, xin.data_ptr(), out.data_ptr(), 1, None)
        torch.cuda.synchronize()
        got = out.float().permute(0, 3, 1, 2)
        ref = ref.relu()
    err = (got - ref).abs()
    print("conv layer=%d B=%d H=%d W=%d rc=%d maxerr=%.4g meanerr=%.4g refmax=%.3g nan=%d" % (
        layer, B, H, W, rc, err.nan_to_num(1e9).max().item(), err.nan_to_num(0).mean().item(), ref.abs().max().item(),
        int(torch.isnan(got).sum().item())), flush=True)
    if err.nan_to_num(1e9).max().item() > 0.1:
        bad = (err.nan_to_num(1e9) > 0.1).nonzero()
        print("   first bad idx:", bad[:4].tolist(), " n_bad=", bad.shape[0], flush=True)


def check_conv_mid():
    _conv_case(1, 8, 128, 1)
    _conv_case(2, 40, 256, 5)
    _conv_case(1, 33, 200, 3)


def check_conv_first():
    _conv_case(1, 8, 128, 0)
    _conv_case(2, 37, 150, 0)


def check_conv_last():
    _conv_case(1, 8, 128, 19)
    _conv_case(2, 37, 150, 19)


def check_dncnn():
    import torch
    import psgla_b200 as P
    from oracle import image_oracle as io_
    sd = io_.make_dncnn_weights(seed=0, n_power_iter=10, spatial=16)
    den = P.DnCNN(pretrained=sd)
    net = io_.DnCNN().cuda()
    net.load_state_dict(sd)
    x = torch.rand(2, 3, 64, 96, device="cuda")
    with torch.no_grad():
        ref = net(x)
    got = den.forward(x)
    torch.cuda.synchronize()
    r_ref, r_got = ref - x, got - x
    print("dncnn full: max|D-Dref|=%.4g  |R|max=%.4g  rel residual err=%.4g" % (
        (got - ref).abs().max().item(), r_ref.abs().max().item(), ((r_got - r_ref).norm() / r_ref.norm()).item()), flush=True)


def check_gmm():
    import numpy as np
    import psgla_b200 as P
    from oracle import gmm2d_oracle as o
    for name in o.PRIOR_NAMES:
        mu, Sig, pi = o.gaussian_mixt_example(name)
        D = P.Theorical_MMSE(mu, Sig, pi)
        Do = o.theorical_mmse(mu, Sig, pi)
        y = np.array([0.0, -2.0])
        rng = np.random.default_rng(0)
        noise = rng.standard_normal((299, 2))
        Xo = o.snopnp_ula(300, y, y, 0.3, np.eye(2), 1, Do, 2 / 3, noise=noise)
        X64 = P.SnoPnP_ULA(300, y, y, 0.3, np.eye(2), 1, D, 2 / 3, noise=noise)
        X32 = P.SnoPnP_ULA(300, y, y, 0.3, np.eye(2), 1, D, 2 / 3, noise=noise, dtype="float32")
        print("gmm psgla %-22s fp64 err %.3g  fp32 err %.3g" % (name, np.abs(X64 - Xo).max(), np.abs(X32 - Xo).max()), flush=True)
        Xo = o.pnp_ula(300, y, y, 0.1, np.eye(2), 1, Do, 0.5, 1.5, noise=noise)
        X64 = P.PnP_ULA(300, y, y, 0.1, np.eye(2), 1, D, 0.5, 1.5, noise=noise)
        X32 = P.PnP_ULA(300, y, y, 0.1, np.eye(2), 1, D, 0.5, 1.5, noise=noise, dtype="float32")
        print("gmm ula   %-22s fp64 err %.3g  fp32 err %.3g" % (name, np.abs(X64 - Xo).max(), np.abs(X32 - Xo).max()), flush=True)


def check_gmm_speed():
    import time
    import numpy as np
    import torch
    import psgla_b200 as P
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    D = P.Theorical_MMSE(mu, Sig, pi)
    for alg, args in (("psgla", dict(delta=0.3, alpha=2 / 3)), ("pnp_ula", dict(delta=0.1, alpha=1.5, epsilon=0.5))):
        for nc in (1 << 20, 1000000, 148 * 2048 * 4):
            ch = P.GMMChains(alg, np.array([0.0, -2.0]), A=np.eye(2), sigma=1, denoiser=D, n_chains=nc, **args)
            ch.run(100)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ch.run(2000)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            print("gmm speed %s chains=%d: %.3f ms for 2000 steps -> %.3e chain-steps/s" % (alg, nc, ms, nc * 2000 / ms * 1e3), flush=True)


def check_iter_breakdown():
    """Where one PSGLA image iteration spends its time: per-kernel CUDA-event timings, with and without an L2 flush."""
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    B, H, W = int(os.environ.get("DIAG_B", "32")), 256, 256
    dev = torch.device("cuda")
    den = P.DnCNN(pretrained=P.random_dncnn_state_dict(0, scale=0.5), device=dev)
    im = torch.rand(1, 3, H, W, device=dev)
    dg, init, y, mask = P.make_inpainting(im, 0.5, 1.0, 0)
    s = 2 / 255
    run = P.psgla_run(init, dg, den, 1.0, 5.0, s, s * s, n_iter=1000, n_inter=10, n_inter_mmse=10, seed=0, n_chains=B)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    shape = P._lib.ImgShape(B, 3, H, W)
    ws, den_in = den.buffers(shape)
    half = (B * H * W * 64 * 2 + 1023) // 1024 * 1024
    bufs = [ws.data_ptr(), ws.data_ptr() + half]
    out = torch.empty(B, 3, H, W, device=dev)

    def timed(fn, reps=10, do_flush=False):
        fn()
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(reps):
            if do_flush:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / reps * 1e3

    it = [0]

    def step():
        run.step(it[0])
        it[0] += 1

    print("B=%d step            : %8.1f us   (with L2 flush %8.1f us)" % (B, timed(step), timed(step, do_flush=True)), flush=True)
    print("pre                  : %8.1f us" % timed(lambda: run.pre(0, run.pre_params)), flush=True)
    conv = lambda l, i, o: P._lib.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), 20, l, shape, i, o, 1, None), "conv")
    print("layer 0 (3->64, SS)  : %8.1f us" % timed(lambda: conv(0, den_in.data_ptr(), bufs[0])), flush=True)
    print("layer 5 (64->64)     : %8.1f us   (flush %8.1f us)" % (timed(lambda: conv(5, bufs[0], bufs[1])),
                                                                   timed(lambda: conv(5, bufs[0], bufs[1]), do_flush=True)), flush=True)
    print("layer 19 (64->3 raw) : %8.1f us" % timed(lambda: conv(19, bufs[1], out.data_ptr())), flush=True)
    post = P._lib.PostParams(1.0, 1.0, 0.5, 0.5)
    print("dncnn+post (20 conv) : %8.1f us" % timed(lambda: den.residual_post(shape, den_in, run.base, post, run.X, None, run.mean, run.mean2)), flush=True)

    def hidden18():
        for l in range(1, 19):
            conv(l, bufs[l & 1], bufs[(l + 1) & 1])
    print("18 hidden layers     : %8.1f us" % timed(hidden18), flush=True)


def check_step_series():
    """Per-iteration device time of the first 80 PSGLA iterations after start-up (clock / power ramp effects)."""
    import subprocess as sp
    import torch
    import psgla_b200 as P
    B, H, W = int(os.environ.get("DIAG_B", "32")), 256, 256
    dev = torch.device("cuda")
    den = P.DnCNN(pretrained=P.random_dncnn_state_dict(0, scale=0.5), device=dev)
    im = torch.rand(1, 3, H, W, device=dev)
    dg, init, y, mask = P.make_inpainting(im, 0.5, 1.0, 0)
    s = 2 / 255
    run = P.psgla_run(init, dg, den, 1.0, 5.0, s, s * s, n_iter=1000, n_inter=10, n_inter_mmse=10, seed=0, n_chains=B)
    torch.cuda.synchronize()
    smi = sp.Popen(["nvidia-smi", "--query-gpu=clocks.sm,power.draw,clocks_event_reasons.sw_power_cap", "--format=csv,noheader",
                    "-lms", "20"], stdout=sp.PIPE, text=True)
    ev = []
    for i in range(80):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run.step(i)
        e1.record()
        ev.append((e0, e1))
    torch.cuda.synchronize()
    import time
    time.sleep(0.1)
    smi.terminate()
    ms = [a.elapsed_time(b) for a, b in ev]
    print("step ms:", " ".join("%.2f" % m for m in ms), flush=True)
    print("clocks:", " | ".join(l.strip() for l in smi.stdout.read().splitlines()[:40]), flush=True)


def check_drunet_breakdown():
    """DRUNet: time per stage (CUDA events) and whole PSGLA iteration, 256x256 (or DIAG_HW=HxW), DIAG_B chains."""
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    B = int(os.environ.get("DIAG_B", "16"))
    H, W = [int(v) for v in os.environ.get("DIAG_HW", "256x256").split("x")]
    dev = torch.device("cuda")
    den = P.DRUNet(pretrained=P.random_drunet_state_dict(0), device=dev)
    im = torch.rand(1, 3, H, W, device=dev)
    dg, init, y, mask = P.make_inpainting(im, 0.5, 1.0, 0)
    s = 5 / 255
    run = P.psgla_run(init, dg, den, 1.0, 25.0, s, s * s, n_iter=1000, n_inter=10, n_inter_mmse=10, seed=0, n_chains=B)

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e3

    it = [0]

    def step():
        run.step(it[0])
        it[0] += 1
    for _ in range(5):
        step()
    t_step = timed(step, 10)
    flop = 4235136.0 * B * H * W
    print("DRUNet B=%d %dx%d  PSGLA iteration %.1f us -> %.1f image-it/s, %.1f TFLOP/s" % (B, H, W, t_step, B / t_step * 1e6, flop / t_step / 1e6), flush=True)
    # individual general layers
    def layer(mode, h, w, cin, cout, res):
        wt = torch.zeros(9 * cout * cin, device=dev, dtype=torch.bfloat16)
        ho, wo = {0: (h, w), 1: (h // 2, w // 2), 2: (2 * h, 2 * w)}[mode]
        x = torch.zeros(B * h * w * cin, device=dev, dtype=torch.bfloat16)
        o = torch.zeros(B * ho * wo * cout, device=dev, dtype=torch.bfloat16)
        r = torch.zeros_like(o) if res else None
        f = lambda: P._lib.check(lib.psgla_convg_layer(mode, B, h, w, cin, cout, wt.data_ptr(), x.data_ptr(),
                                                      r.data_ptr() if res else None, None, o.data_ptr(), 0, None), "convg")
        t = timed(f, 10)
        taps = {0: 9, 1: 4, 2: 4}[mode]
        npx = B * (ho * wo if mode != 2 else h * w)
        fl = 2.0 * taps * cin * cout * npx
        print("  mode %d %4dx%-4d %3d->%3d res=%d : %7.1f us  %.0f TFLOP/s" % (mode, h, w, cin, cout, res, t, fl / t / 1e6), flush=True)
    for sc, c in ((1, 128), (2, 256), (3, 512)):
        layer(0, H >> sc, W >> sc, c, c, 0)
        layer(0, H >> sc, W >> sc, c, c, 1)
    for sc, c in ((0, 64), (1, 128), (2, 256)):
        layer(1, H >> sc, W >> sc, c, 2 * c, 0)
        layer(2, H >> (sc + 1), W >> (sc + 1), 2 * c, c, 0)


def check_host_overhead():
    """Single chain (the reference's shape of run): host enqueue time per iteration vs device time per iteration."""
    import time
    import torch
    import psgla_b200 as P
    dev = torch.device("cuda")
    den = P.DnCNN(pretrained=P.random_dncnn_state_dict(0, scale=0.5), device=dev)
    im = torch.rand(1, 3, 256, 256, device=dev)
    s = 2 / 255
    for name, (dg, init) in (("inpaint", P.make_inpainting(im, 0.5, 1.0, 0)[:2]), ("deblur", P.make_deblurring(im, 4, "uniform")[:2])):
        run = P.psgla_run(init, dg, den, 1.0, 5.0, s, s * s, n_iter=2000, n_inter=10, n_inter_mmse=10, seed=0, n_chains=1)
        for i in range(30):
            run.step(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(30, 70):  # 40 x 21 launches stay below the driver's launch queue depth: pure host cost
            run.step(i)
        t_host = (time.perf_counter() - t0) / 40 * 1e6
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(70, 370):
            run.step(i)
        e1.record()
        torch.cuda.synchronize()
        print("single chain %-8s host enqueue %.1f us/iteration, device %.1f us/iteration" % (name, t_host, e0.elapsed_time(e1) / 300 * 1e3), flush=True)
        pre_t = []
        for _ in range(3):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                run.pre(0, run.pre_params)
            e1.record()
            torch.cuda.synchronize()
            pre_t.append(e0.elapsed_time(e1) / 20 * 1e3)
        print("   pre kernel alone: %.1f us" % min(pre_t), flush=True)
    B = 32
    dg, init, y = P.make_deblurring(im, 4, "uniform")
    run = P.psgla_run(init, dg, den, 1.0, 5.0, s, s * s, n_iter=100, n_inter=10, n_inter_mmse=10, seed=0, n_chains=B)
    run.pre(0, run.pre_params)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        run.pre(0, run.pre_params)
    e1.record()
    torch.cuda.synchronize()
    print("deblur pre kernel B=32: %.1f us" % (e0.elapsed_time(e1) / 10 * 1e3), flush=True)


def check_mma_rate():
    """Cycles per tcgen05.mma (M128 x N x K16 bf16) for SS / shifted-SS / TS operand sources, one CTA and all SMs."""
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    iters = 2000
    for grid in (148,):
        out = torch.zeros(grid, dtype=torch.int64, device="cuda")
        for mode, name in ((0, "SS"), (1, "SS+128B"), (2, "TS"), (3, "TS alt-D"), (4, "SS alt-D")):
            row = []
            for n in ((16, 32, 64, 96, 128, 192, 256) if mode < 3 else (16, 32, 64, 96, 128)):
                P._lib.check(lib.psgla_selftest_mma_rate(mode, n, iters, grid, out.data_ptr(), None), "mma_rate")
                torch.cuda.synchronize()
                row.append("N=%d: %.1f" % (n, out.double().mean().item() / (iters * 4)))
            print("mma_rate grid=%d %-8s cycles/MMA  %s" % (grid, name, "  ".join(row)), flush=True)


def check_mma_pattern():
    """The conv kernel's MMA issue pattern alone (no loaders, no epilogue, no TMA): cycles per MMA."""
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    out = torch.zeros(148, dtype=torch.int64, device="cuda")
    for mode, name in ((2, "TS same operands"), (5, "conv pattern, commit per row"), (6, "conv pattern, no commits"), (7, "conv pattern, A fixed slot")):
        for n in (64, 16):
            iters = 500
            P._lib.check(lib.psgla_selftest_mma_rate(mode, n, iters, 148, out.data_ptr(), None), "mma_rate")
            torch.cuda.synchronize()
            per = out.double().mean().item() / (iters * (4 if mode < 5 else 36))
            print("mma_pattern %-32s N=%d: %.1f cycles/MMA" % (name, n, per), flush=True)


def check_mma_rate2():
    """cycles per M256 x N x K16 MMA of a CTA pair (cta_group::2)."""
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    for pairs in (1, 74):
        out = torch.zeros(pairs, dtype=torch.int64, device="cuda")
        for mode, name in ((0, "TS"), (1, "SS")):
            row = []
            for n in (32, 64, 128, 256):
                iters = 500
                P._lib.check(lib.psgla_selftest_mma_rate2(mode, n, iters, pairs, out.data_ptr(), None), "mma_rate2")
                torch.cuda.synchronize()
                row.append("N=%d: %.1f" % (n, out.double().mean().item() / (iters * 4)))
            print("mma_rate2 pairs=%d %s cycles/MMA  %s" % (pairs, name, "  ".join(row)), flush=True)


def check_umma2():
    """cta_group::2 self-test: D[256 x 64] = A B^T by a CTA pair."""
    import torch
    import psgla_b200 as P
    lib = P._lib.lib()
    torch.manual_seed(0)
    a = torch.randn(256, 64, device="cuda").to(torch.bfloat16).contiguous()
    b = torch.randn(64, 64, device="cuda").to(torch.bfloat16).contiguous()
    ref = a.float() @ b.float().t()
    for mode in (1, 0):
        d = torch.full((256, 64), float("nan"), device="cuda")
        P._lib.check(lib.psgla_selftest_umma2(a.data_ptr(), b.data_ptr(), d.data_ptr(), mode, None), "selftest2")
        torch.cuda.synchronize()
        err = (d - ref).abs()
        print("umma2 mode %d: max err %.3g (rows 0-127: %.3g, rows 128-255: %.3g; cols 0-31: %.3g, cols 32-63: %.3g)"
              % (mode, err.max().item(), err[:128].max().item(), err[128:].max().item(), err[:, :32].max().item(),
                 err[:, 32:].max().item()), flush=True)
        if err.max().item() > 1e-3:
            # which B rows did each column block see?  compare against the swapped halves
            swapped = a.float() @ torch.cat([b[32:], b[:32]]).float().t()
            print("   vs swapped B halves: %.3g" % (d - swapped).abs().max().item(), flush=True)


CHECKS = {k[6:]: v for k, v in list(globals().items()) if k.startswith("check_")}

if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--one":
        CHECKS[sys.argv[2]]()
        sys.exit(0)
    names = sys.argv[1:] or list(CHECKS)
    for n in names:
        print("=== %s" % n, flush=True)
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", n], timeout=300, capture_output=True, text=True,
                               env=dict(os.environ))
            print(r.stdout[-4000:], end="")
            if r.returncode != 0:
                print("--- rc=%d stderr tail:\n%s" % (r.returncode, r.stderr[-2500:]))
        except subprocess.TimeoutExpired:
            print("--- TIMEOUT")
