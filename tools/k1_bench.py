"""K1 (colorize) measurement: one JSON line with the colorize ms on (a) 64 rendered 1080p views, (b) white noise metres,
(c) the u16 image re-colorized, the median ms of that u16 image, and a digest of the outputs (also over odd-sized batches
that exercise partial blocks and misaligned image starts).  Times are CUDA events, 20 calls after 3 warm-ups.
Run from the repository root: python tools/k1_bench.py"""
import hashlib, json, os, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import numpy as np
    import torch
    from bodyslam_b200 import mdem, ops, synthetic as S
    dev = torch.device("cuda:0")
    import bench
    args = bench.parse()
    cfg, F, E, res, vl, trunc = bench.workload(args)
    B, Hh, Ww = 64, 1080, 1920
    K1080 = tuple(k * 3.0 for k in cfg["K"])
    Eb = E[np.linspace(0, len(E) - 1, B).astype(int)]
    d1080, _ = S.render(cfg["surface"], Eb, K=K1080, W=Ww, H=Hh, device=dev, with_color=False)
    metres = (d1080.to(torch.float32) / 1000.0).contiguous()
    del d1080
    g = torch.Generator(device=dev).manual_seed(1)
    noise = (torch.rand((B, Hh, Ww), device=dev, generator=g) * 10.0).contiguous()
    lut = mdem.get_cmap_lut("viridis")

    def timed(fn, n=20, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    out = {}
    h = hashlib.sha256()
    for name, x in (("rendered", metres), ("noise", noise)):
        rgba, u16 = ops.colorize_u16(lut, depth_m=x, invalid_val=0)
        h.update(rgba.cpu().numpy().tobytes()); h.update(u16.cpu().numpy().tobytes())
        out[name + "_ms"] = timed(lambda: ops.colorize_u16(lut, depth_m=x, invalid_val=0))
        if name == "rendered":
            out["u16_recolor_ms"] = timed(lambda: ops.colorize_u16(lut, depth_u16=u16, invalid_val=0))
            r2, _ = ops.colorize_u16(lut, depth_u16=u16, invalid_val=0)
            h.update(r2.cpu().numpy().tobytes())
            out["median_ms"] = timed(lambda: ops.median_u16(u16, invalid_val=0)) if hasattr(ops, "median_u16") else None
    # odd sizes: partial blocks, misaligned image starts
    for shp in ((3, 479, 641), (5, 33, 17), (2, 1080, 1921)):
        x = (torch.rand(shp, device=dev, generator=g) * 3.0)
        x[x < 0.1] = 0
        rgba, u16 = ops.colorize_u16(lut, depth_m=x.contiguous(), invalid_val=0)
        h.update(rgba.cpu().numpy().tobytes()); h.update(u16.cpu().numpy().tobytes())
    out["digest"] = h.hexdigest()[:16]
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
