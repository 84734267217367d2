"""Per-CTA phase timeline of k_render inside the real step (debug flag 4 -> cbev_debug_read_trace).
Prints phase durations and how many CTAs are in their store phase over time.
Usage: render_trace.py [x|brake] [flags] [--mask-dtype float32|uint8]  (uint8: the 0 / 1 byte planes of mask_dtype)."""
import sys, torch, numpy as np
sys.path.insert(0, ".")
from carlabev_env_b200 import engine as E
from carlabev_env_b200.pool import pack_pool
from carlabev_env_b200.vector_env import load_town01_map
if __name__ == "__main__":
    N = 4096
    mask_dtype = "float32"
    if "--mask-dtype" in sys.argv:
        k = sys.argv.index("--mask-dtype")
        mask_dtype = sys.argv[k + 1]
        del sys.argv[k:k + 2]
    brake = len(sys.argv) > 1 and sys.argv[1] == "brake"
    from carlabev_env_b200.scenes import build_pool
    scenes = build_pool([dict(scene="lead_brake", level=1 + i % 3, scene_seed=i) for i in range(1024)])
    eng = E.Engine(N, action_mode=E.ACTION_CONTINUOUS, max_actors=4, autoreset=E.AUTORESET_NEXT_STEP, ring_slots=64,
                   mask_dtype=mask_dtype)
    eng.upload_map(load_town01_map()); eng.upload_pool(pack_pool(scenes))
    eng.reset(torch.arange(N, dtype=torch.int32) % len(scenes))
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    acts = [torch.rand(N, 3, device="cuda", generator=g) * torch.tensor([1, 2, 1], device="cuda") - torch.tensor([0, 1, 0], device="cuda") for _ in range(64)]
    if brake:
        for a in acts: a[:, 0] = 0; a[:, 2] = 1
    extra = int(sys.argv[2], 0) if len(sys.argv) > 2 else 0
    eng.set_debug_flags(4 | extra)
    for i in range(40): eng.step(acts[i % 64])
    torch.cuda.synchronize()
    out = []
    for i in range(6):
        eng.step(acts[(40 + i) % 64]); torch.cuda.synchronize()
        out.append(eng.read_trace().astype(np.int64))
    names = ["tma wait", "draw list", "rotate", "resize", "stores"]
    for k, tr in list(enumerate(out[1:]))[-1:]:
        t = tr[:, :6]; t0 = t[:, 0].min()
        ph = np.diff(t, axis=1) / 1e3
        life = (t[:, 5] - t[:, 0]) / 1e3
        print(f"launch {k}: span {(t[:, 5].max() - t0) / 1e3:.1f} us; CTA life mean {life.mean():.1f} p10 {np.percentile(life, 10):.1f} p90 {np.percentile(life, 90):.1f} max {life.max():.1f} us")
        print(f"   draw list, warp 0 only (before the barrier): {((tr[:, 7] - tr[:, 1]) / 1e3).mean():.2f} us")
        print("   phase means (us): " + ", ".join(f"{n} {ph[:, i].mean():.2f} (p90 {np.percentile(ph[:, i], 90):.2f})" for i, n in enumerate(names)))
        starts = np.sort(t[:, 0] - t0) / 1e3
        print(f"   CTA start times: first wave (592th) {starts[591]:.1f} us, median {np.median(starts):.1f}, last {starts[-1]:.1f} us; last finish {(t[:, 5].max() - t0) / 1e3:.1f}")
        # concurrency of the store phase sampled every 10 us
        grid = np.arange(0, (t[:, 5].max() - t0) / 1e3, 10.0)
        s0, s1 = (t[:, 4] - t0) / 1e3, (t[:, 5] - t0) / 1e3
        c0, c1 = (t[:, 0] - t0) / 1e3, (t[:, 4] - t0) / 1e3
        print("   t(us): storing CTAs / computing CTAs: " + "  ".join(f"{int(x)}:{int(((s0 <= x) & (s1 > x)).sum())}/{int(((c0 <= x) & (c1 > x)).sum())}" for x in grid))
        heavy = (ph[:, 4] > 2.0 * np.median(ph[:, 4]))
        print(f"   CTAs with a store phase > 2x median (reset frames): {int(heavy.sum())}, their mean store phase {ph[heavy, 4].mean() if heavy.any() else 0:.1f} us vs median {np.median(ph[:, 4]):.1f}")
