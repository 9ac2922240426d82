"""Times the pyramid build of a small batch on both paths: the cluster build (pyr_build_cluster_kernel, 8 or 16 CTAs per
image) and the one-launch grid build (pyr_build_fused_kernel), for 1 to 16 KITTI-sized images (1241 x 376, 3 levels built)
and a few at 1024 x 768.  The threshold of the cluster build (KLT_PYR_CLUSTER_MAX_ITEMS in klt_pyramid.cu) and its CTAs per
image come from this sweep.

    python scripts/pyr_cluster_sweep.py            # builds the three library variants, then times each in a subprocess

Log of the run behind the defaults: profiles/r03/pyr_cluster_sweep.log.

Every build reads level 0 from a pool of distinct images larger than L2, as in bench.py.  The builds of one configuration
are queued back to back between two CUDA events (launch i builds items [i B, (i + 1) B) of the pool), so the figure is the
time a build adds to a stream, CPU launch path excluded.  The card's name and power limit are printed with the numbers."""
import ctypes, os, subprocess, sys, statistics
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = {   # name -> extra nvcc flags
    "cluster16": "-DKLT_PYR_CLUSTER_CTAS=16 -DKLT_PYR_CLUSTER_MAX_ITEMS=16",
    "cluster8": "-DKLT_PYR_CLUSTER_CTAS=8 -DKLT_PYR_CLUSTER_MAX_ITEMS=16",
    "fused": "-DKLT_PYR_CLUSTER_MAX_ITEMS=0",
}
SHAPES = [((376, 1241), list(range(1, 17))), ((768, 1024), [1, 2, 4, 8])]


def measure(variant):
    import torch
    from visual_odom_pipeline_b200 import _lib, tracker as T
    L = _lib.load()
    ctx = _lib.default_context(0)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for (h, w), batches in SHAPES:
        pool = max(16, (160 << 20) // (h * ((w + 127) // 128 * 128)))        # > L2 (126 MB)
        imgs = T.alloc_image_batch(pool, h, w)
        imgs.copy_(torch.randint(0, 256, (pool, h, w), dtype=torch.uint8, device="cuda"))
        lay = _lib.klt_pyr_layout()
        assert L.klt_pyr_plan(w, h, 21, 21, 3, pool, ctypes.byref(lay)) == 0
        lay.level[0].pitch = imgs.stride(1)
        lay.level[0].batch_stride = imgs.stride(0)
        buf = torch.zeros(int(lay.bytes), dtype=torch.uint8, device="cuda")
        for B in batches:
            slots = pool // B
            def build(i):
                assert L.klt_pyr_build(ctx.handle, imgs.data_ptr(), ctypes.byref(lay), buf.data_ptr(), (i % slots) * B, B, st) == 0
            for i in range(50):
                build(i)
            runs = []
            for r in range(5):
                n = 400
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for i in range(n):
                    build(r * n + i)
                e1.record()
                torch.cuda.synchronize()
                runs.append(e0.elapsed_time(e1) * 1e3 / n)
            print("%-9s %4dx%-4d B=%2d  %6.2f us per build (median of 5 x 400; min %.2f, max %.2f)"
                  % (variant, w, h, B, statistics.median(runs), min(runs), max(runs)), flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--measure":
        measure(sys.argv[2])
        sys.exit(0)
    import importlib.util
    spec = importlib.util.spec_from_file_location("klt_build", os.path.join(ROOT, "visual-odom-pipeline_b200", "build.py"))
    bmod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bmod)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("card: %s" % smi, flush=True)
    for name, extra in VARIANTS.items():
        lib = bmod.build(variant=name, extra=extra.split())
        env = dict(os.environ, KLT_LIB_PATH=lib)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--measure", name], env=env, check=True)
