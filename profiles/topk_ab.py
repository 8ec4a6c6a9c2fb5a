"""A/B timing of the device top-K path (stocs_b200_score_sharded_device, the kPrune kernel) between
library builds (development tool).  On a B200, with each build named by NAME=PATH of its library:
    echo parent=/tmp/a/libstocs_b200.so new=/tmp/b/libstocs_b200.so parent=... new=... | python profiles/topk_ab.py
Each build runs in its own process (STOCS_B200_LIB selects the library).  Per workload it prints the
mean kernel time and call time of one launch, a hash of the K records, and the per-launch rejection
counters of stocs_b200_get_counters: [4] after the coarse test, [5] before a queue drain, [8] after
the brick-bit refinement (a build without that slot reports 0).  Workloads: S1 (10^6 hypotheses),
S1-fit (generated once, cached in the temporary directory), S1/8, and the two extreme S2 model sizes
(384, 1024 points, 10^6 hypotheses each on the S2 class maps).  The hashes must not change between
builds."""
import sys, os, ctypes, subprocess, hashlib, tempfile

STEPS, WARM, K = 20, 3, 32

if len(sys.argv) > 1:
    sys.path.insert(0, '.')
    import numpy as np, torch, bench
    from model_matching_b200 import Context, synth
    sc, mpos, mnrm, T = bench.workload(0, 1000000)
    s = torch.cuda.Stream()
    sp = ctypes.c_void_p(s.cuda_stream)
    out = '%-10s' % sys.argv[1]

    def counters(ctx):
        c = np.zeros(9, np.int64)
        ctx._check(ctx._L.stocs_b200_get_counters(ctx.h, c.ctypes.data_as(ctypes.c_void_p), 9))
        return c

    def run(ctx, name, TT):
        global out
        H = len(TT)
        dT = torch.from_numpy(TT).cuda()
        drec = torch.zeros(K * 64, dtype=torch.uint8, device='cuda')
        with torch.cuda.stream(s):
            for _ in range(WARM):
                ctx.score_sharded_device(dT.data_ptr(), H, 0, K, drec.data_ptr(), sp)
            torch.cuda.synchronize()
            ctx.kernel_ms_stats(reset=True)
            c0 = counters(ctx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for _ in range(STEPS):
                ctx.score_sharded_device(dT.data_ptr(), H, 0, K, drec.data_ptr(), sp)
            e1.record(s)
            torch.cuda.synchronize()
        n, kms, _ = ctx.kernel_ms_stats()
        dc = (counters(ctx) - c0) // STEPS
        rec = hashlib.sha1(drec.cpu().numpy().tobytes()).hexdigest()[:8]
        out += ' | %s kernel %.4f call %.4f ms rec %s rej %d/%d/%d' % (
            name, kms, e0.elapsed_time(e1) / STEPS, rec, dc[4], dc[5], dc[8])

    ctx = Context(0); ctx.upload_model(mpos, mnrm); ctx.upload_scene(sc['pos'], sc['nrm'], sc['cls'])
    fitp = os.path.join(tempfile.gettempdir(), 'topk_ab_s1fit_T.npy')
    if not os.path.exists(fitp):
        Tf, info = bench.fitted_hypotheses(ctx, len(T))
        np.save(fitp, Tf)
    Tf = np.load(fitp)
    run(ctx, 'S1', T)
    run(ctx, 'S1-fit', Tf)
    run(ctx, 'S1/8', T[:125000])
    ctx.close()
    for k, m in enumerate(bench.S2_MODEL_POINTS):
        if m not in (384, 1024):
            continue
        p, nrm = synth.make_model(m)
        c = Context(0); c.upload_model(p, nrm)
        c.upload_scene(sc['pos'], sc['nrm'], synth.class_map(len(sc['pos']), 1000 + k))
        T2, _ = synth.make_hypotheses(1000000, sc['pos'], p, sc['gt_R'], sc['gt_t'], seed=1000 + k)
        run(c, 'S2/M%d' % m, T2)
        c.close()
    print(out, flush=True)
else:
    for v in sys.stdin.read().split():
        name, _, path = v.partition('=')
        env = dict(os.environ, STOCS_B200_LIB=os.path.abspath(path))
        subprocess.run([sys.executable, 'profiles/topk_ab.py', name], env=env, check=True)
