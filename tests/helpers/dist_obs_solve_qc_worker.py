"""Worker of tests/test_outlier_qc.py (run under torchrun, one rank per GPU): the distributed obs-space solve with
outlier thresholds against the replicated one on the same synthetic obs block, with 5 % gross errors.  Rank 0 prints
one JSON line."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from efa_xray_b200 import engine, _lib  # noqa: E402
from efa_xray_b200.synth import draw_obs_locations  # noqa: E402


def main():
    rank, world, lr = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(lr)
    dev = torch.device('cuda', lr)
    dist.init_process_group('nccl', device_id=dev)
    nobs, nens, cutoff = int(sys.argv[1]), int(sys.argv[2]), float(sys.argv[3])
    block = int(sys.argv[4]) if len(sys.argv) > 4 else 1
    rng = np.random.default_rng(7)
    lat, lon = draw_obs_locations(rng, nobs, 181, 360)
    assim = (rng.uniform(0, 1, nobs) > 0.05).astype(np.uint8)
    error = rng.uniform(0.5, 2.0, nobs)
    value = rng.normal(0, 1, nobs)
    gross = rng.uniform(0, 1, nobs) < 0.05
    value[gross] += rng.choice([-1.0, 1.0], gross.sum()) * rng.uniform(8.0, 15.0, gross.sum()) * np.sqrt(error[gross])
    obs = engine.ObsArrays(value=value, error=error, lat=lat, lon=lon,
                           halfwidth=np.full(nobs, cutoff / 2) * rng.choice([0.5, 1.0, 2.0], nobs), assimilate=assim,
                           row0=np.zeros(nobs, np.int64), row1=np.zeros(nobs, np.int64), tw0=np.ones(nobs), tw1=np.zeros(nobs),
                           threshold=np.where(rng.uniform(0, 1, nobs) < 0.9, 3.0, np.inf))
    lam, phi = np.radians(lon), np.radians(lat)
    amp = rng.normal(0, 1, (4, nens))
    B = np.stack([np.cos((i + 1) * lam + 0.3 * i) * np.cos((i % 3 + 1) * phi) * np.cos(phi) for i in range(4)], 1)
    Y = B @ amp + 0.3 * rng.standard_normal((nobs, nens))
    Yp0 = torch.as_tensor(Y - Y.mean(1, keepdims=True)).to(dev)
    Ym0 = torch.as_tensor(Y.mean(1)).to(dev)
    obs_dev, geo = engine.upload_obs(obs, dev, engine.LOC_GC)

    def run(distributed):
        ym, yp = Ym0.clone(), Yp0.clone()
        rec = torch.empty((8, nobs), dtype=torch.float64, device=dev)
        cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        plan = engine.ObsPlan(obs_dev, geo, nobs, engine.LOC_GC, rank, world, block) if distributed else \
            engine.ObsPlan(obs_dev, geo, nobs, engine.LOC_GC)
        plan.finish()
        if distributed:
            ok = engine.obs_solve_distributed(ym, yp, obs_dev, geo, nens, engine.LOC_GC, rec, cnt, 'f64', plan)
        else:
            engine.obs_solve(ym, yp, obs_dev, geo, nens, engine.LOC_GC, rec, cnt, 'f64', plan=plan)
            ok = True
        torch.cuda.synchronize()
        _lib.call('exb_obs_solve_async_status')
        plan.destroy()
        r = rec.cpu().numpy()
        return ok, ym.cpu().numpy(), yp.cpu().numpy(), r, int(cnt[0].item()), int((assim.astype(bool) & (r[7] == 0)).sum())

    ref = run(False)
    got = run(True)
    m = ~np.isnan(ref[3])
    out = dict(ok=bool(got[0]), world=world, block=block, pairs=[got[4], ref[4]], rejected=[got[5], ref[5]],
               maxdiff_yp=float(np.abs(got[2] - ref[2]).max()), maxdiff_ym=float(np.abs(got[1] - ref[1]).max()),
               nan_pattern_equal=bool((np.isnan(got[3]) == np.isnan(ref[3])).all()),
               maxdiff_rec=float(np.abs(got[3][m] - ref[3][m]).max()))
    if rank == 0:
        print('RESULT ' + json.dumps(out))
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
