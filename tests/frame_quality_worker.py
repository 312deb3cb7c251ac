"""Per-frame signal quality in a process of its own (used by test_gpu_frame_quality.py; not collected as tests).

The demapper's output lag is read from DABSTAR_DEMAP_LAG once per process and DABSTAR_TRACE's round lines once per process,
so each forced-lag configuration and each traced segment layout runs in a fresh process:

    python frame_quality_worker.py MODE IN_DIR OUT_DIR

writes OUT_DIR/out.npz. MODE:

* batch    DabProcessor with set_frame_quality over the 256 copies of demap_worker.batch_source() (768 demapper CTAs, past one
           wave at every lag; every source ends in a cut frame), then every source decoded alone;
* segments DabProcessor with set_segmentation and set_frame_quality over demap_worker.segment_recording(); IN_DIR/in.npz holds
           segment_frames, warmup and max_window.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import demap_worker as W  # noqa: E402


def records(dp, r: int, n_max: int) -> np.ndarray:
    """frame_quality of recording r padded with NaN to n_max rows."""
    q = dp.frame_quality(r)
    out = np.full((n_max, 6), np.nan, np.float32)
    out[:q.shape[0]] = q
    return out


def mode_batch(ctx, inp, out_dir):
    import torch
    from dabstar_b200 import api
    srcs = [W.batch_source(i)[0] for i in range(W.N_SRC)]
    dev = [torch.from_numpy(srcs[i % W.N_SRC]).cuda() for i in range(W.N_COPIES)]
    torch.cuda.synchronize()
    dp = api.DabProcessor(W.N_COPIES, input_format=api.FMT_U8, scan_mode=True, ctx=ctx)
    dp.set_frame_quality(True)
    rounds = W.traced(os.path.join(out_dir, "trace.txt"), lambda: dp.run_ptrs([t.data_ptr() for t in dev], [t.shape[0] for t in dev], api.MEM_DEVICE))
    out = dict(rounds=rounds,
               n_frames=np.array([dp.n_frames(r) for r in range(W.N_COPIES)], np.int64),
               quality=np.stack([records(dp, r, W.F_MAX) for r in range(W.N_COPIES)]))
    del dp, dev
    single_n, single_q = [], []
    for i in range(W.N_SRC):
        dp1 = api.DabProcessor(1, input_format=api.FMT_U8, scan_mode=True, ctx=ctx)
        dp1.set_frame_quality(True)
        dp1.run([srcs[i]])
        single_n.append(dp1.n_frames(0))
        single_q.append(records(dp1, 0, W.F_MAX))
    out["single_n_frames"] = np.array(single_n, np.int64)
    out["single_quality"] = np.stack(single_q)
    np.savez(os.path.join(out_dir, "out.npz"), **out)


def mode_segments(ctx, inp, out_dir):
    from dabstar_b200 import api
    seg_frames, warmup, max_window = int(inp["segment_frames"]), int(inp["warmup"]), int(inp["max_window"])
    dp = api.DabProcessor(1, input_format=api.FMT_U8, scan_mode=True, max_window=max_window, ctx=ctx)
    dp.set_segmentation(seg_frames, warmup)
    dp.set_frame_quality(True)
    rounds = W.traced(os.path.join(out_dir, "trace.txt"), lambda: dp.run([W.segment_recording()]))
    res = dp.result(0)
    out = dict(rounds=rounds, warmup_frames=dp.warmup_frames(0), quality=dp.frame_quality(0), counters=res.counters,
               pos=np.array([(i.sym0_pos, i.start_index) for i in res.info], np.int64).reshape(-1, 2),
               phase_cp=np.array([i.phase_cp for i in res.info], np.float32))
    np.savez(os.path.join(out_dir, "out.npz"), **out)


def main():
    mode, in_dir, out_dir = sys.argv[1:4]
    from dabstar_b200 import api
    ctx = api.Context(0)
    path = os.path.join(in_dir, "in.npz")
    inp = dict(np.load(path)) if os.path.exists(path) else {}
    {"batch": mode_batch, "segments": mode_segments}[mode](ctx, inp, out_dir)


if __name__ == "__main__":
    main()
