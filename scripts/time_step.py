"""CUDA-event time of the fused step alone on bench.py's tuning workload: 4 x 12 MP, bilinear demosaic, the chain of
Bayer_02_Demosaic_02_sRGB_11_13_01_14 (gain -> 3x10 polynomial -> gamma -> tone curve), through ops.PipelineStep
(coefficient preparation + step kernel + finaliser).  The library is the one RISP_LIB_PATH names, so different builds,
e.g. the parent commit's, can be compared in one session:

    RISP_LIB_PATH=build/abl/<variant>.so python scripts/time_step.py [launches=200] [repeats=5] [width=4000]

Prints one JSON line: ms per step for each repeat of `launches` back-to-back launches, and their median.
"""
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from reconfigisp_b200 import _lib, ops  # noqa: E402

N, H, W = 4, 3000, 4000


def main():
    launches = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    W = int(sys.argv[3]) if len(sys.argv) > 3 else globals()['W']
    g = torch.Generator().manual_seed(3)
    raw = torch.rand(N, 1, H, W, generator=g).cuda()
    gt = torch.rand(N, 3, H, W, generator=g).cuda()
    ident = [0.0] * 30
    ident[6] = ident[17] = ident[28] = 1.0
    params = torch.tensor([[1.05, 1.0, 0.95] + ident + [0.5, 0.25, 0.5, 0.75]]).cuda()
    step = ops.PipelineStep(N, H, W, 'bilinear', ops.Chain(['gain', 'poly10', 'gamma', ('gtm', 4)]), 'cuda')
    for _ in range(20):
        step(raw, gt, params)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        e0.record()
        for _ in range(launches):
            step(raw, gt, params)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / launches)
    print(json.dumps({'lib': os.path.relpath(_lib.LIB_PATH), 'W': W, 'launches': launches, 'ms': [round(x, 5) for x in ms],
                      'median_ms': round(statistics.median(ms), 5), 'gpu': torch.cuda.get_device_name()}))


if __name__ == '__main__':
    main()
