#!/usr/bin/env python
"""build_repeat.py -- synth_ms / build_ms of the C2 graph (bench.py's generator) built five times in one process.

The first build of a process includes its first multi-GB allocations, whose cost varies from run to run; the later ones
show the steady state of the build kernels.

    python profiles/microbench/build_repeat.py [label]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch                                                    # noqa: E402
import recommendersystems_b200 as rs                            # noqa: E402
from bench import scaled_spec                                   # noqa: E402

out = []
for _ in range(5):
    g = rs.Graph.synthetic(scaled_spec(1.0), stream=torch.cuda.current_stream().cuda_stream)
    g.buildGraph()
    info = g.info()
    out.append(f"{info.synth_ms:.1f}/{info.build_ms:.1f}")
    g.close()
print(sys.argv[1] if len(sys.argv) > 1 else "", " ".join(out), flush=True)
