"""CUDA-event time of the embedding forward with and without `output_hidden_states` at 512x512x320 (smb-vision-base):
`model(x)` with the flag off, with all 13 states, and `EmbeddingRunner(layers=(3, 6, 9, 12))` end to end (H2D, forward,
D2H of the four states) per volume.  Prints one JSON line with the card name and power limit beside the numbers.

    python tools/hidden_states_time.py [--iters 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    import __graft_entry__ as ge
    from oracle import videomae_oracle as vo
    from smb_vision_b200.inference import EmbeddingRunner
    from smb_vision_b200.modeling import B200VideoMAEModel

    cfg = vo.OracleConfig()
    torch.manual_seed(0)
    m = B200VideoMAEModel(ge.hf_config({k: getattr(cfg, k) for k in cfg.__dataclass_fields__})).cuda().eval()
    x = vo.synthetic_volume(cfg, 1, 7)
    xd = x.cuda()

    def timed(fn, n):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / n

    res = {}
    with torch.no_grad():
        for _ in range(2):  # alternate the two variants twice: the spread between rounds is the noise
            res.setdefault("forward_ms", []).append(timed(lambda: m(xd), args.iters))
            res.setdefault("forward_all_states_ms", []).append(timed(lambda: m(xd, output_hidden_states=True), args.iters))
    vols = [x.pin_memory() for _ in range(args.iters)]
    for layers, key in ((None, "runner_last_ms"), ((3, 6, 9, 12), "runner_layers_3_6_9_12_ms")):
        r = EmbeddingRunner(m, layers=layers)
        for _ in r.embed_stream(iter(vols[:3])):
            pass
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in r.embed_stream(iter(vols)):
            pass
        b.record()
        b.synchronize()
        res[key] = a.elapsed_time(b) / len(vols)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    res["gpu"] = q
    print(json.dumps(res))


if __name__ == "__main__":
    main()
