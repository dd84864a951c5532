"""Embedding extraction on the B200 path — the role of the reference's `src/run_inference.py` / `run_inspect.py`.

    python examples/extract_embeddings.py --synthetic 6 --save_dir /tmp/emb --format parquet --model_id smb-vision-base

Volumes are sharded over the ranks in contiguous chunks with no collective (run_inspect.py:206-241); each rank streams its
chunk through `EmbeddingRunner` (H2D of volume i+1 and D2H of embedding i-1 overlap the compute of volume i) and writes
`<stem>.npy` (run_inference.py:89-96) or `model_id=<id>/<uid>.parquet` (run_inspect.py:140-175) from a writer pool; files
that already exist are skipped (run_inspect.py:33-50).
"""
from __future__ import annotations

import argparse
import glob
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--volumes", nargs="*", default=[], help=".npy files, one resampled volume [X,Y,Z] each (fp32 or int16 HU)")
    ap.add_argument("--synthetic", type=int, default=0)
    ap.add_argument("--model_name_or_path", default=None)
    ap.add_argument("--image_size", type=int, default=512)
    ap.add_argument("--depth", type=int, default=320)
    ap.add_argument("--save_dir", required=True)
    ap.add_argument("--format", default="parquet", choices=["parquet", "npy"])
    ap.add_argument("--model_id", default="smb-vision-base")
    ap.add_argument("--config_overrides", default="")
    ap.add_argument("--layers", default="", help="comma-separated hidden-state indices (0 = patch embedding, k = block k), "
                    "e.g. 3,6,9,12: each embedding is then [len(layers), N, d] instead of last_hidden_state")
    args = ap.parse_args(argv)

    from transformers import VideoMAEConfig

    from smb_vision_b200.data import VolumePreprocessor
    from smb_vision_b200.distributed import shard_volumes
    from smb_vision_b200.inference import EmbeddingRunner
    from smb_vision_b200.modeling import B200VideoMAEModel
    from smb_vision_b200.output import EmbeddingWriter, processed_uids

    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    config = VideoMAEConfig.from_pretrained(args.model_name_or_path) if args.model_name_or_path else VideoMAEConfig()
    config.update({k: type(getattr(config, k))(v) for k, v in (kv.split("=") for kv in args.config_overrides.split(",") if kv)})
    config.update(dict(image_size=args.image_size, patch_size=16, num_channels=1, num_frames=args.depth, tubelet_size=16))
    torch.manual_seed(0)
    model = (B200VideoMAEModel.from_pretrained(args.model_name_or_path, config=config) if args.model_name_or_path
             else B200VideoMAEModel(config)).to(dev).eval()

    if args.synthetic:
        g = torch.Generator().manual_seed(0)
        items = [(f"synthetic_{i:04d}", torch.randint(-1100, 1500, (args.image_size, args.image_size, args.depth), generator=g, dtype=torch.int16))
                 for i in range(args.synthetic)]
    else:
        files = sorted(f for pat in args.volumes for f in glob.glob(pat))
        items = [(os.path.basename(f).replace(".npy", ""), f) for f in files]
    done = processed_uids(args.save_dir) if args.format == "parquet" else {f[:-4] for f in os.listdir(args.save_dir)} if os.path.isdir(args.save_dir) else set()
    items = [it for it in items if it[0] not in done]
    items = shard_volumes(items, rank, world)

    prep = VolumePreprocessor(args.image_size, args.depth, device=dev)
    layers = [int(k) for k in args.layers.split(",") if k] or None
    runner = EmbeddingRunner(model, preprocess=prep, layers=layers)
    writer = EmbeddingWriter(args.save_dir, fmt=args.format, model_id=args.model_id)

    def raw_stream():
        for _, src in items:
            raw = src if torch.is_tensor(src) else torch.from_numpy(np.load(src))
            yield raw.pin_memory()

    for (uid, _), emb in zip(items, runner.embed_stream(raw_stream())):
        writer.submit(uid, emb)
    return writer.close()


if __name__ == "__main__":
    main()
