"""torchrun worker: sharded training with split_special_tokens over NCCL must reproduce the single-GPU result."""
import os
import pathlib
import sys

import torch
import torch.distributed as dist

ROOT = pathlib.Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
import _bootstrap  # noqa: F401,E402
from tests.helpers import split_train_oracle as sto  # noqa: E402
from transformer_lm_b200 import _lib  # noqa: E402
from transformer_lm_b200.synth import synth_host  # noqa: E402
from transformer_lm_b200.train import train_bpe  # noqa: E402

EOT = "<|endoftext|>"


def main():
    out = pathlib.Path(sys.argv[1])
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = _lib.Context(local)
    path = ROOT / "tests" / "fixtures" / "tinystories_sample.txt"
    got = train_bpe(path, 1000, [EOT], ctx=ctx, distributed=True, split_special_tokens=True)
    assert got == sto.train_bpe(path, 1000, [EOT]), "rank %d differs from the split oracle" % rank
    big = out / "big.txt"
    if rank == 0:
        synth_host("owt", 78, 320 << 20).tofile(big)
    dist.barrier()
    got = train_bpe(big, 3000, [EOT], ctx=ctx, distributed=True, split_special_tokens=True)
    single = train_bpe(big, 3000, [EOT], ctx=ctx, split_special_tokens=True)
    assert got == single, "rank %d differs from the single-GPU split training" % rank
    dist.barrier()
    (out / ("ok.%d" % rank)).write_text("ok")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
