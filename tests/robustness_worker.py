"""Worker of tests/test_gpu_robustness.py (one process per GPU, launched by torch.distributed.run): the protected
SRGAN generator's prune sweep over 13 seeded inputs, every rank pruning its identical replica and evaluating its
contiguous slice of the inputs.  Prints the merged per-level results on rank 0."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import ipr_gan_b200
    ipr_gan_b200.enable_dropin()
    import models
    from configs import presets
    from ipr_gan_b200 import robustness
    os.environ["IPR_VGG_RANDOM_INIT"] = "1"
    torch.manual_seed(4)                                 # the same weights and trigger as the test's _srgan()
    m = models.SRGAN(presets.srgan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.srgan_blackbox())
    m = models.WhiteBoxWrapper(m, presets.whitebox("G"))
    inputs = torch.rand(13, 3, 24, 24, generator=torch.Generator().manual_seed(11))
    rows = robustness.prune_sweep(m, (0.0, 0.5), inputs=inputs, batch=4)
    if rank == 0:
        print("RESULT " + json.dumps(rows))
    sys.stdout.flush()
    torch.cuda.synchronize()
    os._exit(0)


if __name__ == "__main__":
    main()
