"""Worker of tests/test_gpu_verify_families.py (one process per GPU, launched by torch.distributed.run): the protected
SRGAN generator's verification sweep over N seeded inputs, every rank evaluating its contiguous slice, the sums merged
by one all-reduce.  Prints the merged result on rank 0."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    n, batch = int(sys.argv[1]), int(sys.argv[2])
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import ipr_gan_b200
    ipr_gan_b200.enable_dropin()
    import models
    from configs import presets
    from ipr_gan_b200 import verify
    os.environ["IPR_VGG_RANDOM_INIT"] = "1"
    torch.manual_seed(1234)                              # the same weights and trigger on every rank (and in the test)
    m = models.SRGAN(presets.srgan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.srgan_blackbox())
    inputs = torch.rand(n, 3, 24, 24, generator=torch.Generator().manual_seed(11))
    res = verify.image_verification_sweep(m.G, m.fn_inp, m.fn_out, inputs, batch=batch)
    if rank == 0:
        res["world"] = dist.get_world_size()
        print("RESULT " + json.dumps(res))
    sys.stdout.flush()
    torch.cuda.synchronize()
    os._exit(0)


if __name__ == "__main__":
    main()
