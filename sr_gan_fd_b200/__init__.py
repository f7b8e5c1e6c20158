"""sr_gan_fd_b200 -- B200-native (sm_100a) RRDBNet generator for MiNeves00/SR-GAN-FD: drop-in modules whose forward and
backward run in hand-written tcgen05/TMA CUDA kernels behind the C ABI of ``include/b200sr.h``."""
from .rrdbnet import (BSRGAN, BasicSRRRDBNet, RRDBNet, RRDBTrunk, RealRRDBNet, bsrgan_x2, bsrgan_x4, native_generator, native_trunk,
                      real_rrdbnet_x4, rrdbnet_x1, rrdbnet_x2, rrdbnet_x4, rrdbnet_x8)
from .function import attach_grad_bucket_hook

__all__ = ["RRDBNet", "BSRGAN", "RealRRDBNet", "rrdbnet_x1", "rrdbnet_x2", "rrdbnet_x4", "rrdbnet_x8", "bsrgan_x2",
           "bsrgan_x4", "real_rrdbnet_x4", "RRDBTrunk", "native_trunk", "BasicSRRRDBNet", "native_generator",
           "attach_grad_bucket_hook"]
