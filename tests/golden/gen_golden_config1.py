"""Golden vectors FROM THE UNMODIFIED REFERENCE for BASELINE config 1 (MNIST-shaped 1x32x32, T=20, k=11, sigma=7, Constant,
B=4, full-size Unet).  Needs the reference checkout (ref_shim.REF_ROOT).  The weights are UO.make_unet_state_dict(64, (1, 2, 4, 8),
1, seed=0), which the test rebuilds bit for bit, so the 226 MB state dict itself is not stored.

    python tests/golden/gen_golden_config1.py     ->  tests/golden/config1_mnist.npz
"""
import os, sys
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.path.insert(0, HERE)
import ref_shim  # noqa
import unet_oracle as UO  # noqa
from gen_golden import quiet, save  # noqa


def main():
    torch.set_num_threads(8)
    m = ref_shim.import_reference('deblurring-diffusion-pytorch', 'deblurring_diffusion_pytorch')
    unet = quiet(m.Unet, dim=64, dim_mults=(1, 2, 4, 8), channels=1)
    unet.load_state_dict(UO.make_unet_state_dict(64, (1, 2, 4, 8), 1, seed=0))
    gd = m.GaussianDiffusion(unet, image_size=32, device_of_kernel='cpu', channels=1, timesteps=20,
                             kernel_std=7.0, kernel_size=11, blur_routine='Constant', loss_type='l1')
    torch.manual_seed(1234)
    x = torch.rand(4, 1, 32, 32) * 2 - 1
    t = torch.randint(0, 20, (4,))
    with torch.no_grad():
        loss = gd.p_losses(x, t)
        y = unet(gd.q_sample(x_start=x, t=t), t)
    save('config1_mnist', x=x, t=t, loss=loss, y=y)


if __name__ == '__main__':
    main()
