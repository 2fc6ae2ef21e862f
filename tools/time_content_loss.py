"""Times the VGG19 content loss of the RealESRGAN generator step (train_realesrgan.py:477) at the training shape,
16 x 3 x 256 x 256 with the RealESRGAN node set: forward + backward of resr_b200.model.ContentLoss against the same loss
through torchvision VGG19 with bf16 autocast, channels_last and cudnn.benchmark (the library bar of tools/library_bar.py).
The two arms alternate over several repetitions after every shape has been warmed up; CUDA events time each. Then the
generator step with the content term added: pixel + content L1 through generator_apply, USM and both backwards.
Development aid: the torchvision arm is never part of the product path. Prints the card name and power limit."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

NODES = ["features.2", "features.7", "features.16", "features.25", "features.34"]
WEIGHTS = [0.1, 0.1, 1.0, 1.0, 1.0]
MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the numbers still stand; say the limit is unknown
        q = f"power limit unknown ({type(e).__name__})"
    return f"{name}, {q}"


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    import resr_b200
    from torchvision.models import vgg19
    from torchvision.models.feature_extraction import create_feature_extractor
    from torchvision import transforms
    assert torch.cuda.is_available(), "time_content_loss.py measures on the GPU"
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    vgg = vgg19(weights=None).eval()
    wgt = torch.tensor(WEIGHTS, device=dev)
    sr = torch.rand(16, 3, 256, 256, device=dev)
    hr = torch.rand(16, 3, 256, 256, device=dev)

    native = resr_b200.model.ContentLoss(NODES, MEAN, STD, vgg=vgg).to(dev)
    x_n = sr.clone().requires_grad_(True)

    def run_native():
        x_n.grad = None
        (native(x_n, hr) * wgt).sum().backward()

    torch.backends.cudnn.benchmark = True
    fe = create_feature_extractor(vgg.to(dev), NODES).to(memory_format=torch.channels_last)
    for p in fe.parameters():
        p.requires_grad_(False)
    norm = transforms.Normalize(MEAN, STD)
    x_l = sr.clone().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    hr_l = hr.contiguous(memory_format=torch.channels_last)

    def run_library():
        x_l.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            fs = fe(norm(x_l))
            with torch.no_grad():
                fg = fe(norm(hr_l))
            loss = sum(w * F.l1_loss(fs[k].float(), fg[k].float()) for w, k in zip(WEIGHTS, NODES))
        loss.backward()

    for _ in range(3):
        run_native()
        run_library()
    torch.cuda.synchronize()
    arms = {"native": [], "library": []}
    for _ in range(5):
        arms["native"].append(timed(run_native, 5))
        arms["library"].append(timed(run_library, 5))
    print(f"card: {card()}")
    for k, v in arms.items():
        v = sorted(v)
        print(f"content loss fwd+bwd 16x3x256x256 RealESRGAN nodes, {k}: median {v[len(v) // 2]:.2f} ms "
              f"(min {v[0]:.2f}, max {v[-1]:.2f}) over {len(v)} x 5 calls")

    # the generator step with the content term: sr = G(lr); g = L1(usm(sr), hr) + sum(w * content(usm(sr), hr))
    from oracle import generator as og
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.random_state_dict(0))
    g = g.to(dev).train()
    usm = resr_b200.imgproc.USMSharp(50, 0).to(dev)
    lr = torch.rand(16, 3, 64, 64, device=dev)

    def step(with_content):
        for p in g.parameters():
            p.grad = None
        out = usm(g(lr), 0.5, 10)
        loss = F.l1_loss(out, hr)
        if with_content:
            loss = loss + (native(out, hr) * wgt).sum()
        loss.backward()

    for _ in range(2):
        step(False)
        step(True)
    torch.cuda.synchronize()
    res = {False: [], True: []}
    for _ in range(3):
        for wc in (False, True):
            res[wc].append(timed(lambda: step(wc), 3))
    for wc, v in res.items():
        v = sorted(v)
        print(f"generator step 16x3x64x64, pixel{' + content' if wc else ''} loss through USM: median {v[len(v) // 2]:.2f} ms "
              f"(min {v[0]:.2f}, max {v[-1]:.2f})")


if __name__ == "__main__":
    main()
