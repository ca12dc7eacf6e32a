"""Drop-in for the hologram-path functions of the reference's ``generate_hologram.py``:
target preparation (PIL, byte-exact with the reference), the algorithm call, analytic
deflect / lens holograms and the expected-outcome preview on the device."""
from __future__ import annotations

import os

import numpy as np
import PIL.ImageOps
from PIL import Image as im

from . import constants as c
from . import wavefront_correction as wfc
from .algorithms import gerchberg_saxton, gradient_descent, weighted_gerchberg_saxton
from .engine import get_engine

# -alg choices -> hologram functions (the reference sends every choice but GS to gradient descent)
ALGORITHMS = {"gerchberg_saxton": gerchberg_saxton, "gradient_descent": gradient_descent,
              "weighted_gerchberg_saxton": weighted_gerchberg_saxton}


def main(args):
    """reference: generate_hologram.py:13-21."""
    if args.img_name is None:
        hologram = np.zeros((c.slm_height, c.slm_width))
    else:
        hologram = make_hologram(args)
    hologram = transform_hologram(hologram, args)
    if args.preview:
        show_expected_outcome(hologram, args)
    save_hologram_and_gif(hologram, args)


def expected_outcome(hologram, norm=255, precision="fp64"):
    """Numeric part of show_expected_outcome (generate_hologram.py:24-29):
    |fft2(exp(1j*hologram))|^2 / max * norm."""
    hologram = np.asarray(hologram, dtype=np.float64)
    eng = get_engine(hologram.shape, precision)
    return eng.to_host(eng.expected_outcome(hologram, norm))


def show_expected_outcome(hologram, args):
    """reference: generate_hologram.py:24-34."""
    normed = expected_outcome(hologram, find_out_norm(args))
    im.fromarray(normed).resize((c.slm_height, c.slm_height)).show()


def find_out_norm(args):
    """reference: generate_hologram.py:37-42."""
    if args.img_name is None:
        return 255
    img = im.open(f"images/{args.img_name}").convert("L")
    return np.amax(np.array(img))


def pad_to_square(img):
    """Pads the image with black pixels to make it square (reference: generate_hologram.py:45-67)."""
    width, height = img.size
    if width == height:
        return img
    new_size = max(width, height)
    new_img = im.new("L", (new_size, new_size), 0)
    new_img.paste(img, ((new_size - width) // 2, (new_size - height) // 2))
    return new_img


def make_hologram(args):
    """reference: generate_hologram.py:70-79."""
    algorithm = ALGORITHMS.get(args.algorithm, gradient_descent)
    target = prepare_target(args.img_name, args)
    if getattr(args, "gif", False):
        add_gif_dirs(args)
        remove_files_in_dir(args.gif_source_dir)
    hologram, _, _ = algorithm(target, args)
    return hologram


def add_gif_dirs(args):
    """reference: generate_hologram.py:90-99 -- where the per-iteration frames and the finished GIF go."""
    if args.gif_type == "h":
        args.gif_dest_dir = "holograms"
    elif args.gif_type == "i":
        args.gif_dest_dir = "images"
    os.makedirs(args.gif_dest_dir, exist_ok=True)
    args.gif_source_dir = f"{args.gif_dest_dir}/gif_source"
    os.makedirs(args.gif_source_dir, exist_ok=True)


def remove_files_in_dir(dir_name):
    """reference: generate_hologram.py:216-219."""
    for file in os.listdir(dir_name):
        os.remove(f"{dir_name}/{file}")


def create_gif(img_dir, outgif_path):
    """All images of ``img_dir`` (in os.listdir order, like generate_hologram.py:206-213) -> one animated GIF.
    imageio is used when it is installed (the reference's writer), Pillow's GIF encoder otherwise."""
    files = [f"{img_dir}/{f}" for f in os.listdir(img_dir)]
    try:
        import imageio
    except ImportError:
        frames = [im.open(f).convert("L") for f in files]
        if frames:
            frames[0].save(outgif_path, save_all=True, append_images=frames[1:], loop=0)
        return
    with imageio.get_writer(outgif_path, mode="I") as writer:
        for f in files:
            writer.append_data(imageio.imread(f))


def transform_hologram(hologram, args):
    """reference: generate_hologram.py:82-87."""
    if args.deflect is not None:
        hologram = deflect_hologram(hologram, args.deflect)
    if args.lens:
        hologram = add_lens(hologram, args.lens)
    return hologram


def prepare_target(img_name, args):
    """reference: generate_hologram.py:102-110 (host-side PIL pipeline, unchanged)."""
    target_img = im.open(f"images/{img_name}").convert("L")
    if args.invert:
        target_img = PIL.ImageOps.invert(target_img)
    target_img = pad_to_square(target_img)
    if args.quarterize:
        target_img = quarter(target_img)
    resized = target_img.resize((int(c.slm_width), int(c.slm_height)))
    return np.array(resized)


def save_hologram(hologram, args):
    """reference: generate_hologram.py:113-122 (the .npy part of save_hologram_and_gif)."""
    img_name = os.path.basename(args.img_name).split(".")[0] if args.img_name else "analytical"
    dest_dir = args.destination_directory
    if not os.path.exists(dest_dir):
        os.makedirs(dest_dir)
    name = wfc.originalize_name(f"{dest_dir}/{make_hologram_name(args, img_name)}.npy")
    np.save(name, hologram)
    return name


def save_hologram_and_gif(hologram, args):
    """reference: generate_hologram.py:113-128."""
    save_hologram(hologram, args)
    if getattr(args, "gif", False):
        img_name = os.path.basename(args.img_name).split(".")[0] if args.img_name else "analytical"
        create_gif(args.gif_source_dir, wfc.originalize_name(f"{args.gif_dest_dir}/{make_hologram_name(args, img_name)}.gif"))


def make_hologram_name(args, img_name):
    """reference: generate_hologram.py:131-154 (including the runs of spaces its f-string embeds)."""
    alg_params = ""
    transforms = ""
    img_transforms = ""
    if args.deflect:
        transforms += f"_deflect_x{args.deflect[0]}_y{args.deflect[1]}"
    if args.lens:
        transforms += f"_lens{args.lens}"
    if args.algorithm == "gradient_descent":
        alg_params += f"_lr{args.learning_rate}_mr{args.white_attention}_unsettle{args.unsettle}"
    if args.quarterize:
        img_transforms += "_quarter"
    if args.invert:
        img_transforms += "_inverted"
    if args.img_name is None:
        return f"{img_name}{transforms}"
    pad = " " * 8
    return f"{img_name}{img_transforms}{pad}_{args.algorithm}{pad}{alg_params}{pad}_loops{args.max_loops}{pad}{transforms}"


def quarter(image):
    """reference: generate_hologram.py:166-175."""
    w, h = image.size
    resized = image.resize((w // 2, h // 2))
    ground = im.new("L", (w, h))
    ground.paste(resized)
    return ground


def deflect_hologram(hologram, angle: tuple):
    """(hologram + deflect_2pi(angle)) % 2pi on the device (reference: generate_hologram.py:178-182)."""
    hologram = np.asarray(hologram, dtype=np.float64)
    if hologram.shape[-2:] != (c.slm_height, c.slm_width):
        raise ValueError(f"operands could not be broadcast together with shapes {hologram.shape} "
                         f"({c.slm_height},{c.slm_width})")
    eng = wfc._util_engine()
    deflect = eng.deflect_phase(angle, c.px_distance, c.wavelength, c.u, (c.slm_height, c.slm_width))
    return eng.to_host(eng.add_mod2pi(hologram, deflect))


def add_lens(hologram, focal_len: float, uint8_quirk: bool = True):
    """(hologram + lens(f, shape)) % 2pi (reference: generate_hologram.py:185-186)."""
    hologram = np.asarray(hologram, dtype=np.float64)
    eng = wfc._util_engine()
    ln = eng.lens_phase(focal_len, c.px_distance, c.wavelength, hologram.shape[-2:], uint8_quirk)
    return eng.to_host(eng.add_mod2pi(hologram, ln))


def lens(focal_length, shape, uint8_quirk: bool = True):
    """Thin-lens phase (reference: generate_hologram.py:189-203).  With ``uint8_quirk`` (default)
    the result is the reference's uint8 array holding the truncated phase 0..6; pass False for the
    float64 phase the reference presumably intended."""
    eng = wfc._util_engine()
    out = eng.to_host(eng.lens_phase(focal_length, c.px_distance, c.wavelength, tuple(shape), uint8_quirk))
    return out.astype(np.uint8) if uint8_quirk else out


def build_parser():
    """The reference's command line (generate_hologram.py:222-369): same flags, defaults and types, so existing
    invocations keep working; ``--precision`` is the one addition."""
    import argparse
    p = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                                description="Phase hologram for a transmissive SLM, computed on a B200 (drop-in for the "
                                            "reference's generate_hologram.py).  Holograms are saved as .npy files.")
    p.add_argument("img_name", nargs="?", default=None, type=str, help="target image inside images/; omit for a pure deflect/lens hologram")
    p.add_argument("-ii", "--incomming_intensity", type=str, default="uniform", help="illumination image path, or 'uniform'")
    p.add_argument("-ig", "--initial_guess", type=str, default="random", choices=["random", "fourier"], help="initial guess of gradient_descent")
    p.add_argument("-dest_dir", "--destination_directory", type=str, default="holograms", help="where the hologram is saved")
    p.add_argument("-q", "--quarterize", action="store_true", help="shrink the target into one quadrant of a black image")
    p.add_argument("-i", "--invert", action="store_true", help="invert the target image")
    p.add_argument("-alg", "--algorithm", default="gerchberg_saxton", choices=list(ALGORITHMS))
    p.add_argument("-tol", "--tolerance", default=0, metavar="FLOAT", type=float, help="stop when the error falls to this value")
    p.add_argument("-l", "--max_loops", default=42, metavar="INTEGER", type=int, help="upper bound on the number of iterations")
    p.add_argument("-lr", "--learning_rate", default=0.005, type=float, help="gradient descent step")
    p.add_argument("-wa", "--white_attention", metavar="FLOAT", default=1, type=float, help="error weight of white areas (gradient descent)")
    p.add_argument("-u", "--unsettle", default=0, metavar="INTEGER", type=int, help="number of learning-rate doublings (gradient descent)")
    p.add_argument("-gif", action="store_true", help="animated GIF of the iterations")
    p.add_argument("-gif_t", "--gif_type", choices=["h", "i"], default="i", help="GIF of holograms (h) or of reconstructed images (i)")
    p.add_argument("-gif_skip", default=1, type=int, metavar="INTEGER", help="every gif_skip-th iteration becomes a GIF frame")
    p.add_argument("-plot_error", action="store_true", help="plot the error curve")
    p.add_argument("-p", "--preview", action="store_true", help="show the expected outcome")
    p.add_argument("-deflect", nargs=2, type=float, metavar=("X_ANGLE", "Y_ANGLE"), default=None,
                   help="add a deflection hologram (units: a quarter of the first diffraction maximum)")
    p.add_argument("-lens", default=None, type=float, metavar="FOCAL_LENGTH", help="add a lens of this focal length [m]")
    p.add_argument("--precision", default=None, choices=["fp32", "fp64"], help="engine arithmetic (default fp32)")
    p.add_argument("--weight_limit", default=10.0, type=float, metavar="FLOAT",
                   help="weighted_gerchberg_saxton: the weights stay within [1/limit, limit] (>= 1)")
    return p


def cli(argv=None):
    args = build_parser().parse_args(argv)
    args.random_seed = 42                       # generate_hologram.py:370-371
    args.print_info = True
    args.correspond_to2pi = 256                 # read by the "-gif -gif_t h" frames (the reference's parser omits it, SURVEY A.7)
    os.makedirs(args.destination_directory, exist_ok=True)
    main(args)


if __name__ == "__main__":
    cli()
