"""Radiance-field model containers with the reference's parameter names.

The render path is model-agnostic in the reference: ``run_network`` just calls
``network(inputs)`` (nerf/render.py:73).  The B200 path instead reads the weights of a known
architecture and evaluates the whole MLP inside one fused CUDA kernel, so it has to recognise
the model.  Recognition is structural (state-dict keys), which means the *reference's own*
``NeRF`` (nerf/nerf.py:52-94) and ``FilmSirenNeRF`` (pi_GAN/modules.py:70-118) instances and
checkpoints work unchanged, and so do the stand-alone classes below (same keys, same
initialisation order, so ``torch.manual_seed(s); NeRF()`` gives bit-identical weights to the
reference class -- pinned by tests/golden/weights_sha.json).

Nothing here computes an MLP in PyTorch: ``forward`` goes to the CUDA extension.
"""
from __future__ import annotations

import math

import numpy as np
import torch

# ---- canonical flat fp32 parameter layout (must match csrc/layout.h) -------------------------
NERF_KEYS = (
    [(f"layers_pos.{i}", s) for i, s in enumerate(
        [(256, 60), (256, 256), (256, 256), (256, 256), (256, 256), (256, 316), (256, 256), (256, 256)])]
    + [("layers_dir.0", (256, 256)), ("layers_dir.1", (128, 280)),
       ("output_layer_sigma", (1, 256)), ("output_layer_rgb", (3, 128))]
)
FILM_KEYS_DIR = (
    [("input_layer", (256, 3))]
    + [(f"hidden_layers.{i}", (256, 256)) for i in range(7)]
    + [("output_layer_sigma.0", (1, 256)), ("hidden_layer_rgb", (256, 259)), ("output_layer_rgb.0", (3, 256))]
)
FILM_KEYS_NODIR = FILM_KEYS_DIR[:9] + [("hidden_layer_rgb", (256, 256)), ("output_layer_rgb.0", (3, 256))]


def _numel(keys):
    return sum(o * i + o for _, (o, i) in keys)


# SirenNeRF (nerf/nerf.py:120-170): same topology as NeRF with sin(30 (W x + b)) layers and raw 3-d inputs
SIREN_KEYS = (
    [(f"layers_pos.{i}", s) for i, s in enumerate(
        [(256, 3), (256, 256), (256, 256), (256, 256), (256, 256), (256, 259), (256, 256), (256, 256)])]
    + [("layers_dir.0", (256, 256)), ("layers_dir.1", (128, 259)),
       ("output_layer_sigma", (1, 256)), ("output_layer_rgb", (3, 128))]
)

NERF_NUMEL = _numel(NERF_KEYS)          # 593,924  (SURVEY.md 2.1 #3)
FILM_NUMEL = _numel(FILM_KEYS_DIR)      # 529,156  (SURVEY.md 2.1 #5)
SIREN_NUMEL = _numel(SIREN_KEYS)        # 562,052

KIND_NERF = 0
KIND_FILM = 1
KIND_SIREN = 2


def model_kind(model) -> int:
    """Structural dispatch; anything else is a TypeError (no fallback by design, SURVEY 8b)."""
    if hasattr(model, "module") and isinstance(model, torch.nn.DataParallel):
        model = model.module
    if all(hasattr(model, a) for a in ("layers_pos", "layers_dir", "output_layer_sigma", "output_layer_rgb")):
        w0 = model.layers_pos[0].weight
        if tuple(w0.shape) == (256, 60):
            return KIND_NERF
        if tuple(w0.shape) == (256, 3):
            return KIND_SIREN
        raise TypeError("NeRF-shaped model with an unknown first layer %s" % (tuple(w0.shape),))
    if all(hasattr(model, a) for a in ("input_layer", "hidden_layers", "hidden_layer_rgb", "output_layer_rgb")):
        return KIND_FILM
    raise TypeError(
        f"{type(model).__name__} is not a NeRF / FilmSirenNeRF radiance field; the B200 render path "
        "evaluates known architectures in a fused kernel and has no generic-callable fallback")


def param_list(model, kind: int | None = None):
    """Parameters in canonical flat order (weight, bias per layer)."""
    kind = model_kind(model) if kind is None else kind
    sd = dict(model.named_parameters())
    if kind == KIND_NERF:
        keys = NERF_KEYS
    elif kind == KIND_SIREN:
        keys = SIREN_KEYS
    else:
        keys = FILM_KEYS_DIR if getattr(model, "use_dir", True) else FILM_KEYS_NODIR
    out = []
    for name, (o, i) in keys:
        w, b = sd[name + ".weight"], sd[name + ".bias"]
        if tuple(w.shape) != (o, i) or tuple(b.shape) != (o,):
            raise TypeError(f"{name}: expected weight {(o, i)}, got {tuple(w.shape)}")
        out += [w, b]
    return out


def flat_params(model, kind: int | None = None) -> torch.Tensor:
    """One flat fp32 tensor of all parameters (differentiable: grads flow back to each
    nn.Parameter through torch.cat's backward; the flat layout is also the all-reduce bucket)."""
    ps = param_list(model, kind)
    return torch.cat([p.reshape(-1) for p in ps]).float()


def film_tensor(model) -> torch.Tensor:
    """[9,512] gamma||beta tensor from the ``film_params`` list set by set_film_params
    (pi_GAN/modules.py:96-99).  Raises ValueError when unset, like the reference (:107)."""
    fp = getattr(model, "film_params", None)
    if fp is None:
        raise ValueError("film_params not set")
    if isinstance(fp, torch.Tensor):
        return fp
    return torch.stack([torch.cat([g, b]) for (g, b) in fp])


# ---- stand-alone model classes (same keys / init order as the reference) ---------------------
class _Dense(torch.nn.Linear):
    """Linear + named activation, Xavier-uniform with the activation's gain, zero bias
    (nerf/nerf.py:5-28)."""

    def __init__(self, i, o, activation="linear"):
        self.activation_name = activation
        super().__init__(i, o)

    def reset_parameters(self):
        torch.nn.init.xavier_uniform_(self.weight, gain=torch.nn.init.calculate_gain(self.activation_name))
        torch.nn.init.zeros_(self.bias)


class NeRF(torch.nn.Module):
    """8x256 ReLU trunk with posenc(L=10/4); parameter names as nerf/nerf.py:52-73."""

    def __init__(self):
        super().__init__()
        dims = [(60, 256)] + [(256, 256)] * 4 + [(316, 256)] + [(256, 256)] * 2
        self.layers_pos = torch.nn.ModuleList([_Dense(i, o, "relu") for i, o in dims])
        self.layers_dir = torch.nn.ModuleList([_Dense(256, 256, "linear"), _Dense(280, 128, "relu")])
        self.output_layer_sigma = _Dense(256, 1, "relu")
        self.output_layer_rgb = _Dense(128, 3, "sigmoid")

    def forward(self, x):
        from . import ops
        return ops.mlp(self, x=x)


class _Siren(torch.nn.Linear):
    """Linear layer whose output goes through sin(30 x) (nerf/nerf.py:97-117): U(+-sqrt(6/in)/30) weights, zero bias."""

    def reset_parameters(self):
        torch.nn.init.uniform_(self.weight, -np.sqrt(6 / self.in_features) / 30, np.sqrt(6 / self.in_features) / 30)
        torch.nn.init.zeros_(self.bias)


class SirenNeRF(torch.nn.Module):
    """NeRF topology with SIREN layers and raw (un-encoded) inputs; parameter names and init order as
    nerf/nerf.py:120-150 (selected by `use_siren`, nerf/train_nerf.py:89-91)."""

    def __init__(self):
        super().__init__()
        dims = [(3, 256)] + [(256, 256)] * 4 + [(259, 256)] + [(256, 256)] * 2
        self.layers_pos = torch.nn.ModuleList([_Siren(i, o) for i, o in dims])
        torch.nn.init.uniform_(self.layers_pos[0].weight, -1 / 30, 1 / 30)            # nerf.py:135
        self.layers_dir = torch.nn.ModuleList([_Dense(256, 256, "linear"), _Siren(259, 128)])
        self.output_layer_sigma = _Dense(256, 1, "relu")
        self.output_layer_rgb = _Dense(128, 3, "sigmoid")

    def forward(self, x):
        from . import ops
        return ops.mlp(self, x=x)


class _FilmSiren(torch.nn.Module):
    """Parameter holder for one FiLM-SIREN layer (pi_GAN/modules.py:8-31 init)."""

    def __init__(self, i, o, c=6, w_0=30, is_first_layer=False):
        super().__init__()
        self.weight = torch.nn.Parameter(torch.zeros(o, i))
        self.bias = torch.nn.Parameter(torch.zeros(o))
        wr = 1 / i if is_first_layer else np.sqrt(c / i) / w_0
        br = np.sqrt(1 / i)
        torch.nn.init.uniform_(self.weight, -wr, wr)
        torch.nn.init.uniform_(self.bias, -br, br)


class FilmSirenNeRF(torch.nn.Module):
    """FiLM-conditioned SIREN field; names as pi_GAN/modules.py:70-94."""

    def __init__(self, hidden_dim=256, hidden_layers=8, c=6, w_0=30, use_dir=True):
        super().__init__()
        assert hidden_dim == 256 and hidden_layers == 8 and w_0 == 30, "fused kernel is specialised to 8x256, w0=30"
        self.use_dir = use_dir
        self.film_params = None
        self.input_layer = _FilmSiren(3, 256, c, w_0, True)
        self.hidden_layers = torch.nn.ModuleList([_FilmSiren(256, 256, c, w_0) for _ in range(7)])
        self.output_layer_sigma = torch.nn.Sequential(torch.nn.Linear(256, 1), torch.nn.ReLU())
        self.hidden_layer_rgb = _FilmSiren(259 if use_dir else 256, 256, c, w_0)
        self.output_layer_rgb = torch.nn.Sequential(torch.nn.Linear(256, 3), torch.nn.Sigmoid())
        self.n_layers = 7

    def set_film_params(self, mapping_tensor):
        self.film_params = [torch.chunk(mapping_tensor[i], 2) for i in range(mapping_tensor.shape[0])]

    def forward(self, x, film_params=None):
        if film_params is not None:
            self.film_params = film_params
        elif self.film_params is None:
            raise ValueError
        from . import ops
        return ops.mlp(self, x=x)


class MappingNetwork(torch.nn.Module):
    """z -> film_params[B,9,512] (gamma || beta per FiLM layer); module names, creation order (= RNG consumption) and the
    gamma = 1 / beta = 0 head-bias init of pi_GAN/modules.py:34-68.  B x 256 GEMMs: stays on cuBLAS (SURVEY 8f rank 2); the
    nine heads run as ONE GEMM on the concatenated weights."""

    def __init__(self, input_dim=256, output_dim=256, output_layers=8, hidden_dim=256, hidden_layers=3):
        super().__init__()
        self.input_layer = torch.nn.Sequential(torch.nn.Linear(input_dim, hidden_dim), torch.nn.LeakyReLU(0.2))
        hidden = []
        for _ in range(hidden_layers - 1):
            hidden += [torch.nn.Linear(hidden_dim, hidden_dim), torch.nn.LeakyReLU(0.2)]
        self.hidden_layers = torch.nn.Sequential(*hidden)
        heads = [torch.nn.Linear(hidden_dim, 2 * output_dim) for _ in range(output_layers + 1)]
        with torch.no_grad():
            for head in heads:
                head.bias[:output_dim] = 1
                head.bias[output_dim:] = 0
        self.output_layers = torch.nn.ModuleList(heads)

    def forward(self, input_tensor):
        h = self.hidden_layers(self.input_layer(input_tensor))
        w = torch.cat([head.weight for head in self.output_layers])
        b = torch.cat([head.bias for head in self.output_layers])
        return torch.nn.functional.linear(h, w, b).reshape(h.shape[0], len(self.output_layers), -1)


class Renderer:
    """Camera / sampling settings + the render call of pi_GAN/modules.py:120-161 (poses drawn with np.random like the reference)."""

    def __init__(self, width, height, near=0.1, far=1.9, fov=12, coarse_samples=64, fine_samples=128, horizontal_std=0.3,
                 vertical_std=0.15):
        self.width, self.height, self.fov = width, height, fov
        self.focal = width / 2 / np.tan(fov / 2 * np.pi / 180)
        self.near, self.far = near, far
        self.coarse_samples, self.fine_samples = coarse_samples, fine_samples
        self.horizontal_std, self.vertical_std = horizontal_std, vertical_std

    def set_params(self, width=None, height=None, near=None, far=None, fov=None, coarse_samples=None, fine_samples=None,
                   horizontal_std=None, vertical_std=None):
        refocus = width is not None or fov is not None
        for name, v in (("width", width), ("height", height), ("near", near), ("far", far), ("fov", fov), ("coarse_samples", coarse_samples),
                        ("fine_samples", fine_samples), ("horizontal_std", horizontal_std), ("vertical_std", vertical_std)):
            if v is not None:
                setattr(self, name, v)
        if refocus:
            self.focal = self.width / 2 / np.tan(self.fov / 2 * np.pi / 180)

    def draw_pose(self, theta=None, phi=None):
        """(theta, phi) ~ N(0, std) in the reference's draw order (theta first), then the camera matrix."""
        from . import pigan_render
        theta = np.random.randn() * self.horizontal_std if theta is None else theta
        phi = np.random.randn() * self.vertical_std if phi is None else phi
        return pigan_render.camera_pos_to_transform_matrix(1, theta, phi)

    def __call__(self, model, theta=None, phi=None):
        from . import pigan_render
        return pigan_render.render_image(self.width, self.height, self.focal, self.draw_pose(theta, phi), self.near, self.far, model, model,
                                         self.coarse_samples, self.fine_samples)


class Generator(torch.nn.Module):
    """pi-GAN generator (pi_GAN/modules.py:164-197): same constructor, sub-module names and state-dict keys.  forward() maps
    z[B,input_dim] to film_params and renders ALL B latents through pigan_render.render_batch -- one launch sequence, with the
    autograd graph to the FiLM-SIREN weights and, through film_params, to the mapping network -- instead of the reference's
    per-latent Python loop; poses and jitter are drawn in the reference's order."""

    def __init__(self, input_dim, output_size, near=0.1, far=1.9, fov=12, coarse_samples=64, fine_samples=128, horizontal_std=0.3,
                 vertical_std=0.15, use_dir=True):
        super().__init__()
        self.input_dim = input_dim
        self.film_siren_nerf = FilmSirenNeRF(use_dir=use_dir)
        self.mapping_network = MappingNetwork(input_dim=input_dim)
        self.renderer = Renderer(output_size, output_size, near, far, fov, coarse_samples, fine_samples, horizontal_std, vertical_std)

    def forward(self, input_tensor, *, poses=None, t_rand=None, precision=None):
        """poses / t_rand[B, H*W, coarse_samples] / precision: keyword-only additions (parity runs pass the jitter tensor)."""
        from . import pigan_render
        film_params = self.mapping_network(input_tensor)
        r = self.renderer
        if poses is None:
            poses = [r.draw_pose() for _ in range(film_params.shape[0])]
        return pigan_render.render_batch(self.film_siren_nerf, film_params, poses, r.width, r.height, r.focal, r.near, r.far,
                                         r.coarse_samples, r.fine_samples, t_rand=t_rand, precision=precision)

    def get_mapping(self, input_tensor):
        return self.mapping_network(input_tensor)

    def set_film_params(self, film_params):
        self.film_siren_nerf.set_film_params(film_params)

    def set_resolution(self, resolution):
        self.renderer.set_params(width=resolution, height=resolution)

    def render(self, theta=None, phi=None):
        return self.renderer(self.film_siren_nerf, theta, phi)


def damp_nerf_(model: NeRF) -> NeRF:
    """'Trained-like' 1/f synthetic field used for end-to-end parity (SURVEY.md 8d): scale the
    posenc band i columns by 2^-i, sigma head x8, sigma bias -1."""
    with torch.no_grad():
        for i in range(10):
            s = 2.0 ** (-i)
            model.layers_pos[0].weight[:, 6 * i:6 * i + 6] *= s
            model.layers_pos[5].weight[:, 6 * i:6 * i + 6] *= s
        for i in range(4):
            model.layers_dir[1].weight[:, 256 + 6 * i:256 + 6 * i + 6] *= 2.0 ** (-i)
        model.output_layer_sigma.weight *= 8.0
        model.output_layer_sigma.bias.fill_(-1.0)
    return model
