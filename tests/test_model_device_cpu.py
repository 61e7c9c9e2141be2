"""Models whose parameters are on the CPU are refused before anything is launched (no GPU and no libb2r.so needed)."""
import pytest
import torch

from msra_practice_project_b200 import models, nerf_render, ops


def test_cpu_model_is_refused():
    nerf, film_model = models.NeRF(), models.FilmSirenNeRF()
    film, rays, z = torch.zeros(2, 9, 512), torch.zeros(2, 2, 3), torch.zeros(2, 512)
    calls = [lambda: ops.mlp(nerf, x=torch.zeros(4, 6)),
             lambda: ops.mlp_film_batched(film_model, film, rays, z, 512),
             lambda: ops.mlp_film_batched_train(film_model, film, rays, z, 512),
             lambda: nerf_render.density_lattice(nerf, N=8),
             lambda: nerf_render.create_mesh(nerf, None, 8, narrow_band=4)]
    for call in calls:
        with pytest.raises(RuntimeError, match="CUDA device"):
            call()
