"""The nerf2mesh.py hot loop on the GPU: density-grid query (nerf2mesh.py:27-40,69-87) and marching cubes
(nerf2mesh.py:98, third-party torchmcubes in the reference) -- and, beyond the reference, the finished mesh: vertices in
world coordinates with analytic normals and the field's colours (`extract_mesh`), written as binary PLY (`write_ply`).

`density_grid` never materialises the res^3 x 3 position tensor on the host: positions are generated on the
device per chunk with numpy-1.23 linspace semantics (float64, end point pinned) and rounded to fp16 exactly
like `grid.to(torch.float16)`.  Slab sharding across ranks = one contiguous range of the flat grid per rank
(axis 0 of density[i,j,k], i.e. the y coordinate under meshgrid's 'xy' indexing).
"""
from __future__ import annotations

from typing import NamedTuple, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import ops
from ._lib import HBR_MC_BRICK
from .encoder import PositionalEncoder
from .hash_encoding import HashEncoder
from .test_hash import MLP_3D


def _unwrap(m):
    return m.module if isinstance(m, nn.DataParallel) else m


def view_dir_encoding(dir_encoder: PositionalEncoder, device) -> torch.Tensor:
    """PositionalEncoder((0,0,1) in fp16) as fp32 values (nerf2mesh.py:69-70,81): one row for every grid point."""
    v = torch.zeros((1, 3), device=device, dtype=torch.float16)
    v[..., 2] = 1.0
    return ops.dir_encode(v, dir_encoder.max_seq_len)


def density_grid(encoder: HashEncoder, nerf, dir_encoder: Optional[PositionalEncoder], min_bound, max_bound, res: int,
                 i_begin: int = 0, i_end: Optional[int] = None, chunk: int = 1 << 19, cuda_core_mlp: bool = False) -> torch.Tensor:
    """Field values on planes [i_begin, i_end) of the res^3 grid.

    With a dir_encoder: (planes, res, res, 4) = [rgb, density], the layout nerf2mesh.py:86-87 saves to
    density_grid_w_rgb.npy.  With dir_encoder=None: (planes, res, res) density only (all marching cubes needs,
    nerf2mesh.py:95)."""
    mlp = _unwrap(nerf)
    if not isinstance(encoder, HashEncoder) or not isinstance(mlp, MLP_3D):
        raise TypeError("density_grid needs the native HashEncoder and MLP_3D")
    mlp._check_native()
    i_end = res if i_end is None else i_end
    table = encoder._flat_table()
    if not table.is_cuda:
        raise RuntimeError("density_grid needs the encoder on a CUDA device (there is no CPU fallback)")
    p0, count = i_begin * res * res, (i_end - i_begin) * res * res
    denc = view_dir_encoding(dir_encoder, table.device) if dir_encoder is not None else None
    with torch.no_grad():
        out = ops.grid_density([float(v) for v in min_bound], [float(v) for v in max_bound], res, p0, count, table,
                               encoder._geom(), mlp._flat_params(), mlp._dims(), denc, chunk=chunk, cuda_core_mlp=cuda_core_mlp)
    return out.view((i_end - i_begin, res, res, 4) if denc is not None else (i_end - i_begin, res, res))


def marching_cubes_counts(density: torch.Tensor, iso: float, i_begin: int = 0, i_end: Optional[int] = None) -> Tuple[int, int]:
    """(vertices, triangles) owned by planes [i_begin, i_end): welded vertices = iso-crossing grid edges."""
    c = ops.mc_count(density, iso, i_begin, i_end).tolist()
    return int(c[0]), int(c[1])


def marching_cubes(density: torch.Tensor, iso: float):
    """torchmcubes.marching_cubes-shaped call (nerf2mesh.py:98): (verts (V,3) fp32 in grid-index coordinates along
    axes (0,1,2), faces (F,3) int32).  Inside test: density < iso.  One welded vertex per crossing edge."""
    nv, nt = marching_cubes_counts(density, iso)
    verts, faces, _ = ops.mc_emit(density, iso, nv, nt)
    return verts, faces


def _device_for(t: torch.Tensor) -> torch.device:
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise RuntimeError("marching cubes / grid_interp run on a CUDA device (there is no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def marching_cubes_xyz(vol: torch.Tensor, iso: float):
    """torchmcubes.marching_cubes as nerf2mesh.py:95-98 calls it: `vol` may live on the CPU (it does there) -- it is
    uploaded, meshed on the GPU and the result returned on vol's device.  Vertices are (x, y, z) = (index along axis 2,
    axis 1, axis 0), torchmcubes' order for a volume indexed [z, y, x]; faces (F,3) int32."""
    dev = _device_for(vol)
    d = vol.detach().to(dev, torch.float32).contiguous()
    with torch.cuda.device(dev):
        verts, faces = marching_cubes(d, iso)
        verts = verts.flip(-1).contiguous()
    return verts.to(vol.device), faces.to(vol.device)


def grid_interp(vol: torch.Tensor, points: torch.Tensor) -> torch.Tensor:
    """torchmcubes.grid_interp (nerf2mesh.py:99): vol (C,Nz,Ny,Nx) or (Nz,Ny,Nx), points (V,3) as (x,y,z) -> (V,C)."""
    dev = _device_for(vol if vol.is_cuda else points)
    v = vol.detach().to(dev, torch.float32)
    if v.dim() == 3:
        v = v[None]
    with torch.cuda.device(dev):
        out = ops.grid_interp(v.contiguous(), points.detach().to(dev, torch.float32).contiguous())
    return out.to(points.device)


# ---------------------------------------------------------------------------------------------------------------
# the finished mesh: world coordinates, analytic normals, the field's colours, binary PLY
# ---------------------------------------------------------------------------------------------------------------
class Mesh(NamedTuple):
    """Device tensors (CPU tensors when read back by `read_ply`): vertices (V,3) fp32 world coordinates, faces (F,3) int32
    counter-clockwise seen from outside, normals (V,3) fp32 outward unit vectors (0 where the field is flat), colors (V,3)
    fp32 raw ELU output of the colour head (uint8 after `read_ply`)."""
    vertices: torch.Tensor
    faces: torch.Tensor
    normals: torch.Tensor
    colors: torch.Tensor


def _native_field(encoder, nerf):
    mlp = _unwrap(nerf)
    if not isinstance(encoder, HashEncoder) or not isinstance(mlp, MLP_3D):
        raise TypeError("needs the native HashEncoder and MLP_3D")
    mlp._check_native()
    table = encoder._flat_table()
    if not table.is_cuda:
        raise RuntimeError("the field runs on a CUDA device (there is no CPU fallback)")
    return table, encoder._geom(), mlp._flat_params(), mlp._dims()


def _density_and_grad(x, table, geom, params, dims):
    """fp32 kernels, no autograd graph: features, density (n,) and d density / dx (n,3) at positions x (n,3) fp32."""
    feat = ops.hash_encode_fwd(x, table, geom)
    dens, act = ops.mlp_fwd_f32(feat, None, 1, params, dims, keep_act=True)
    ones = torch.ones((x.shape[0],), device=x.device, dtype=torch.float32)
    # density-only backward with dparams=None: d density / d features, no weight-gradient kernel (LeakyReLU' included)
    dfeat, _ = ops.mlp_bwd_f32(feat, None, 1, params, dims, ones, act, True, False, None)
    return feat, dens[:, 0], ops.hash_encode_dx(x, table, geom, dfeat)


def field_gradient(encoder: HashEncoder, nerf, x: torch.Tensor, chunk: int = 1 << 20) -> Tuple[torch.Tensor, torch.Tensor]:
    """(density (N,), grad (N,3)): the density head's LeakyReLU output and its analytic gradient with respect to the fp32
    world positions x (N,3), by hash_encode_fwd -> density-only mlp_fwd_f32 -> mlp_bwd_f32 (d out = 1) ->
    hash_encode_dx.  fp32 kernels only, no autograd graph; `chunk` points per pass bound the (act_rows x chunk)
    activation buffer."""
    table, geom, params, dims = _native_field(encoder, nerf)
    x = x.detach().to(table.device, torch.float32).contiguous()
    n = x.shape[0]
    dens = torch.empty((n,), device=x.device, dtype=torch.float32)
    grad = torch.empty((n, 3), device=x.device, dtype=torch.float32)
    with torch.no_grad():
        for s in range(0, n, chunk):
            _, d, g = _density_and_grad(x[s:s + chunk], table, geom, params, dims)
            dens[s:s + chunk] = d
            grad[s:s + chunk] = g
    return dens, grad


def vertex_attributes(encoder: HashEncoder, nerf, dir_encoder: PositionalEncoder, x: torch.Tensor,
                      chunk: int = 1 << 20) -> Tuple[torch.Tensor, torch.Tensor]:
    """(normals (N,3), colors (N,3)) at world positions x: n = -grad/|grad| (outward: the object is where the density is
    high; (0,0,0) where grad = 0), colours = the full fp32 field's raw RGB seen head-on, i.e. with the view direction
    d = -n (the direction a ray travels into the surface; (0,0,1), nerf2mesh's direction, where n = 0) encoded by
    dir_encode as training encodes rays_d, one direction row per vertex.  One hash-grid pass per chunk serves both."""
    table, geom, params, dims = _native_field(encoder, nerf)
    x = x.detach().to(table.device, torch.float32).contiguous()
    n = x.shape[0]
    normals = torch.empty((n, 3), device=x.device, dtype=torch.float32)
    colors = torch.empty((n, 3), device=x.device, dtype=torch.float32)
    with torch.no_grad():
        for s in range(0, n, chunk):
            feat, _, g = _density_and_grad(x[s:s + chunk], table, geom, params, dims)
            nrm = torch.linalg.vector_norm(g, dim=1, keepdim=True)
            flat = nrm == 0
            unit = g / torch.where(flat, torch.ones_like(nrm), nrm)
            normals[s:s + chunk] = -unit
            d = torch.where(flat, unit.new_tensor([0.0, 0.0, 1.0]), unit)
            out, _ = ops.mlp_fwd_f32(feat, ops.dir_encode(d, dir_encoder.max_seq_len), 1, params, dims, keep_act=False)
            colors[s:s + chunk] = out[:, :3]
    return normals, colors


def world_axes(min_bound, max_bound, res: int, device=None) -> torch.Tensor:
    """(3, res) fp32: per INDEX axis (0: y, 1: x, 2: z, formats.grid_axes) the fp16-rounded linspace coordinates the density
    grid was evaluated at (grid_points_kernel)."""
    from .formats import grid_axes
    ax = grid_axes([float(v) for v in min_bound], [float(v) for v in max_bound], res)
    return torch.from_numpy(np.stack(ax).astype(np.float16).astype(np.float32)).to(device)


def index_to_world(verts: torch.Tensor, axes: torch.Tensor) -> torch.Tensor:
    """Marching-cubes vertices (V,3) in grid-index units along axes (0,1,2) -> (V,3) world (x, y, z).  Each index axis maps
    through its own table q = axes[a] (world_axes): a fractional index a goes to q[floor a] + (a - floor a)(q[floor a + 1]
    - q[floor a]), so the vertices sit on the field the grid actually sampled.  Index axis 0 is y, axis 1 is x."""
    res = axes.shape[1]
    a = verts.to(axes.device, torch.float32).T                            # (3,V)
    i0 = a.floor().clamp_(0, max(res - 2, 0)).long()
    lo = torch.gather(axes, 1, i0)
    hi = torch.gather(axes, 1, (i0 + 1).clamp_(max=res - 1))
    w = lo + (a - i0) * (hi - lo)
    return torch.stack((w[1], w[0], w[2]), dim=1).contiguous()


# ---------------------------------------------------------------------------------------------------------------
# sparse marching cubes: the same res^3 grid, evaluated and meshed only in the 8^3-cell bricks the surface passes through
# ---------------------------------------------------------------------------------------------------------------
class SparseSurface(NamedTuple):
    """vertices (V,3) fp32 grid-index coordinates and faces (F,3) int32 in marching_cubes' conventions; bricks (n,) int32:
    the active bricks in slot order (closure round by round, brick-index order within a round); rounds: field
    evaluations of brick lists (seeds included); points: field values used ((nb+1)^3 coarse + 729 per active brick)."""
    vertices: torch.Tensor
    faces: torch.Tensor
    bricks: torch.Tensor
    rounds: int
    points: int


def select_bricks(coarse: torch.Tensor, iso: float, brick_density):
    """Seed and close the active brick set.  coarse: the (nb+1)^3 coarse-lattice values; brick_density(bricks) -> (n,9,9,9)
    values of the listed bricks.  Seeds are the bricks whose 8 corner values straddle iso; each round evaluates the bricks
    activated by the last one and activates the face neighbours across every interior 9x9 boundary plane that straddles
    iso, until no brick is added.  Returns (brick map (nb,nb,nb) int32: slot or -1, bricks in slot order, their values
    (n,9,9,9), rounds)."""
    bmap = ops.brick_seed(coarse, iso)
    lists, dens, rounds, base = [], [], 0, 0
    while True:
        lst = ops.brick_compact(bmap, base)
        if lst.shape[0] == 0:
            break
        d = brick_density(lst)
        ops.brick_closure(d, lst, bmap, iso)
        lists.append(lst)
        dens.append(d)
        base += lst.shape[0]
        rounds += 1
    P = HBR_MC_BRICK + 1
    if not lists:
        return bmap, torch.empty((0,), device=bmap.device, dtype=torch.int32), \
            torch.empty((0, P, P, P), device=bmap.device, dtype=torch.float32), 0
    return bmap, torch.cat(lists), torch.cat(dens), rounds


def sparse_surface_index(res: int, iso: float, coarse: torch.Tensor, brick_density) -> SparseSurface:
    """Sparse marching cubes of the res^3 grid whose values at the coarse lattice are `coarse` and on bricks
    `brick_density(bricks)` gives (select_bricks): seed, closure rounds, then one welded vertex per crossing edge of the
    active bricks' cells.  The result equals marching_cubes of the dense grid restricted to those cells; it is the dense
    mesh when every crossing cell lies in an active brick.  A surface component that crosses no coarse-lattice edge of a
    brick and never reaches a seeded brick through crossing boundary planes is not meshed.  Vertex and face order is a
    deterministic function of the brick list."""
    if res < 2:
        raise ValueError(f"res {res} < 2")
    if tuple(coarse.shape) != (ops.brick_count(res) + 1,) * 3:
        raise ValueError(f"coarse lattice {tuple(coarse.shape)} does not match res {res}")
    bmap, bricks, dens, rounds = select_bricks(coarse, iso, brick_density)
    verts, faces = ops.brick_mc(dens, bricks, bmap, res, iso)
    return SparseSurface(verts, faces, bricks, rounds, coarse.numel() + dens.numel())


def sparse_field_surface(encoder: HashEncoder, nerf, min_bound, max_bound, res: int, iso: float, chunk: int = 1 << 19,
                         cuda_core_mlp: bool = False) -> SparseSurface:
    """sparse_surface_index on the field: coarse lattice and bricks evaluated with density_grid's positions, encoder and
    density head, so every value equals density_grid's at the same grid index."""
    table, geom, params, dims = _native_field(encoder, nerf)
    mn, mx = [float(v) for v in min_bound], [float(v) for v in max_bound]
    with torch.no_grad():
        coarse = ops.coarse_density(mn, mx, res, table, geom, params, dims, chunk, cuda_core_mlp)
        return sparse_surface_index(res, iso, coarse, lambda b: ops.brick_density(mn, mx, res, b, table, geom, params, dims,
                                                                                  chunk, cuda_core_mlp))


# ---------------------------------------------------------------------------------------------------------------
# floaters: connected components of a mesh, and keeping the ones that matter
# ---------------------------------------------------------------------------------------------------------------
class MeshComponents(NamedTuple):
    """labels (V,) int32: the smallest vertex index of each vertex's component; roots (C,) int64: the components' root
    indices (labels[r] == r), ascending; faces / vertices (C,) int64: each component's face and vertex count, in roots'
    order (a face belongs to the component of its first vertex)."""
    labels: torch.Tensor
    roots: torch.Tensor
    faces: torch.Tensor
    vertices: torch.Tensor


def mesh_components(faces: torch.Tensor, nv: int) -> MeshComponents:
    """Connected components of the mesh whose (F,3) faces index nv vertices (hbr_mesh_components on the GPU): two vertices
    are connected when a chain of faces joins them; a vertex no face uses is a component of its own."""
    labels, face_count, vertex_count = ops.mesh_components(faces, nv)
    roots = torch.nonzero(vertex_count).squeeze(1)             # every root counts itself; every other index holds 0
    return MeshComponents(labels, roots, face_count[roots].long(), vertex_count[roots].long())


def keep_components(comp: MeshComponents, min_faces: int = 0, largest: Optional[int] = None) -> torch.Tensor:
    """bool (C,): the components with >= min_faces faces that are, when largest = k is given, also among the k largest by
    face count.  Every component tied with the k-th largest count is kept, so the choice depends on the mesh as a set, not
    on its vertex order.  The defaults keep everything."""
    keep = comp.faces >= min_faces
    if largest is not None:
        if largest < 1:
            raise ValueError(f"largest = {largest}: keep at least one component (or pass None)")
        if largest < comp.faces.shape[0]:
            keep &= comp.faces >= torch.topk(comp.faces, largest).values[-1]
    return keep


def filter_surface(vertices: torch.Tensor, faces: torch.Tensor, keep_vertex: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Stable compaction of a mesh to the vertices where keep_vertex (V,) bool holds and the faces whose three vertices are
    all kept: (vertex_index (V',) int64 -- the kept vertices' rows of `vertices`, ascending -- and the kept faces (F',3)
    int32 re-indexed to them, in their original order)."""
    if tuple(keep_vertex.shape) != (vertices.shape[0],) or keep_vertex.dtype != torch.bool:
        raise ValueError(f"keep_vertex must be ({vertices.shape[0]},) bool, got {tuple(keep_vertex.shape)} {keep_vertex.dtype}")
    faces = faces.to(torch.int32)
    new_id = torch.cumsum(keep_vertex, 0, dtype=torch.int32) - 1            # V <= 2^31 - 1 (hbr_mesh_components)
    kept = faces[keep_vertex.index_select(0, faces.reshape(-1)).view(-1, 3).all(1)]
    return torch.nonzero(keep_vertex).squeeze(1), new_id.index_select(0, kept.reshape(-1)).view(-1, 3)


def filter_by_components(vertices: torch.Tensor, faces: torch.Tensor, min_faces: int = 0, largest: Optional[int] = None):
    """mesh_components -> keep_components -> filter_surface: (vertex_index, faces', the components, their keep mask)."""
    comp = mesh_components(faces, vertices.shape[0])
    keep = keep_components(comp, min_faces, largest)
    keep_root = torch.zeros((vertices.shape[0],), device=faces.device, dtype=torch.bool)
    keep_root[comp.roots[keep]] = True
    vertex_index, faces = filter_surface(vertices, faces, keep_root.index_select(0, comp.labels))
    return vertex_index, faces, comp, keep


def filter_components(m: Mesh, min_faces: int = 0, largest: Optional[int] = None) -> Mesh:
    """The mesh without its floaters: the components keep_components keeps, compacted stably (filter_surface).  Positions,
    normals and colours of the kept vertices are gathered, so each stays bitwise what it was."""
    vi, faces, _, _ = filter_by_components(m.vertices, m.faces, min_faces, largest)
    return Mesh(m.vertices[vi], faces, m.normals[vi], m.colors[vi])


def extract_mesh(encoder: HashEncoder, nerf, dir_encoder: PositionalEncoder, min_bound, max_bound, res: int = 256,
                 iso: float = 30.0, chunk: int = 1 << 20, sparse: bool = False, min_component_faces: int = 0,
                 largest_components: Optional[int] = None) -> Mesh:
    """Checkpoint -> oriented, coloured, world-space mesh: density_grid (density only, the tensor-core path) ->
    marching_cubes -> index_to_world and the winding swap -> normals and colours at the world vertices
    (vertex_attributes).

    sparse=True replaces density_grid + marching_cubes by sparse_field_surface: the same grid, evaluated and meshed only in
    the 8^3-cell bricks reached from the coarse lattice's crossings (memory and time follow the surface, not res^3).  It
    gives the dense mesh whenever every crossing cell lies in an active brick, and drops a component that fits inside one
    brick without crossing a coarse-lattice edge and never touches a seeded brick.  Its vertex and face order is
    deterministic.

    min_component_faces / largest_components drop floaters (keep_components' rule) right after marching cubes, in grid-index
    space, so no attribute work is spent on them; the result equals filter_components of the unfiltered mesh.  With the
    defaults no labelling runs.

    Conventions:
    * World mapping: index axis 0 is y, 1 is x, 2 is z; each axis maps through fp16(linspace(min, max, res)), the
      coordinates the grid was evaluated at, linearly between grid points.
    * Normals are outward, n = -grad sigma / |grad sigma| (the object is sigma > iso); (0,0,0) where grad sigma = 0.
    * Winding: counter-clockwise seen from outside, in world coordinates (world_surface: the index -> world permutation
      swaps x and y and so reverses the tables' handedness; two columns of the faces are swapped).
    * Colours: the field's raw RGB (ELU output, not clamped) seen head-on, view direction -n ((0,0,1) where n = 0).
    * Order: vertex and face order follow hbr_mc_emit's atomic cursors and are NOT stable across runs; every per-vertex
      value is a deterministic function of the vertex position."""
    if sparse:
        vidx, faces = sparse_field_surface(encoder, nerf, min_bound, max_bound, res, iso)[:2]
    else:
        dens = density_grid(encoder, nerf, None, min_bound, max_bound, res)
        vidx, faces = marching_cubes(dens, iso)
        del dens
    if min_component_faces > 0 or largest_components is not None:
        vi, faces, _, _ = filter_by_components(vidx, faces, min_component_faces, largest_components)
        vidx = vidx[vi]
    return index_surface_mesh(encoder, nerf, dir_encoder, vidx, faces, min_bound, max_bound, res, chunk)


def index_surface_mesh(encoder: HashEncoder, nerf, dir_encoder: PositionalEncoder, vidx: torch.Tensor, faces: torch.Tensor,
                       min_bound, max_bound, res: int, chunk: int = 1 << 20) -> Mesh:
    """extract_mesh's steps after marching cubes, for a surface in grid-index coordinates of the res^3 grid (marching_cubes'
    or sparse_surface_index's conventions): index_to_world, the winding swap, normals and colours."""
    verts, faces = _index_to_world_surface(vidx, faces, min_bound, max_bound, res)
    normals, colors = vertex_attributes(encoder, nerf, dir_encoder, verts, chunk)
    return Mesh(verts, faces, normals, colors)


def world_surface(density: torch.Tensor, iso: float, min_bound, max_bound) -> Tuple[torch.Tensor, torch.Tensor]:
    """Marching cubes of a (res,res,res) density grid over [min_bound, max_bound] (laid out as density_grid writes it) ->
    (vertices (V,3) fp32 world, faces (F,3) int32 counter-clockwise seen from outside, the object being density > iso).
    The tables wind counter-clockwise about the direction of decreasing density in index coordinates; the index -> world
    permutation swaps x and y, which reverses handedness, so two columns of the faces are swapped."""
    res = density.shape[0]
    if tuple(density.shape) != (res, res, res):
        raise ValueError(f"expected a (res,res,res) grid, got {tuple(density.shape)}")
    vidx, faces = marching_cubes(density, iso)
    return _index_to_world_surface(vidx, faces, min_bound, max_bound, res)


def _index_to_world_surface(vidx, faces, min_bound, max_bound, res):
    verts = index_to_world(vidx, world_axes(min_bound, max_bound, res, vidx.device))
    return verts, faces[:, [0, 2, 1]].contiguous()


_PLY_VERTEX = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4"),
                        ("red", "u1"), ("green", "u1"), ("blue", "u1")])
_PLY_FACE = np.dtype([("n", "u1"), ("v", "<i4", (3,))])
_PLY_PROPS = ["property float x", "property float y", "property float z", "property float nx", "property float ny",
              "property float nz", "property uchar red", "property uchar green", "property uchar blue"]
_PLY_FACE_PROP = "property list uchar int vertex_indices"


def write_ply(path: str, mesh: Mesh) -> None:
    """Binary little-endian PLY: vertex x y z nx ny nz (float) red green blue (uchar = round(clamp(c, 0, 1) * 255)),
    face `list uchar int vertex_indices`.  Whole arrays at once (numpy structured arrays), no per-element loop."""
    v = mesh.vertices.detach().float().cpu().numpy()
    nv = mesh.normals.detach().float().cpu().numpy()
    c = torch.round(torch.nan_to_num(mesh.colors.detach().float(), nan=0.0).clamp(0, 1) * 255).to(torch.uint8).cpu().numpy()
    f = mesh.faces.detach().to(torch.int32).cpu().numpy()
    va = np.empty(v.shape[0], dtype=_PLY_VERTEX)
    for i, k in enumerate(("x", "y", "z")):
        va[k] = v[:, i]
        va["n" + k] = nv[:, i]
    for i, k in enumerate(("red", "green", "blue")):
        va[k] = c[:, i]
    fa = np.empty(f.shape[0], dtype=_PLY_FACE)
    fa["n"] = 3
    fa["v"] = f
    header = "\n".join(["ply", "format binary_little_endian 1.0", f"element vertex {va.shape[0]}", *_PLY_PROPS,
                        f"element face {fa.shape[0]}", _PLY_FACE_PROP, "end_header"]) + "\n"
    with open(path, "wb") as fh:
        fh.write(header.encode("ascii"))
        fh.write(va.tobytes())
        fh.write(fa.tobytes())


def read_ply(path: str) -> Mesh:
    """The files `write_ply` writes (exactly that layout; anything else raises) -> Mesh of CPU tensors, colors uint8."""
    with open(path, "rb") as fh:
        data = fh.read()
    end = data.find(b"end_header\n")
    if not data.startswith(b"ply\n") or end < 0:
        raise ValueError(f"{path}: not a PLY file")
    head = data[:end].decode("ascii").splitlines()
    body = end + len(b"end_header\n")
    try:
        nv = int(head[2].split()[2])
        nf = int(head[3 + len(_PLY_PROPS)].split()[2])
    except (IndexError, ValueError):
        raise ValueError(f"{path}: unexpected PLY header") from None
    want = ["ply", "format binary_little_endian 1.0", f"element vertex {nv}", *_PLY_PROPS, f"element face {nf}",
            _PLY_FACE_PROP]
    if head != want:
        raise ValueError(f"{path}: unexpected PLY header {head}")
    va = np.frombuffer(data, dtype=_PLY_VERTEX, count=nv, offset=body)
    fa = np.frombuffer(data, dtype=_PLY_FACE, count=nf, offset=body + nv * _PLY_VERTEX.itemsize)
    if body + nv * _PLY_VERTEX.itemsize + nf * _PLY_FACE.itemsize != len(data) or (fa["n"] != 3).any():
        raise ValueError(f"{path}: body does not match the header")
    col = lambda *ks: torch.from_numpy(np.stack([va[k] for k in ks], axis=1).copy())     # noqa: E731
    return Mesh(col("x", "y", "z"), torch.from_numpy(fa["v"].copy()), col("nx", "ny", "nz"), col("red", "green", "blue"))
