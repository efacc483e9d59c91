"""Run the REFERENCE's own classes (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

Imports ``iPERCore`` from the staged tree ``oracle/_ref`` (oracle/build_ref.py) and builds the real
``iPERCore.models.imitator.Imitator`` on synthetic assets, because the real ones are not available offline (SURVEY.md §8c):

* ``neural_renderer`` (third-party CUDA extension, absent): a stub module with upstream's ``look_at`` /
  ``vertices_to_faces`` (plain torch) and ``rasterize_face_index_map_and_weight_map`` backed by oracle/raster_ref.c on the
  host (device tensors make a CPU round trip).  It is only installed when no ``neural_renderer`` is registered yet, so
  ``ipercore_b200.patch.install()`` (which registers the CUDA drop-in) takes precedence when called first.
* ``easydict`` (not installed): 5-line attribute dict.  ``np.int`` / ``np.float`` shims for numpy >= 1.24 (mesh.py).
* SMPLH pkl ``smpl_model_with_hand_v2.pkl``: the SMPLH-shaped random model of oracle/lbs_ref.synthetic_smplh written in the
  pkl layout ``bodynets/batch_smplh.py:76-135`` / ``smplx/body_models.py:205-296`` read.
* ``smpl_faces.npy``: the ``f`` vertex ids of assets/configs/pose3d/mapper_uv.txt (SURVEY.md §8c).
* generator checkpoint: oracle/weights.synth_state_dict saved with torch.save (221-key reference layout).

Used by tests/test_reference_integration_*.py, bench.py --impl reference and bench.py's gpu_library_baseline leg.
"""
import importlib.util
import os
import pickle
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
STAGED = os.path.join(HERE, "_ref")


def ref_root():
    if os.path.isdir(os.path.join(STAGED, "iPERCore")):
        return STAGED
    raise FileNotFoundError("the reference tree is not staged under oracle/_ref: run oracle/build_ref.py")


def available():
    try:
        ref_root()
        return True
    except FileNotFoundError:
        return False


class AttrDict(dict):
    """stand-in for easydict.EasyDict (attribute access, nested dicts wrapped on read)."""

    def __getattr__(self, k):
        try:
            v = self[k]
        except KeyError:
            raise AttributeError(k)
        if isinstance(v, dict) and not isinstance(v, AttrDict):
            v = AttrDict(v)
            self[k] = v
        return v

    def __setattr__(self, k, v):
        self[k] = v


def _stub_neural_renderer():
    import torch
    from . import raster
    nr = types.ModuleType("neural_renderer")
    nr.__doc__ = "oracle stub of iPERDance/neural_renderer (CPU, oracle/raster_ref.c)"

    def look_at(vertices, eye, at=(0, 0, 0), up=(0, 1, 0)):
        dev = vertices.device
        eye_t = torch.tensor(eye, dtype=torch.float32, device=dev)
        at_t = torch.tensor(at, dtype=torch.float32, device=dev)
        up_t = torch.tensor(up, dtype=torch.float32, device=dev)
        bs = vertices.shape[0]
        eye_t = eye_t[None].repeat(bs, 1); at_t = at_t[None].repeat(bs, 1); up_t = up_t[None].repeat(bs, 1)
        z = torch.nn.functional.normalize(at_t - eye_t, eps=1e-5)
        x = torch.nn.functional.normalize(torch.cross(up_t, z, dim=1), eps=1e-5)
        y = torch.nn.functional.normalize(torch.cross(z, x, dim=1), eps=1e-5)
        r = torch.cat((x[:, None], y[:, None], z[:, None]), dim=1)
        return torch.matmul(vertices - eye_t[:, None, :], r.transpose(1, 2))

    def vertices_to_faces(vertices, faces):
        bs, nv = vertices.shape[:2]
        faces = faces + (torch.arange(bs, dtype=torch.int32, device=vertices.device) * nv)[:, None, None]
        return vertices.reshape(bs * nv, 3)[faces.long()]

    def rasterize_face_index_map_and_weight_map(faces, image_size=256, anti_aliasing=False, near=0.1, far=100):
        fim, wim = raster.rasterize_fim_wim(faces.detach().float().cpu().numpy(), image_size, near, far)
        return torch.from_numpy(fim).to(faces.device), torch.from_numpy(wim).to(faces.device)

    nr.look_at, nr.vertices_to_faces = look_at, vertices_to_faces
    nr.rasterize_face_index_map_and_weight_map = rasterize_face_index_map_and_weight_map
    nr.IS_ORACLE_STUB = True
    return nr


def install_import_shims(stub_renderer=True):
    """Make ``import iPERCore`` work here: path, easydict, numpy aliases and (unless one is registered) the nr stub."""
    root = ref_root()
    if root not in sys.path:
        sys.path.insert(0, root)
    if not hasattr(np, "int"):
        np.int = int
    if not hasattr(np, "float"):
        np.float = float
    if "easydict" not in sys.modules:
        ed = types.ModuleType("easydict")
        ed.EasyDict = AttrDict
        sys.modules["easydict"] = ed
    if stub_renderer and "neural_renderer" not in sys.modules:
        sys.modules["neural_renderer"] = _stub_neural_renderer()
    return root


def load_by_path(name, relpath):
    """Import one reference file WITHOUT running its package __init__ chain (e.g. the generator alone)."""
    spec = importlib.util.spec_from_file_location(name, os.path.join(ref_root(), relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def reference_generator_module():
    """The reference's attlwb_spade_resunet.py as a module (bg_inpaintor.py resolved as its sibling)."""
    if "refgen.attlwb_spade_resunet" in sys.modules:
        return sys.modules["refgen.attlwb_spade_resunet"]
    install_import_shims(stub_renderer=False)
    pkg = types.ModuleType("refgen")
    pkg.__path__ = [os.path.join(ref_root(), "iPERCore/models/networks/generators")]
    sys.modules["refgen"] = pkg
    load_by_path("refgen.bg_inpaintor", "iPERCore/models/networks/generators/bg_inpaintor.py")
    return load_by_path("refgen.attlwb_spade_resunet", "iPERCore/models/networks/generators/attlwb_spade_resunet.py")


def generator_cfg():
    import toml
    cfg = toml.load(os.path.join(ref_root(), "assets/configs/neural_renders/AttLWB-SPADE.toml"))
    return AttrDict(cfg["Generator"])


def reference_generator(seed=0, device="cpu"):
    """The reference AttentionLWBGenerator with the synthetic 221-key checkpoint loaded strictly."""
    from . import weights
    gen = reference_generator_module()
    net = gen.AttentionLWBGenerator(generator_cfg(), temporal=False).eval()
    net.load_state_dict(weights.synth_state_dict(seed), strict=True)
    return net.to(device)


# ----------------------------------------------------------------------------------------------------------------------
# synthetic assets in the reference's file formats
# ----------------------------------------------------------------------------------------------------------------------
def smplh_pkl_dict(model):
    """oracle/lbs_ref.synthetic_smplh model -> the dict layout of smpl_model_with_hand_v2.pkl."""
    nv, nj = model["v_template"].shape[0], model["J_regressor"].shape[0]
    parents = np.asarray(model["parents"]).astype(np.int64)
    kintree = np.stack([np.where(parents < 0, 2 ** 32 - 1, parents), np.arange(nj)]).astype(np.int64)
    kintree[0, 0] = -1
    npb = (nj - 1) * 9
    # body_models.py:284-288: posedirs (nv,3,npb) -> reshape(-1, npb).T = (npb, nv*3)
    posedirs = np.ascontiguousarray(model["posedirs"].T).reshape(nv, 3, npb)
    rng = np.random.Generator(np.random.PCG64(17))
    comps = np.linalg.qr(rng.standard_normal((45, 45)))[0].astype(np.float32)
    return dict(f=model["faces"].astype(np.uint32), v_template=model["v_template"].astype(np.float64),
                shapedirs=model["shapedirs"].astype(np.float64), J_regressor=model["J_regressor"].astype(np.float64),
                posedirs=posedirs.astype(np.float64), kintree_table=kintree, weights=model["lbs_weights"].astype(np.float64),
                hands_componentsl=comps, hands_componentsr=comps[::-1].copy(),
                hands_meanl=model["hands_mean"][:45].astype(np.float64), hands_meanr=model["hands_mean"][45:].astype(np.float64))


def make_assets(workdir, seed=0):
    """Write smpl_model_with_hand_v2.pkl, smpl_faces.npy and the generator checkpoint under workdir; returns the paths."""
    import torch
    from . import lbs_ref, synth, weights
    os.makedirs(workdir, exist_ok=True)
    tpl = synth.load_template()
    model = lbs_ref.synthetic_smplh(template=synth.base_verts(tpl).astype(np.float32) * 0.9)
    model["faces"] = tpl["faces"]
    paths = dict(smpl=os.path.join(workdir, "smpl_model_with_hand_v2.pkl"), faces=os.path.join(workdir, "smpl_faces.npy"),
                 ckpt=os.path.join(workdir, "AttLWB-SPADE_id_G_synthetic.pth"))
    with open(paths["smpl"], "wb") as f:
        pickle.dump(smplh_pkl_dict(model), f, protocol=2)
    np.save(paths["faces"], tpl["faces"].astype(np.int32))
    torch.save(weights.synth_state_dict(seed), paths["ckpt"])
    return paths, model


def make_opt(workdir, image_size=512, num_source=2, seed=0):
    """The option object Imitator / FlowComposition read (deploy.toml + AttLWB-SPADE.toml, asset paths -> workdir)."""
    import toml
    root = ref_root()
    cfg = toml.load(os.path.join(root, "assets/configs/deploy.toml"))
    paths, model = make_assets(workdir, seed)
    opt = AttrDict(cfg)
    opt.image_size, opt.num_source = image_size, num_source
    for k in ("fim_enc_path", "uv_map_path", "part_path", "front_path", "head_path", "facial_path"):
        opt[k] = os.path.join(root, cfg[k].lstrip("./"))
    opt.face_path, opt.smpl_model_hand, opt.smpl_model = paths["faces"], paths["smpl"], paths["smpl"]
    opt.load_path_G = paths["ckpt"]
    opt.neural_render_cfg = AttrDict(toml.load(os.path.join(root, cfg["neural_render_cfg_path"].lstrip("./"))))
    out_dir = os.path.join(workdir, "out")
    os.makedirs(out_dir, exist_ok=True)
    opt.meta_data = AttrDict(personalized_ckpt_path=os.path.join(workdir, "no_personalized.pth"), checkpoints_dir=out_dir)
    opt.output_dir = out_dir
    return opt, model


def build_imitator(opt, device):
    """The real iPERCore.models.imitator.Imitator (whatever neural_renderer / generator factory is registered)."""
    import torch
    root = install_import_shims()
    from iPERCore.models.imitator import Imitator
    cwd = os.getcwd()
    os.chdir(root)          # FlowComposition._create_render leaves head/front/facial json at their cwd-relative defaults
    try:
        return Imitator(opt, device=torch.device(device))
    finally:
        os.chdir(cwd)


def synthetic_clip(model, n_frames, ns=2, seed=5):
    """(src_smpl (ns,85), tgt_smpls (T,85)) for the synthetic SMPLH model: moderate random poses, one shape."""
    rng = np.random.Generator(np.random.PCG64(seed))
    shape = (rng.standard_normal((1, 10)) * 0.5).astype(np.float32)
    src = np.concatenate([np.tile([[0.9, 0.0, -0.25]], (ns, 1)), rng.standard_normal((ns, 72)) * 0.15,
                          np.repeat(shape, ns, 0)], 1).astype(np.float32)
    base = rng.standard_normal((1, 72)) * 0.2
    tgt = np.concatenate([np.tile([[1.0, 0.05, -0.2]], (n_frames, 1)) + rng.standard_normal((n_frames, 3)) * 0.02,
                          base + rng.standard_normal((n_frames, 72)) * 0.1, rng.standard_normal((n_frames, 10))],
                         1).astype(np.float32)
    return src, tgt


def write_source_images(workdir, ns, image_size, seed=1):
    """ns PNG source images (uint8 RGB of oracle.synth.smooth_image) -> list of paths, as source_setup loads them."""
    import cv2
    from . import synth
    imgs = synth.smooth_image((ns, 3, image_size, image_size), seed=seed)
    paths = []
    for i in range(ns):
        p = os.path.join(workdir, "src_%02d.png" % i)
        cv2.imwrite(p, ((imgs[i].transpose(1, 2, 0)[:, :, ::-1] + 1) / 2 * 255).clip(0, 255).astype(np.uint8))
        paths.append(p)
    return paths
