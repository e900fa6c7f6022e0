"""Model compiler: MJCF (the subset the two reference XMLs use) -> TsgModel.

Replaces, for the hot path, what ``MjModel.from_xml_path`` does inside gym's
``MujocoEnv.__init__`` (reference call sites: tr_env.py:274-276,
tensegrity_env.py:239-241).  Constants follow
/root/reference/3prism_jonathan_steady_side.xml and
/root/reference/3prism_jonathan_steady_side_uneven_ground.xml; derived values
(inertia from geoms, invweight0, meaninertia, fromto frames, spring lengths at
qpos0, normalised height field) restate the MuJoCo 2.3.7 compiler rules.

The ctypes structures mirror include/tsg_model.h field by field.
"""
from __future__ import annotations

import ctypes as C
import json
import math
import os
import xml.etree.ElementTree as ET

import numpy as np

NBAR, NGEOM_BAR, NTEN, NACT, NQ, NV, NBODY = 3, 5, 9, 6, 21, 18, 4
GEOM_SPHERE, GEOM_CYLINDER = 2, 5
FLOOR_PLANE, FLOOR_HFIELD = 0, 1
DYN_NONE, DYN_FILTER = 0, 2
FLAG_ACTVEL_WHEN_CLAMPED, FLAG_CROSSBAR_DERIV, FLAG_FIXNORMAL = 1, 2, 4
ENV_TR, ENV_LEGACY = 0, 1
TASKS = {"straight": 0, "turn": 1, "aiming": 2, "tracking": 3, "vel_track": 4}
HEADING_SLOTS, NPOSE, NDRAW = 32, 6, 10

ASSET_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "assets")

d = C.c_double
i32 = C.c_int32


class TsgModel(C.Structure):
    _fields_ = [
        ("struct_bytes", i32), ("flags", C.c_uint32),
        ("timestep", d), ("gravity", d * 3), ("tolerance", d), ("ls_tolerance", d),
        ("impratio", d), ("mpr_tolerance", d),
        ("iterations", i32), ("ls_iterations", i32), ("mpr_iterations", i32), ("pad0_", i32),
        ("body_mass", d * NBAR), ("body_inertia", (d * 3) * NBAR), ("body_invweight0", (d * 2) * NBAR),
        ("meaninertia", d), ("qpos0", d * NQ),
        ("geom_type", (i32 * NGEOM_BAR) * NBAR), ("pad1_", i32),
        ("geom_size", ((d * 3) * NGEOM_BAR) * NBAR), ("geom_pos", ((d * 3) * NGEOM_BAR) * NBAR),
        ("geom_quat", ((d * 4) * NGEOM_BAR) * NBAR), ("geom_rbound", (d * NGEOM_BAR) * NBAR),
        ("ten_body", (i32 * 2) * NTEN), ("ten_site", ((d * 3) * 2) * NTEN),
        ("ten_stiffness", d * NTEN), ("ten_damping", d * NTEN), ("ten_lengthspring", (d * 2) * NTEN),
        ("act_tendon", i32 * NACT), ("act_dyntype", i32), ("ctrllimited", i32), ("forcelimited", i32), ("pad2_", i32),
        ("act_dynprm0", d), ("act_gain", d), ("act_bias", d * 3), ("ctrlrange", d * 2), ("forcerange", d * 2),
        ("solref", d * 2), ("solimp", d * 5), ("friction", d * 5), ("condim", i32),
        ("floor_type", i32), ("floor_pos", d * 3), ("floor_mat", d * 9),
        ("hf_nrow", i32), ("hf_ncol", i32), ("hf_size", d * 4), ("hf_data", C.POINTER(C.c_float)),
    ]


class TsgEnvConfig(C.Structure):
    _fields_ = [
        ("struct_bytes", i32), ("env_kind", i32), ("task", i32), ("frame_skip", i32), ("obs_dim", i32),
        ("use_cap_velocity", i32), ("terminate_when_unhealthy", i32), ("is_test", i32),
        ("reward_delay_steps", i32), ("max_episode_steps", i32), ("warmup_steps", i32), ("npose", i32),
        ("desired_direction", d), ("ctrl_cost_weight", d), ("healthy_reward", d), ("yaw_reward_weight", d),
        ("min_reset_heading", d), ("max_reset_heading", d),
        ("tendon_reset_mean", d), ("tendon_reset_stdev", d), ("tendon_min_length", d), ("tendon_max_length", d),
        ("waypt_range", d * 2), ("waypt_angle_range", d * 2),
        ("ditch_reward_max", d), ("ditch_reward_stdev", d), ("waypt_reward_amplitude", d), ("waypt_reward_stdev", d),
        ("kill_force", d), ("reset_pose", (d * NQ) * NPOSE),
        ("use_obs_noise", i32), ("pad_noise_", i32), ("obs_noise_tendon_stdev", d), ("obs_noise_cap_pos_stdev", d),
        ("reset_noise_scale", d), ("use_contact_forces", i32), ("pad_contact_", i32), ("contact_cost_weight", d),
        ("contact_force_range", d * 2),
    ]


# --------------------------------------------------------------------------- helpers
def _floats(s):
    return [float(x) for x in s.split()]


def quat_mul(a, b):
    return np.array([
        a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3],
        a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
        a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1],
        a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])


def quat2mat(q):
    q = np.asarray(q, float)
    w, x, y, z = q
    return np.array([
        [w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)],
        [2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)],
        [2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z]])


def _z2quat(vec):
    """mjuu_z2quat: rotation taking +z to `vec` (used for fromto geoms)."""
    v = np.asarray(vec, float)
    v = v / np.linalg.norm(v)
    axis = np.cross([0.0, 0.0, 1.0], v)
    s = np.linalg.norm(axis)
    axis = np.array([1.0, 0.0, 0.0]) if s < 1e-10 else axis / s
    ang = math.atan2(s, v[2])
    return np.array([math.cos(ang / 2), *(axis * math.sin(ang / 2))])


def load_heightfield_png(path):
    """PNG -> (nrow, ncol, float32 data in [0,1]); MuJoCo: grey = red channel, rows reversed
    (image top = +y), then (v - min) / (max - min) in float32."""
    from PIL import Image

    im = np.array(Image.open(path))
    grey = im[..., 0] if im.ndim == 3 else im
    data = grey[::-1].astype(np.float32)
    emin, emax = np.float32(data.min()), np.float32(data.max())
    data = data - emin
    if emax - emin > 1e-15:
        data = data / np.float32(emax - emin)
    return data.shape[0], data.shape[1], np.ascontiguousarray(data, np.float32)


# --------------------------------------------------------------------------- MJCF -> dict
def parse_mjcf(xml_path):
    """Parse the reference MJCF subset into a plain dict of model constants."""
    root = ET.parse(xml_path).getroot()
    base = os.path.dirname(os.path.abspath(xml_path))
    comp = root.find("compiler")
    assert comp is None or comp.get("coordinate", "local") == "local"
    opt = root.find("option")
    o = dict(opt.attrib) if opt is not None else {}
    assert o.get("cone", "pyramidal") == "elliptic" and o.get("solver", "Newton") == "Newton"
    assert o.get("integrator", "Euler") == "implicitfast"
    md = {
        "timestep": float(o.get("timestep", 0.002)),
        "gravity": _floats(o.get("gravity", "0 0 -9.81")),
        "iterations": int(o.get("iterations", 100)),
        "tolerance": float(o.get("tolerance", 1e-8)),
        "ls_iterations": int(o.get("ls_iterations", 50)),
        "ls_tolerance": float(o.get("ls_tolerance", 0.01)),
        "impratio": float(o.get("impratio", 1.0)),
        "mpr_iterations": int(o.get("mpr_iterations", 50)),
        "mpr_tolerance": float(o.get("mpr_tolerance", 1e-6)),
        "flags": FLAG_ACTVEL_WHEN_CLAMPED | FLAG_FIXNORMAL,
    }
    dflt = root.find("default")
    dgeom = dict(dflt.find("geom").attrib) if dflt is not None and dflt.find("geom") is not None else {}
    dten = dict(dflt.find("tendon").attrib) if dflt is not None and dflt.find("tendon") is not None else {}
    dgen = dict(dflt.find("general").attrib) if dflt is not None and dflt.find("general") is not None else {}

    def gattr(g, k, default=None):
        return g.get(k, dgeom.get(k, default))

    world = root.find("worldbody")
    # ---- floor
    floor = [g for g in world.findall("geom") if g.get("name") == "floor"][0]
    ftype = floor.get("type", "sphere")
    md["floor_pos"] = _floats(floor.get("pos", "0 0 0"))
    md["floor_mat"] = quat2mat(_floats(floor.get("quat", "1 0 0 0"))).reshape(-1).tolist()
    if ftype == "plane":
        md["floor_type"] = FLOOR_PLANE
        md["hfield"] = None
    else:
        assert ftype == "hfield"
        md["floor_type"] = FLOOR_HFIELD
        hf = [h for h in root.find("asset").findall("hfield") if h.get("name") == floor.get("hfield")][0]
        nrow, ncol, data = load_heightfield_png(os.path.join(base, hf.get("file")))
        md["hfield"] = {"nrow": nrow, "ncol": ncol, "size": _floats(hf.get("size")), "data": data}
    fcondim = int(floor.get("condim", dgeom.get("condim", 3)))
    # ---- bars
    bodies = world.findall("body")
    assert len(bodies) == NBAR
    site_of = {}
    qpos0, gtype, gsize, gpos, gquat, grb, masses, inertias = [], [], [], [], [], [], [], []
    condim, friction, solref, solimp = fcondim, None, None, None
    for b, body in enumerate(bodies):
        assert body.find("freejoint") is not None
        bq = np.array(_floats(body.get("quat", "1 0 0 0")))
        bq = bq / np.linalg.norm(bq)  # compiler normalises body quats
        qpos0 += _floats(body.get("pos")) + bq.tolist()
        geoms = body.findall("geom")
        assert len(geoms) == NGEOM_BAR
        bt, bs, bp, bqg, brb = [], [], [], [], []
        mtot, Itot = 0.0, np.zeros((3, 3))
        for g in geoms:
            t = g.get("type", "sphere")
            size = _floats(gattr(g, "size"))
            mass = float(g.get("mass"))
            if g.get("fromto") is not None:
                ft = np.array(_floats(g.get("fromto")))
                pos = 0.5 * (ft[:3] + ft[3:])
                vec = ft[:3] - ft[3:]
                quat = _z2quat(vec)
                size = [size[0], 0.5 * np.linalg.norm(vec)]
            else:
                pos = np.array(_floats(g.get("pos", "0 0 0")))
                quat = np.array(_floats(g.get("quat", "1 0 0 0")))
                quat = quat / np.linalg.norm(quat)
            if t == "sphere":
                ty, sz = GEOM_SPHERE, [size[0], 0.0, 0.0]
                Il = np.eye(3) * (0.4 * mass * size[0] ** 2)
                rb = size[0]
            else:
                assert t == "cylinder"
                ty, sz = GEOM_CYLINDER, [size[0], size[1], 0.0]
                r, hl = size[0], size[1]
                ixx = mass * (r * r / 4 + hl * hl / 3)
                Il = np.diag([ixx, ixx, mass * r * r / 2])
                rb = math.sqrt(r * r + hl * hl)
            Rg = quat2mat(quat)
            Ig = Rg @ Il @ Rg.T
            Itot += Ig + mass * (pos @ pos * np.eye(3) - np.outer(pos, pos))
            mtot += mass
            bt.append(ty); bs.append(sz); bp.append(pos.tolist()); bqg.append(quat.tolist()); brb.append(rb)
            condim = max(condim, int(gattr(g, "condim", 3)))
            fr = _floats(gattr(g, "friction", "1 0.005 0.0001"))
            sr = _floats(gattr(g, "solref", "0.02 1"))
            si = _floats(gattr(g, "solimp", "0.9 0.95 0.001 0.5 2"))
            assert friction in (None, fr) and solref in (None, sr) and solimp in (None, si)
            friction, solref, solimp = fr, sr, si
        com = sum(m_ * np.array(p_) for m_, p_ in zip([float(g.get("mass")) for g in geoms], bp)) / mtot
        assert np.abs(com).max() < 1e-12, "bar COM must sit at the body origin"
        assert np.abs(Itot - np.diag(np.diag(Itot))).max() < 1e-12, "principal axes must be the body axes"
        masses.append(mtot); inertias.append(np.diag(Itot).tolist())
        gtype.append(bt); gsize.append(bs); gpos.append(bp); gquat.append(bqg); grb.append(brb)
        for s in body.findall("site"):
            site_of[s.get("name")] = (b, _floats(s.get("pos", "0 0 0")))
    # floor params must agree with the bars' (MuJoCo would mix; equal here)
    assert _floats(floor.get("friction", dgeom.get("friction", "1 0.005 0.0001"))) == friction
    assert solref[0] < 0 and solref[1] < 0, "only direct (negative) solref is restated"
    md.update(qpos0=qpos0, geom_type=gtype, geom_size=gsize, geom_pos=gpos, geom_quat=gquat, geom_rbound=grb,
              body_mass=masses, body_inertia=inertias, condim=condim, solref=solref, solimp=solimp,
              friction=[friction[0], friction[0], friction[1], friction[2], friction[2]])
    md["body_invweight0"] = [[1.0 / m_, float(np.mean(1.0 / np.array(I_)))] for m_, I_ in zip(masses, inertias)]
    md["meaninertia"] = float(np.mean([v for m_, I_ in zip(masses, inertias) for v in [m_] * 3 + list(I_)]))
    # ---- tendons
    tendons = root.find("tendon").findall("spatial")
    assert len(tendons) == NTEN
    tname, tb, ts, tk, tdmp, tls = [], [], [], [], [], []
    xpos = [np.array(qpos0[7 * b:7 * b + 3]) for b in range(NBAR)]
    xmat = [quat2mat(qpos0[7 * b + 3:7 * b + 7]) for b in range(NBAR)]
    for t in tendons:
        sites = [s.get("site") for s in t.findall("site")]
        assert len(sites) == 2
        (b0, p0), (b1, p1) = site_of[sites[0]], site_of[sites[1]]
        tname.append(t.get("name")); tb.append([b0, b1]); ts.append([p0, p1])
        tk.append(float(t.get("stiffness", dten.get("stiffness", 0))))
        tdmp.append(float(t.get("damping", dten.get("damping", 0))))
        sl = _floats(t.get("springlength", dten.get("springlength", "-1")))
        if len(sl) == 1:
            sl = [sl[0], sl[0]]
        if sl[0] < 0:  # compiler: use the length at qpos0
            L0 = float(np.linalg.norm((xpos[b1] + xmat[b1] @ np.array(p1)) - (xpos[b0] + xmat[b0] @ np.array(p0))))
            sl = [L0, L0]
        tls.append(sl)
    md.update(ten_body=tb, ten_site=ts, ten_stiffness=tk, ten_damping=tdmp, ten_lengthspring=tls)
    # ---- actuators (<general tendon=...>, attributes from the default class)
    acts = root.find("actuator").findall("general")
    assert len(acts) == NACT
    md["act_tendon"] = [tname.index(a.get("tendon")) for a in acts]

    def aattr(k, default):
        vals = {a.get(k, dgen.get(k, default)) for a in acts}
        assert len(vals) == 1
        return vals.pop()

    dyn = aattr("dyntype", "none")
    md["act_dyntype"] = {"none": DYN_NONE, "filter": DYN_FILTER}[dyn]
    md["act_dynprm0"] = _floats(aattr("dynprm", "1 0 0"))[0]
    assert aattr("gaintype", "fixed") == "fixed"
    md["act_gain"] = _floats(aattr("gainprm", "1 0 0"))[0]
    bias = aattr("biastype", "none")
    md["act_bias"] = (_floats(aattr("biasprm", "0 0 0")) + [0, 0, 0])[:3] if bias == "affine" else [0.0, 0.0, 0.0]
    md["ctrllimited"] = int(aattr("ctrllimited", "false") == "true")
    md["ctrlrange"] = _floats(aattr("ctrlrange", "0 0"))
    md["forcelimited"] = int(aattr("forcelimited", "false") == "true")
    md["forcerange"] = _floats(aattr("forcerange", "0 0"))
    return md


# --------------------------------------------------------------------------- dict <-> json, dict -> struct
def save_model_json(md, path):
    out = {k: v for k, v in md.items() if k != "hfield"}
    if md.get("hfield") is not None:
        hf = md["hfield"]
        npy = os.path.splitext(path)[0] + "_hfield.npy"
        np.save(npy, hf["data"])
        out["hfield"] = {"nrow": hf["nrow"], "ncol": hf["ncol"], "size": hf["size"], "data_file": os.path.basename(npy)}
    else:
        out["hfield"] = None
    with open(path, "w") as f:
        json.dump(out, f, indent=1)


def load_model_json(path):
    with open(path) as f:
        md = json.load(f)
    if md.get("hfield") is not None:
        hf = md["hfield"]
        hf["data"] = np.load(os.path.join(os.path.dirname(os.path.abspath(path)), hf["data_file"])).astype(np.float32)
    return md


_ASSET_BY_XML = {
    "3prism_jonathan_steady_side.xml": "model_flat.json",
    "3prism_jonathan_steady_side_uneven_ground.xml": "model_uneven.json",
}


def load_model(xml_file=None):
    """XML path (parsed if it exists), or the name of a reference XML / 'flat' / 'uneven'
    (served from assets/, which tools/extract_assets.py generated from those XMLs)."""
    if xml_file is None:
        xml_file = "flat"
    if isinstance(xml_file, dict):
        return xml_file
    if os.path.isfile(xml_file) and xml_file.endswith(".xml"):
        return parse_mjcf(xml_file)
    if os.path.isfile(xml_file) and xml_file.endswith(".json"):
        return load_model_json(xml_file)
    key = os.path.basename(xml_file)
    if key == "legacy_flat":
        # DERIVED variant (not a reference file): bars, sites, tendons and filter actuators of the uneven-ground
        # XML on a flat plane at z = 0.  The SB3 checkpoints' `_last_obs` fit this bar geometry exactly and the
        # pretrained policies reproduce the reference's training statistics on it (tests/test_gpu_parity.py).
        md = dict(load_model("uneven"))
        md.update(floor_type=FLOOR_PLANE, floor_pos=[0.0, 0.0, 0.0], hfield=None, source="derived: uneven XML bars on a plane")
        return md
    name = {"flat": "model_flat.json", "uneven": "model_uneven.json"}.get(key, _ASSET_BY_XML.get(key))
    if name is None:
        raise FileNotFoundError(f"model file not found: {xml_file}")
    return load_model_json(os.path.join(ASSET_DIR, name))


def _fill(dst, src):
    a = np.asarray(src)
    flat = np.ctypeslib.as_array(dst).reshape(-1)
    flat[:] = a.reshape(-1)


def model_struct(md):
    """dict -> (TsgModel, keepalive) ; keepalive holds the height-field buffer."""
    m = TsgModel()
    m.struct_bytes = C.sizeof(TsgModel)
    m.flags = int(md["flags"])
    for k in ("timestep", "tolerance", "ls_tolerance", "impratio", "mpr_tolerance", "meaninertia",
              "act_dynprm0", "act_gain"):
        setattr(m, k, float(md[k]))
    for k in ("iterations", "ls_iterations", "mpr_iterations", "act_dyntype", "ctrllimited", "forcelimited",
              "condim", "floor_type"):
        setattr(m, k, int(md[k]))
    for k in ("gravity", "body_mass", "body_inertia", "body_invweight0", "qpos0", "geom_type", "geom_size",
              "geom_pos", "geom_quat", "geom_rbound", "ten_body", "ten_site", "ten_stiffness", "ten_damping",
              "ten_lengthspring", "act_tendon", "act_bias", "ctrlrange", "forcerange", "solref", "solimp",
              "friction", "floor_pos", "floor_mat"):
        _fill(getattr(m, k), md[k])
    keep = None
    if md.get("hfield") is not None:
        hf = md["hfield"]
        keep = np.ascontiguousarray(hf["data"], np.float32)
        m.hf_nrow, m.hf_ncol = int(hf["nrow"]), int(hf["ncol"])
        _fill(m.hf_size, hf["size"])
        m.hf_data = keep.ctypes.data_as(C.POINTER(C.c_float))
    return m, keep


# --------------------------------------------------------------------------- per-env parameters
# the row layout of include/tsg.h (TSG_PARAM_*): field -> (offset, width)
PARAM_FIELDS = (("ten_stiffness", 0, NTEN), ("ten_damping", 9, NTEN), ("ten_lengthspring", 18, 2 * NTEN),
                ("act_gain", 36, 1), ("act_bias", 37, 3), ("act_dynprm0", 40, 1))
NPARAM = 41


def nominal_params(md):
    """the nominal per-env parameter row [41] of a model dict: its tendon and actuator constants"""
    row = np.zeros(NPARAM)
    for name, off, w in PARAM_FIELDS:
        row[off:off + w] = np.asarray(md[name], np.float64).reshape(-1)
    return row


def param_overrides(row):
    """per-env parameter row [41] -> the model-dict fields it replaces (keyword overrides of a model dict)"""
    row = np.asarray(row, np.float64)
    if row.shape != (NPARAM,):
        raise ValueError(f"a parameter row has {NPARAM} values, got shape {row.shape}")
    out = {}
    for name, off, w in PARAM_FIELDS:
        v = row[off:off + w]
        if name == "ten_lengthspring":
            out[name] = v.reshape(NTEN, 2).tolist()
        elif w == 1:
            out[name] = float(v[0])
        else:
            out[name] = v.tolist()
    return out


def param_scale_ranges(param_ranges):
    """{field: (lo, hi)} of scale factors (each bound a scalar or an array of the field's width; fields not given
    keep scale 1) -> (lo[41], hi[41]).  Raises ValueError on an unknown field, a bad shape, a non-finite bound,
    lo > hi, a negative scale, a dynprm0 scale of 0, or unequal ranges of a tendon's lower and upper lengthspring."""
    lo, hi = np.ones(NPARAM), np.ones(NPARAM)
    fields = {name: (off, w) for name, off, w in PARAM_FIELDS}
    for name, bounds in dict(param_ranges).items():
        if name not in fields:
            raise ValueError(f"unknown per-env parameter {name!r}; known: {', '.join(fields)}")
        off, w = fields[name]
        try:
            b_lo, b_hi = bounds
        except (TypeError, ValueError):
            raise ValueError(f"{name}: expected a (lo, hi) pair") from None
        for dst, b in ((lo, b_lo), (hi, b_hi)):
            a = np.asarray(b, np.float64)
            if a.ndim == 0:
                a = np.full(w, float(a))
            if a.shape != (w,):
                raise ValueError(f"{name}: a bound is a scalar or has {w} values, got shape {a.shape}")
            dst[off:off + w] = a
    if not (np.isfinite(lo).all() and np.isfinite(hi).all()):
        raise ValueError("param ranges must be finite")
    if (lo < 0).any() or (lo > hi).any():
        raise ValueError("param ranges need 0 <= lo <= hi")
    if not lo[40] > 0:
        raise ValueError("the act_dynprm0 scale must be above 0")
    ls = slice(18, 36)
    if not (np.array_equal(lo[ls][0::2], lo[ls][1::2]) and np.array_equal(hi[ls][0::2], hi[ls][1::2])):
        raise ValueError("the lower and upper ten_lengthspring of a tendon share one draw: their ranges must be equal")
    return lo, hi


# --------------------------------------------------------------------------- env config
def load_reset_poses():
    with open(os.path.join(ASSET_DIR, "reset_poses.json")) as f:
        return np.array(json.load(f)["rolling_qpos"], float)


def env_config(md, env_kind="tr_env", desired_action="straight", desired_direction=1,
               terminate_when_unhealthy=True, is_test=False, use_cap_velocity=True,
               ctrl_cost_weight=None, healthy_reward=0.1, reward_delay_seconds=None,
               min_reset_heading=0.0, max_reset_heading=2 * math.pi,
               tendon_reset_mean=None, tendon_reset_stdev=None, tendon_max_length=None, tendon_min_length=-0.45,
               way_pts_range=(2.5, 3.5), way_pts_angle_range=(-math.pi / 6, math.pi / 6),
               ditch_reward_max=300, ditch_reward_stdev=0.15, waypt_reward_amplitude=100, waypt_reward_stdev=0.10,
               yaw_reward_weight=1, max_episode_steps=5000, frame_skip=20, warmup_steps=50,
               use_obs_noise=False, obs_noise_tendon_stdev=0.02, obs_noise_cap_pos_stdev=0.05,
               reset_noise_scale=0.0, use_contact_forces=False, contact_cost_weight=5e-4, contact_force_range=None):
    """Defaults per env: tr_env.py:137-173 / tensegrity_env.py:160-181."""
    legacy = env_kind in ("tensegrity_env", ENV_LEGACY)
    c = TsgEnvConfig()
    c.struct_bytes = C.sizeof(TsgEnvConfig)
    c.env_kind = ENV_LEGACY if legacy else ENV_TR
    c.task = TASKS[desired_action]
    if legacy and desired_action not in ("straight", "turn"):
        raise ValueError("tensegrity_env supports desired_action 'straight' or 'turn'")
    c.frame_skip = frame_skip
    dt = md["timestep"] * frame_skip
    c.use_cap_velocity = int(use_cap_velocity)
    if legacy:
        c.obs_dim = 39
    else:
        c.obs_dim = 27 + (18 if use_cap_velocity else 0) + (3 if desired_action in ("tracking", "aiming", "vel_track") else 0)
    c.terminate_when_unhealthy = int(terminate_when_unhealthy)
    c.is_test = int(is_test)
    if reward_delay_seconds is None:
        reward_delay_seconds = 0.5 if legacy else 0.02
    c.reward_delay_steps = int(reward_delay_seconds / dt)
    if c.reward_delay_steps + 1 > HEADING_SLOTS:
        raise ValueError("reward_delay_seconds too long for the heading ring buffer")
    c.max_episode_steps = max_episode_steps
    c.warmup_steps = warmup_steps
    c.desired_direction = desired_direction
    c.ctrl_cost_weight = (0.001 if legacy else 0.01) if ctrl_cost_weight is None else ctrl_cost_weight
    c.healthy_reward = healthy_reward
    c.yaw_reward_weight = yaw_reward_weight
    c.min_reset_heading, c.max_reset_heading = min_reset_heading, max_reset_heading
    c.tendon_reset_mean = (-0.15 if legacy else 0.15) if tendon_reset_mean is None else tendon_reset_mean
    c.tendon_reset_stdev = (0.1 if legacy else 0.2) if tendon_reset_stdev is None else tendon_reset_stdev
    c.tendon_max_length = (-0.15 if legacy else 0.15) if tendon_max_length is None else tendon_max_length
    c.tendon_min_length = tendon_min_length
    _fill(c.waypt_range, way_pts_range)
    _fill(c.waypt_angle_range, way_pts_angle_range)
    c.ditch_reward_max, c.ditch_reward_stdev = ditch_reward_max, ditch_reward_stdev
    c.waypt_reward_amplitude, c.waypt_reward_stdev = waypt_reward_amplitude, waypt_reward_stdev
    c.kill_force = 1500.0
    if use_obs_noise and legacy:
        raise ValueError("use_obs_noise is a tr_env option (tr_env.py:142)")
    c.use_obs_noise = int(bool(use_obs_noise))          # tr_env.py:142,236
    c.obs_noise_tendon_stdev, c.obs_noise_cap_pos_stdev = obs_noise_tendon_stdev, obs_noise_cap_pos_stdev   # :161-162
    c.reset_noise_scale = float(reset_noise_scale)       # tr_env.py:152,734-743
    c.use_contact_forces = int(bool(use_contact_forces))  # tr_env.py:140,513-516
    c.contact_cost_weight = contact_cost_weight
    if contact_force_range is None:                       # tr_env.py:149-151,255-256
        contact_force_range = (-1000.0, 1000.0) if (desired_action == "turn" and not legacy) else (-1.0, 1.0)
    _fill(c.contact_force_range, contact_force_range)
    poses = np.zeros((NPOSE, NQ))
    if legacy:
        c.npose = 1
        poses[0] = md["qpos0"]          # tensegrity_env.py:439 (init_qpos)
    else:
        c.npose = NPOSE
        poses[:] = load_reset_poses()   # tr_env.py:723-728
    _fill(c.reset_pose, poses)
    return c
