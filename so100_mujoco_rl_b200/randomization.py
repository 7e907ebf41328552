"""Per-env dynamics randomisation: scale ranges for the servo gain, damping, torque limit and joint friction.

Each env of a `BatchedSo100Env` with ranges set holds its own fp32 kp, kv, forcerange and friction loss and redraws them
at every episode reset (include/so100_b200.h, so100_param_ranges; DESIGN.md "Per-env dynamics randomisation"):

    s = lo + (hi - lo) u,  u ~ U[0, 1)
    kp = kp0 s_kp,  kv = kv0 sqrt(s_kp) s_damping,  forcerange = forcerange0 s_forcerange,  frictionloss = frictionloss0 s_frictionloss

where kp0, ... are the model's values.  `damping` is the damping ratio relative to the model's.  A range (1, 1) leaves a
parameter at the model's value.

`Sim2Real` sets actuator latency (a new servo target acts from substep d of the env step, d drawn per env in [lo, hi]
at every episode reset) and Gaussian noise on the observed joint angles (include/so100_b200.h, so100_sim2real;
DESIGN.md "Actuator latency and joint-angle observation noise").
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass, field

import numpy as np

NJ = 6
FIELDS = ("kp", "damping", "forcerange", "frictionloss")
# lo must be > 0 for these (a zero gain or torque limit is not a servo), >= 0 for the others
_POSITIVE = {"kp": True, "damping": False, "forcerange": True, "frictionloss": False}


class So100ParamRanges(ctypes.Structure):
    """ctypes mirror of `so100_param_ranges`."""
    _fields_ = [("struct_size", ctypes.c_int32), ("_pad0", ctypes.c_int32)] + \
               [(f, (ctypes.c_double * 2) * NJ) for f in FIELDS]


class So100ParamView(ctypes.Structure):
    """ctypes mirror of `so100_param_view` (device pointers to [6, N] float32 arrays; NULL = skip)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("kp", "kv", "force_lo", "force_hi", "frictionloss")]


PARAM_NAMES = ("kp", "kv", "force_lo", "force_hi", "frictionloss")


def _ranges(v) -> np.ndarray:
    """(lo, hi) for every joint, or [[lo, hi]] * 6 -> float64 [6, 2]."""
    a = np.asarray(v, dtype=np.float64)
    if a.shape == (2,):
        a = np.broadcast_to(a, (NJ, 2))
    if a.shape != (NJ, 2):
        raise ValueError(f"a range is (lo, hi) or one (lo, hi) per joint ({NJ}), got shape {a.shape}")
    return np.array(a, dtype=np.float64)


@dataclass
class ParamRanges:
    """Scale ranges [lo, hi] per joint.  Each field takes a scalar pair (lo, hi), broadcast to every joint, or a [6, 2] array."""
    kp: np.ndarray = field(default_factory=lambda: (1.0, 1.0))
    damping: np.ndarray = field(default_factory=lambda: (1.0, 1.0))
    forcerange: np.ndarray = field(default_factory=lambda: (1.0, 1.0))
    frictionloss: np.ndarray = field(default_factory=lambda: (1.0, 1.0))

    def __post_init__(self):
        for f in FIELDS:
            setattr(self, f, _ranges(getattr(self, f)))
        self.validate()

    def validate(self) -> None:
        """The checks so100_set_param_ranges makes: finite fp32 bounds, lo <= hi, lo > 0 (kp, forcerange) or >= 0."""
        for f in FIELDS:
            a = getattr(self, f)
            with np.errstate(over="ignore"):
                a32 = a.astype(np.float32)
            for (lo, hi), (lo32, hi32) in zip(a, a32):
                if not (math.isfinite(lo32) and math.isfinite(hi32) and lo <= hi):
                    raise ValueError(f"{f}: every range needs finite bounds with lo <= hi, got ({lo}, {hi})")
                if _POSITIVE[f] and not lo > 0:
                    raise ValueError(f"{f}: lo must be > 0, got {lo}")
                if not _POSITIVE[f] and not lo >= 0:
                    raise ValueError(f"{f}: lo must be >= 0, got {lo}")

    def to_ctypes(self) -> So100ParamRanges:
        r = So100ParamRanges()
        r.struct_size = ctypes.sizeof(So100ParamRanges)
        for f in FIELDS:
            a = getattr(self, f)
            dst = getattr(r, f)
            for j in range(NJ):
                dst[j][0], dst[j][1] = float(a[j, 0]), float(a[j, 1])
        return r

    def to_dict(self) -> dict:
        return {f: getattr(self, f).tolist() for f in FIELDS}

    @classmethod
    def from_dict(cls, d: dict) -> "ParamRanges":
        return cls(**{f: d[f] for f in FIELDS})

    def lo_hi_f32(self) -> tuple[np.ndarray, np.ndarray]:
        """fp32 lo, hi [24] in draw order (kp[6], damping[6], forcerange[6], frictionloss[6]), as the kernel holds them."""
        a = np.concatenate([getattr(self, f) for f in FIELDS]).astype(np.float32)
        return a[:, 0].copy(), a[:, 1].copy()

    @classmethod
    def parse(cls, spec: str) -> "ParamRanges":
        """`"kp=0.7:1.3,damping=0.8:1.2,forcerange=0.8:1.0,frictionloss=0.5:2"`; fields left out stay at 1:1."""
        kw = {}
        for part in (p.strip() for p in spec.split(",")):
            if not part:
                continue
            name, eq, rng = part.partition("=")
            name = name.strip()
            if not eq or name not in FIELDS:
                raise ValueError(f"bad range {part!r}: expected <field>=lo:hi with field one of {', '.join(FIELDS)}")
            if name in kw:
                raise ValueError(f"{name} given twice")
            lo, colon, hi = rng.partition(":")
            if not colon:
                raise ValueError(f"bad range {part!r}: expected lo:hi")
            try:
                kw[name] = (float(lo), float(hi))
            except ValueError:
                raise ValueError(f"bad range {part!r}: bounds must be numbers") from None
        return cls(**kw)


def parse(spec: str) -> ParamRanges:
    return ParamRanges.parse(spec)


# ---------------------------------------------------------------------------------------------------------------- sim2real
class So100Sim2Real(ctypes.Structure):
    """ctypes mirror of `so100_sim2real`."""
    _fields_ = [("struct_size", ctypes.c_int32), ("latency", ctypes.c_int32 * 2), ("_pad0", ctypes.c_int32),
                ("obs_noise", ctypes.c_double * NJ)]


class So100ActuatorView(ctypes.Structure):
    """ctypes mirror of `so100_actuator_view` (device pointers: latency [N] int32, ctrl_prev_hi / _lo [6, N] float32)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("latency", "ctrl_prev_hi", "ctrl_prev_lo")]


ACTUATOR_NAMES = ("latency", "ctrl_prev_hi", "ctrl_prev_lo")


@dataclass
class Sim2Real:
    """Actuator latency in substeps, drawn per env in [lo, hi] at every episode reset, and the std (rad) of the Gaussian
    noise on each observed joint angle (a scalar for every joint, or 6 values).  Neither has a default that stands for the
    physical arm: both are the user's to set."""
    latency: tuple = (0, 0)
    obs_noise: np.ndarray = 0.0

    def __post_init__(self):
        lat = tuple(self.latency)
        if len(lat) != 2 or not all(isinstance(x, (int, np.integer)) and not isinstance(x, bool) for x in lat):
            raise ValueError(f"latency is (lo, hi) in whole substeps, got {self.latency!r}")
        self.latency = (int(lat[0]), int(lat[1]))
        a = np.asarray(self.obs_noise, dtype=np.float64)
        if a.shape == ():
            a = np.full(NJ, float(a))
        if a.shape != (NJ,):
            raise ValueError(f"obs_noise is one std or one per joint ({NJ}), got shape {a.shape}")
        self.obs_noise = a
        self.validate(nsubstep=math.inf)  # the upper latency bound is the model's: checked where the model is known

    def validate(self, nsubstep: int | None = None, task: int | None = None) -> None:
        """The checks so100_set_sim2real makes: 0 <= lo <= hi <= nsubstep (the model's, by default the so100 model's),
        finite fp32 std >= 0, and no noise on Env05 (task 5), whose observed angles are its exact commands."""
        if nsubstep is None:
            from .model import ModelSpec
            nsubstep = ModelSpec.__dataclass_fields__["nsubstep"].default
        lo, hi = self.latency
        if not 0 <= lo <= hi <= nsubstep:
            raise ValueError(f"latency: need 0 <= lo <= hi <= nsubstep ({nsubstep}), got ({lo}, {hi})")
        with np.errstate(over="ignore"):
            a32 = self.obs_noise.astype(np.float32)
        for s, s32 in zip(self.obs_noise, a32):
            if not (math.isfinite(s32) and s >= 0):
                raise ValueError(f"obs_noise: every std must be finite and >= 0, got {s}")
        if task == 5 and (a32 != 0).any():
            raise ValueError("obs_noise: Env05 observes its commanded angles, which carry no noise")

    def to_ctypes(self) -> So100Sim2Real:
        c = So100Sim2Real()
        c.struct_size = ctypes.sizeof(So100Sim2Real)
        c.latency[0], c.latency[1] = self.latency
        for j in range(NJ):
            c.obs_noise[j] = float(self.obs_noise[j])
        return c

    def to_dict(self) -> dict:
        return {"latency": list(self.latency), "obs_noise": self.obs_noise.tolist()}

    @classmethod
    def from_dict(cls, d: dict) -> "Sim2Real":
        return cls(latency=tuple(d["latency"]), obs_noise=d["obs_noise"])

    @staticmethod
    def parse_latency(spec: str) -> tuple[int, int]:
        """`"LO:HI"` (or `"D"` for a fixed latency) in substeps."""
        lo, colon, hi = spec.strip().partition(":")
        try:
            return (int(lo), int(hi if colon else lo))
        except ValueError:
            raise ValueError(f"bad latency {spec!r}: expected LO:HI in whole substeps") from None
