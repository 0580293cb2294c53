"""ctypes binding of csrc/libsnnk.so (the C ABI declared in include/snnk.h).

There is NO fallback: if the shared library is missing, or the device is not a B200 (sm_100), every
compute call raises.  The library is built in-tree by ``__graft_entry__.build()`` / ``build_extension()``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libsnnk.so")
# measuring switch: a differently built copy of the SAME library (kernel experiments); never a fallback
LIB_PATH = os.environ.get("SNNK_LIB_PATH", LIB_PATH)
INCLUDE = os.path.join(os.path.dirname(_HERE), "include", "snnk.h")

SNNK_LIF, SNNK_ALIF, SNNK_IZHIKEVICH = 0, 1, 2
SNNK_FAST_SIGMOID, SNNK_PHI, SNNK_SURROGATE_TRACE = 0, 1, 2
SNNK_F32, SNNK_F64, SNNK_U8, SNNK_I64, SNNK_BITS = 0, 1, 2, 3, 4
SNNK_F_TRACES, SNNK_F_TENSOR_CORE, SNNK_F_INPUT_BINARY, SNNK_F_INPUT_BITS, SNNK_F_RUNS_TILED = 0x1, 0x2, 0x4, 0x8, 0x10
SNNK_F_SWEEP_DONE = 0x20
SNNK_ERR_UNSUPPORTED = -6
SNNK_MAX_CLASSES = 16   # widest readout the kernels take (SnnkDesc.O <= 16, kOMax in csrc/common.cuh)

NVCC_FLAGS = [
	"-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
	"-Xcompiler", "-fPIC", "-shared",
]


class SnnkDesc(ctypes.Structure):
	"""Mirror of ``struct SnnkDesc`` (include/snnk.h)."""
	_fields_ = [
		("B", ctypes.c_int32), ("T", ctypes.c_int32), ("N", ctypes.c_int32), ("H", ctypes.c_int32),
		("O", ctypes.c_int32), ("layer_type", ctypes.c_int32), ("surrogate", ctypes.c_int32),
		("recurrent", ctypes.c_int32), ("alpha", ctypes.c_float), ("rho", ctypes.c_float),
		("theta", ctypes.c_float), ("gamma", ctypes.c_float), ("kappa", ctypes.c_float),
		("flags", ctypes.c_uint32),
		# SNNK_IZHIKEVICH only
		("dt", ctypes.c_float), ("iz_C", ctypes.c_float), ("iz_v_rest", ctypes.c_float), ("iz_v_th", ctypes.c_float),
		("iz_k", ctypes.c_float), ("iz_a", ctypes.c_float), ("iz_b", ctypes.c_float), ("iz_c", ctypes.c_float),
		("iz_d", ctypes.c_float), ("iz_v_peak", ctypes.c_float),
	]


def build_extension(force: bool = False, verbose: bool = False) -> str:
	"""Compile csrc/*.cu for sm_100a into csrc/libsnnk.so (nvcc cross-compiles without a GPU)."""
	srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))] + [INCLUDE]
	if not force and os.path.exists(LIB_PATH):
		if os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(s) for s in srcs):
			return LIB_PATH
	nvcc = os.environ.get("NVCC", "nvcc")
	cmd = [nvcc] + NVCC_FLAGS + ["-o", LIB_PATH, os.path.join(CSRC, "snnk.cu")]
	res = subprocess.run(cmd, capture_output=True, text=True)
	if verbose or res.returncode != 0:
		print(" ".join(cmd))
		print(res.stdout, res.stderr)
	if res.returncode != 0:
		raise RuntimeError("nvcc failed building libsnnk.so:\n" + res.stderr)
	return LIB_PATH


_lib = None
_p = ctypes.c_void_p

_SIGNATURES = {
	"snnk_abi_version": (ctypes.c_int, []),
	"snnk_strerror": (ctypes.c_char_p, [ctypes.c_int]),
	"snnk_last_cuda_error": (ctypes.c_char_p, []),
	"snnk_device_supported": (ctypes.c_int, []),
	"snnk_kernel_name": (ctypes.c_char_p, [ctypes.c_int]),
	"snnk_profile_begin": (ctypes.c_int, []),
	"snnk_profile_end": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)]),
	"snnk_encode": (ctypes.c_int, [
		_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_double,
		ctypes.c_double, ctypes.c_double, ctypes.c_int32, _p, ctypes.c_int32, _p, _p]),
	"snnk_spike_forward": (ctypes.c_int, [_p, _p, ctypes.c_int64, ctypes.c_int64, _p, _p]),
	"snnk_spike_backward": (ctypes.c_int, [ctypes.c_int32, _p, _p, _p, _p, ctypes.c_int64, ctypes.c_int64, _p, _p]),
	"snnk_forward_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(SnnkDesc)]),
	"snnk_backward_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(SnnkDesc)]),
	"snnk_unpack_raster": (ctypes.c_int, [_p, ctypes.c_int64, ctypes.c_int32, _p, _p]),
	"snnk_run_table_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int32]),
	"snnk_run_table_tiled_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32]),
	"snnk_frame_runs": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, _p, _p, _p]),
	"snnk_encode_runs": (ctypes.c_int, [
		_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_double,
		ctypes.c_double, ctypes.c_double, ctypes.c_int32, _p, ctypes.c_int32, _p, _p, _p, ctypes.c_int32, _p]),
	"snnk_forward": (ctypes.c_int, [ctypes.POINTER(SnnkDesc)] + [_p] * 18 + [ctypes.c_size_t, _p, _p, _p]),
	"snnk_forward_nll": (ctypes.c_int, [ctypes.POINTER(SnnkDesc)] + [_p] * 18 + [ctypes.c_size_t, _p, _p] + [_p] * 7 + [_p]),
	"snnk_forward_nll_sweep": (ctypes.c_int, [ctypes.POINTER(SnnkDesc)] + [_p] * 18 + [ctypes.c_size_t, _p, _p] + [_p] * 7
		+ [_p, _p, ctypes.c_size_t, _p]),
	"snnk_head_nll": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, _p, _p, _p, _p, _p, _p, _p, _p]),
	"snnk_input_grad": (ctypes.c_int, [ctypes.POINTER(SnnkDesc), _p, _p, _p, _p]),
	"snnk_backward": (ctypes.c_int, [ctypes.POINTER(SnnkDesc)] + [_p] * 21 + [ctypes.c_size_t, _p, _p, _p]),
	"snnk_adam_step": (ctypes.c_int, [ctypes.c_int32, _p, _p, _p, _p, _p, _p, ctypes.c_float, ctypes.c_float,
		ctypes.c_float, ctypes.c_float, ctypes.c_float, _p]),
	"snnk_adam_dp_buffer_bytes": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int64, ctypes.POINTER(ctypes.c_size_t)]),
	"snnk_adam_step_dp": (ctypes.c_int, [ctypes.c_int32, _p, _p, _p, _p, _p, _p, ctypes.c_float, ctypes.c_float,
		ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_int32, ctypes.c_int32, _p, _p, _p]),
}
EXPORTS = tuple(_SIGNATURES)


def lib() -> ctypes.CDLL:
	"""Loads libsnnk.so; raises (never falls back) when it has not been built."""
	global _lib
	if _lib is None:
		if not os.path.exists(LIB_PATH):
			raise RuntimeError(
				f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
				"`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). There is no CPU or PyTorch "
				"fallback for the spiking hot path.")
		l = ctypes.CDLL(LIB_PATH)
		for name, (res, args) in _SIGNATURES.items():
			fn = getattr(l, name)
			fn.restype = res
			fn.argtypes = args
		if l.snnk_abi_version() != 8:
			raise RuntimeError("libsnnk.so ABI version mismatch; rebuild the extension")
		_lib = l
	return _lib


SNNK_K_COUNT = 12


class kernel_profile:
	"""Context manager around snnk_profile_begin/end -> {kernel name: (total ms, launches)} in ``.result``."""

	def __enter__(self):
		check(lib().snnk_profile_begin(), "snnk_profile_begin")
		self.result = {}
		return self

	def __exit__(self, *exc):
		ms = (ctypes.c_double * SNNK_K_COUNT)()
		n = (ctypes.c_int64 * SNNK_K_COUNT)()
		check(lib().snnk_profile_end(ms, n), "snnk_profile_end")
		for k in range(SNNK_K_COUNT):
			if n[k]:
				self.result[lib().snnk_kernel_name(k).decode()] = (float(ms[k]), int(n[k]))
		return False


def check(rc: int, what: str) -> None:
	if rc != 0:
		l = lib()
		msg = l.snnk_strerror(rc).decode()
		detail = l.snnk_last_cuda_error().decode() if rc == -5 else ""
		raise RuntimeError(f"{what} failed: {msg}" + (f" [{detail}]" if detail else ""))


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
	"""Device pointer of a contiguous CUDA tensor (None -> NULL)."""
	if t is None:
		return None
	if not t.is_cuda:
		raise RuntimeError(
			"the B200 spiking path needs CUDA tensors (got a CPU tensor); there is no CPU fallback")
	if not t.is_contiguous():
		raise RuntimeError("internal error: non-contiguous tensor handed to the C ABI")
	return t.data_ptr()


def stream_ptr() -> int:
	return torch.cuda.current_stream().cuda_stream


def require_b200(device: torch.device) -> None:
	"""Raises unless ``device`` is a CUDA device the library supports (sm_100)."""
	if device.type != "cuda":
		raise RuntimeError(
			f"the B200-native spiking path runs on CUDA sm_100 only (model device is '{device}'); "
			"there is no CPU fallback")
	with torch.cuda.device(device):
		if lib().snnk_device_supported() != 1:
			raise RuntimeError(f"CUDA device {device} is not sm_100 (B200); there is no fallback path")
