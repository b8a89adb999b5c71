"""ctypes binding of libcgan_b200.so (the C-ABI declared in include/cgan_b200.h).

The prototypes are parsed from the header itself, so the Python side can never drift from the
C-ABI, and `tests/test_abi.py` can check that the library exports every declared symbol.
There is NO fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, "..", "include", "cgan_b200.h")
SO_PATH = os.path.join(HERE, "csrc", "libcgan_b200.so")


class ConvDesc(ctypes.Structure):
  """cgan_conv_desc (include/cgan_b200.h)."""
  _fields_ = [(n, ctypes.c_int32) for n in
              ("n", "h", "w", "cin", "cout", "kh", "kw", "stride", "upsample", "oh", "ow", "pad_t", "pad_l")]


class ConvEpilogue(ctypes.Structure):
  """cgan_conv_epilogue (include/cgan_b200.h)."""
  _fields_ = [("bias", ctypes.c_void_p), ("residual", ctypes.c_void_p), ("mask", ctypes.c_void_p),
              ("mask_leak", ctypes.c_float), ("flags", ctypes.c_int32), ("ldy", ctypes.c_int32)]


CONV_RELU, CONV_ROUND_OUT, CONV_IN_TF32, CONV_IN2_TF32 = 1, 2, 4, 8
ACT_ROUND_TF32 = 0x100
OPT_TC_MT, OPT_LAST_PATH, OPT_TC_HALO, OPT_TC_THIN = 1, 2, 3, 6
PATH_NAMES = {0: "simt_fp32", 1: "tcgen05_tf32", 2: "thin_fp32"}

_SCALARS = {"int": ctypes.c_int, "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64,
            "float": ctypes.c_float, "size_t": ctypes.c_size_t, "uint64_t": ctypes.c_uint64}


def parse_header(path=HEADER):
  """Returns {name: (restype, [argtypes])} for every function the header declares."""
  src = open(path).read()
  src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
  src = re.sub(r"//[^\n]*", " ", src)
  protos = {}
  for m in re.finditer(r"(const\s+char\s*\*|int64_t|int)\s+(cgan_\w+)\s*\(([^;{]*)\)\s*;", src):
    ret, name, args = m.group(1), m.group(2), m.group(3)
    restype = ctypes.c_char_p if "char" in ret else (ctypes.c_int64 if ret == "int64_t" else ctypes.c_int)
    argtypes = []
    args = args.strip()
    if args and args != "void":
      for a in args.split(","):
        a = a.strip()
        if "*" in a:
          argtypes.append(ctypes.c_void_p)
        else:
          ty = a.replace("const", "").split()[0]
          argtypes.append(_SCALARS[ty])
    protos[name] = (restype, argtypes)
  return protos


class CganError(RuntimeError):
  pass


_DLL = {}


def load_functions(so_path=SO_PATH):
  """Loads the shared library and returns (dll, protos, {name: typed function}) without creating a device context —
  all the host-side input pipeline (cgan_loader_*) needs."""
  if so_path not in _DLL:
    if not os.path.exists(so_path):
      raise CganError("libcgan_b200.so not found at %s — run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU / PyTorch fallback for the product path)" % so_path)
    dll = ctypes.CDLL(so_path)
    protos = parse_header()
    fn = {}
    for name, (restype, argtypes) in protos.items():
      f = getattr(dll, name)       # AttributeError if the symbol is not exported
      f.restype = restype
      f.argtypes = argtypes
      fn[name] = f
    _DLL[so_path] = (dll, protos, fn)
  return _DLL[so_path]


class Lib(object):
  """Loaded library + one context bound to one CUDA device."""

  def __init__(self, device=0, so_path=SO_PATH):
    self.dll, self.protos, self.fn = load_functions(so_path)
    self.ctx = ctypes.c_void_p()
    rc = self.fn["cgan_ctx_create"](ctypes.byref(self.ctx), device)
    if rc != 0:
      raise CganError("cgan_ctx_create(device=%d) failed with code %d (no CUDA device?)" % (device, rc))
    self.device = device

  def call(self, name, *args):
    rc = self.fn["cgan_" + name](self.ctx, *args)
    if rc != 0:
      raise CganError("cgan_%s failed (%d): %s" % (name, rc, self.fn["cgan_last_error"](self.ctx).decode()))

  def set_stream(self, stream_ptr):
    self.call("ctx_set_stream", stream_ptr)

  def launch_count(self):
    return int(self.fn["cgan_launch_count"](self.ctx))

  def set_option(self, key, value):
    self.call("ctx_set_option", int(key), int(value))

  def get_option(self, key):
    v = ctypes.c_int64(0)
    self.call("ctx_get_option", int(key), ctypes.byref(v))
    return int(v.value)

  def attention_supported(self, batch, lq, lk, dk, dv):
    """cgan_attention_supported: 1 / 0, not an error code."""
    return bool(self.fn["cgan_attention_supported"](self.ctx, int(batch), int(lq), int(lk), int(dk), int(dv)))

  def close(self):
    if self.ctx:
      self.fn["cgan_ctx_destroy"](self.ctx)
      self.ctx = ctypes.c_void_p()


_LIBS = {}


def get_lib(device=0):
  if device not in _LIBS:
    _LIBS[device] = Lib(device)
  return _LIBS[device]
