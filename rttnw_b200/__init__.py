"""rttnw_b200 — B200-native path-tracing backend behind rttnw's scene API.

`scene`  : host mirror of the reference's Hittable / Material / Texture surface (description only)
`render` : contexts, device scenes, `render()`; every computation happens in the CUDA library
`abi`    : ctypes view of include/rttnw_b200.h (the drop-in boundary)
"""
from . import abi, scene  # noqa: F401
from .abi import RtxError  # noqa: F401
from .render import (BuiltinDesc, Context, DeviceScene, env_read, flatten_check, hdr_read, pfm_read,  # noqa: F401
                     pfm_write, png_read_rgba8, png_write_rgba8, render, scene_defaults, shard_spp)
