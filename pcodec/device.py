"""pcodec.device: device-resident files for PyTorch (compress a CUDA tensor, decompress asynchronously on the current stream)."""
from pcodec_b200.device import *  # noqa: F401,F403
from pcodec_b200.device import AsyncStatus, DeviceFile, compress, decompress, prepare, workspace_bytes  # noqa: F401
