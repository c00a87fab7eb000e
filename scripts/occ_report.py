import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from edgerunner_b200 import _lib
lib = C.CDLL(_lib.LIB_PATH)
torch.zeros(1, device='cuda')
buf = C.create_string_buffer(4096)
for smem in (215424, 190720, 166016):
    lib.er_debug_decode_report(buf, 4096, C.c_ulonglong(smem))
    print(buf.value.decode())
