import sys, ctypes as C, torch
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from vit_flax_b200 import _lib
lib=_lib.load()
b,T,h=map(int,sys.argv[1:4])
inner=h*64
qkv=(torch.randn((b*T,3*inner),device='cuda')*1.5).half()
out=torch.zeros((b*T,inner),device='cuda',dtype=torch.float16)
st=C.c_void_p(torch.cuda.current_stream().cuda_stream)
_lib.check(lib.vitb200_attention_tc(st,qkv.data_ptr(),out.data_ptr(),b,T,h,_lib.DT_F16))
torch.cuda.synchronize()
print('ok',b,T,h)
