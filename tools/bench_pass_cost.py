import os, sys, torch
sys.path.insert(0,os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rustyhgi_b200 as hgi
def t(fn,n=30):
    for _ in range(5): fn()
    torch.cuda.synchronize(); a=torch.cuda.Event(enable_timing=True); b=torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): fn()
    b.record(); b.synchronize(); return a.elapsed_time(b)/n*1e3
n=16384
x=torch.arange(n,device='cuda',dtype=torch.int32)
img=((x[None,:]*x[:,None])&255).to(torch.uint8).contiguous()
g=torch.empty_like(img); o=torch.empty_like(img)
ctx=hgi.Context(0)
for L in (4,5,6,8,9,12):
    enc=hgi.Encoder(hgi.Crossed,hgi.Linear(hgi.QuantizationLevel.Medium),L,ctx=ctx); dec=hgi.Decoder(hgi.Crossed,ctx=ctx)
    te=t(lambda: enc.encode_device(img,grids_out=g)); td=t(lambda: dec.decode_device(L,g,images_out=o))
    print(f"L={L}: encode {te:.1f} us, decode {td:.1f} us")
