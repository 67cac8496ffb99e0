import torch, ofdm_b200 as m
from torch.profiler import profile, ProfilerActivity
dev = torch.device("cuda:0")
for (A, N, C, S, U, F) in ((64, 1024, 64, 101, 1, 64), (64, 1024, 64, 101, 4, 64), (256, 4096, 288, 14, 4, 32), (256, 4096, 288, 20, 16, 32)):
    K = N - 1
    rx, pil, _ = m.synth.make_frames_mu_torch(F, A, N, C, S, 4, U, dev, seed=1, chunk=1)
    comb = torch.empty((F, S - U, U, K), dtype=torch.complex64, device=dev)
    bits = torch.empty((F, S - U, U, (K * 4 + 7) // 8), dtype=torch.uint8, device=dev)
    hc = torch.empty((F, U, A, K), dtype=torch.complex64, device=dev)
    st = torch.cuda.Stream(dev)
    with m.LsMrcReceiver(A, N, C, S, 4) as r, torch.cuda.stream(st):
        r.set_pilot(pil); r.set_stream(st.cuda_stream)
        for _ in range(2): r.demod_frames_device_mu(rx, F, U, comb, bits, hc)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(3): r.demod_frames_device_mu(rx, F, U, comb, bits, hc)
            torch.cuda.synchronize()
        r.set_stream(None)
    print("A N S U F =", A, N, S, U, F)
    for e in sorted(p.key_averages(), key=lambda e: -e.device_time_total)[:6]:
        print(f"  {e.device_time_total/3/1000:9.3f} ms/call  {e.key[:80]}")
    del rx, comb, bits, hc; torch.cuda.empty_cache()
