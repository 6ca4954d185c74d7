"""TEST INFRASTRUCTURE ONLY -- named model shapes shared by the fixture generator and the tests.
Shapes come from the reference's yaml configs (SURVEY.md Appendix A); the "tiny" ones are ours, for fast tests."""

AR_ZOO = {
    # name: (E, heads, n_body, n_head_layers, V, block_size, vocab_cond, cond_len)
    "tiny": (128, 2, 2, 2, 512, (4, 4, 4), 10, 1),
    "tiny_txt": (128, 2, 2, 2, 512, (3, 3, 4), 16, 4),
    "ffhq355m": (1024, 16, 24, 4, 2048, (8, 8, 4), 1, 1),        # configs/ffhq/stage2/ffhq256-rqtransformer-8x8x4-350M.yaml:7-30
    "in1400m": (1536, 24, 42, 6, 16384, (8, 8, 4), 1000, 1),     # configs/imagenet256/stage2/in256-rqtransformer-8x8x4-1400M.yaml:7-30
    "cc3m654m": (1280, 20, 26, 4, 16384, (8, 8, 4), 16384, 32),  # configs/cc3m/cc3m-rqtransformer-8x8x4-650M.yaml:11-34
    # BASELINE configs 4 / 5 shapes the reference does not ship as yaml (SURVEY finding 8): the 654M widths on a synthetic 16x16x4
    # grid (measure_throughput f=16), and the "3.9B" text-to-image arch = the 3800M widths (README.md:47,72) + a 32-token prefix
    "cc3m654m_16": (1280, 20, 26, 4, 16384, (16, 16, 4), 16384, 32),
    "t2i3900m": (2560, 40, 42, 6, 16384, (8, 8, 4), 16384, 32),
}
VAE_ZOO = {
    "tiny": dict(K=512, code_shape=(4, 4, 4), ch=32, ch_mult=(1, 2, 4), attn_resolutions=(4,), resolution=16),
    "tiny_attn_mid": dict(K=512, code_shape=(4, 4, 4), ch=32, ch_mult=(1, 1, 2, 4), attn_resolutions=(8,), resolution=32),
    "ffhq": dict(K=2048, attn_resolutions=(16,)),                 # configs/ffhq/stage1/ffhq256-rqvae-8x8x4.yaml:12,30
    "imagenet": dict(K=16384, attn_resolutions=(8,)),             # configs/imagenet256/stage1/in256-rqvae-8x8x4.yaml:12,30
}

# golden files of the reference's AR trajectories beyond tests/golden/ar.pt, split so that every file stays under 1 MB
AR2_FILES = {"ar2": ("cc3m654m",), "ar3": ("cc3m654m_16", "t2i3900m")}


def ar_fixture(name):
    """the tests/golden/<fixture>.pt holding the reference's AR trajectories of model `name`"""
    return next((f for f, names in AR2_FILES.items() if name in names), "ar")


def vae_ddconfig(K, code_shape=(8, 8, 4), embed_dim=256, ch=128, ch_mult=(1, 1, 2, 2, 4, 4), attn_resolutions=(8,),
                 resolution=256, z_channels=256, num_res_blocks=2):
    return dict(double_z=False, z_channels=z_channels, resolution=resolution, in_channels=3, out_ch=3, ch=ch,
                ch_mult=list(ch_mult), num_res_blocks=num_res_blocks, attn_resolutions=list(attn_resolutions), dropout=0.0)
