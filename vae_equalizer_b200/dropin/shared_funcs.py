"""Drop-in for the reference module `optical_DP_channel/shared_funcs.py` (same public names)."""
import _path  # noqa: F401
from vae_equalizer_b200.shared_funcs import *  # noqa: E402,F401,F403
from vae_equalizer_b200.shared_funcs import (BMI, CMA, CMAbatch, CMAflex, CPE, GMI, SER_constell_shaping, SER_IQflip,  # noqa: E402,F401
                                             find_shift, find_shift_symb_full, generate_data_shaping, init,
                                             loss_function_shaping, rcfir, rrcfir, simulate_channel, simulate_dispersion,
                                             soft_dec, twoXtwoFIR, bit_llr)
