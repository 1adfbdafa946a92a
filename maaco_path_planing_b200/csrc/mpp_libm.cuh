// mpp_libm.cuh -- mpp_exp / mpp_pow: __host__ __device__ replicas of the exp and pow of glibc 2.39's x86-64 libm as it
// runs on a CPU with FMA and AVX2 (the `__exp_fma` / `__pow_fma` ifunc variants, both ARM optimized-routines code).
// Each result is bit for bit the host's: the constants and tables below are the library's `__exp_data` /
// `__pow_log_data`, and every fma() stands where that build has a vfmadd (GCC contracted some a*b+c of the C source,
// not others), so the rest of the arithmetic must not be contracted -- device code is compiled with -fmad=false and
// host code with -ffp-contract=off.
//
// Domain: mpp_exp, every double.  mpp_pow, x in [+0, +inf] (not NaN, not negative) and every y, NaN included: MAACO's
// eta'^beta tables (MAACO.py:197-210) only take pow(1/d, beta) with d >= 1e-9.  NaN results are the quieted NaN the x86
// code returns, built from bits so that no device NaN canonicalisation can change them.
// Device code reads the tables from read-only global memory (6 KB, L1 / L2 resident: a whole 128-map 256^2 table build
// takes 0.15 ms on a B200, so staging them in shared memory was not tried); each translation unit that includes this
// header gets its own copy.
#pragma once
#include <stdint.h>
#include <string.h>
#include <math.h>

#ifdef __CUDACC__
#define MPP_LIBM_FN __host__ __device__ __forceinline__
#else
#define MPP_LIBM_FN static inline
#endif

#define MPP_LIBM_EXP_TAB {  \
    0x0000000000000000ull, 0x3ff0000000000000ull, 0x3c9b3b4f1a88bf6eull, 0x3feff63da9fb3335ull, \
    0xbc7160139cd8dc5dull, 0x3fefec9a3e778061ull, 0xbc905e7a108766d1ull, 0x3fefe315e86e7f85ull, \
    0x3c8cd2523567f613ull, 0x3fefd9b0d3158574ull, 0xbc8bce8023f98efaull, 0x3fefd06b29ddf6deull, \
    0x3c60f74e61e6c861ull, 0x3fefc74518759bc8ull, 0x3c90a3e45b33d399ull, 0x3fefbe3ecac6f383ull, \
    0x3c979aa65d837b6dull, 0x3fefb5586cf9890full, 0x3c8eb51a92fdeffcull, 0x3fefac922b7247f7ull, \
    0x3c3ebe3d702f9cd1ull, 0x3fefa3ec32d3d1a2ull, 0xbc6a033489906e0bull, 0x3fef9b66affed31bull, \
    0xbc9556522a2fbd0eull, 0x3fef9301d0125b51ull, 0xbc5080ef8c4eea55ull, 0x3fef8abdc06c31ccull, \
    0xbc91c923b9d5f416ull, 0x3fef829aaea92de0ull, 0x3c80d3e3e95c55afull, 0x3fef7a98c8a58e51ull, \
    0xbc801b15eaa59348ull, 0x3fef72b83c7d517bull, 0xbc8f1ff055de323dull, 0x3fef6af9388c8deaull, \
    0x3c8b898c3f1353bfull, 0x3fef635beb6fcb75ull, 0xbc96d99c7611eb26ull, 0x3fef5be084045cd4ull, \
    0x3c9aecf73e3a2f60ull, 0x3fef54873168b9aaull, 0xbc8fe782cb86389dull, 0x3fef4d5022fcd91dull, \
    0x3c8a6f4144a6c38dull, 0x3fef463b88628cd6ull, 0x3c807a05b0e4047dull, 0x3fef3f49917ddc96ull, \
    0x3c968efde3a8a894ull, 0x3fef387a6e756238ull, 0x3c875e18f274487dull, 0x3fef31ce4fb2a63full, \
    0x3c80472b981fe7f2ull, 0x3fef2b4565e27cddull, 0xbc96b87b3f71085eull, 0x3fef24dfe1f56381ull, \
    0x3c82f7e16d09ab31ull, 0x3fef1e9df51fdee1ull, 0xbc3d219b1a6fbffaull, 0x3fef187fd0dad990ull, \
    0x3c8b3782720c0ab4ull, 0x3fef1285a6e4030bull, 0x3c6e149289cecb8full, 0x3fef0cafa93e2f56ull, \
    0x3c834d754db0abb6ull, 0x3fef06fe0a31b715ull, 0x3c864201e2ac744cull, 0x3fef0170fc4cd831ull, \
    0x3c8fdd395dd3f84aull, 0x3feefc08b26416ffull, 0xbc86a3803b8e5b04ull, 0x3feef6c55f929ff1ull, \
    0xbc924aedcc4b5068ull, 0x3feef1a7373aa9cbull, 0xbc9907f81b512d8eull, 0x3feeecae6d05d866ull, \
    0xbc71d1e83e9436d2ull, 0x3feee7db34e59ff7ull, 0xbc991919b3ce1b15ull, 0x3feee32dc313a8e5ull, \
    0x3c859f48a72a4c6dull, 0x3feedea64c123422ull, 0xbc9312607a28698aull, 0x3feeda4504ac801cull, \
    0xbc58a78f4817895bull, 0x3feed60a21f72e2aull, 0xbc7c2c9b67499a1bull, 0x3feed1f5d950a897ull, \
    0x3c4363ed60c2ac11ull, 0x3feece086061892dull, 0x3c9666093b0664efull, 0x3feeca41ed1d0057ull, \
    0x3c6ecce1daa10379ull, 0x3feec6a2b5c13cd0ull, 0x3c93ff8e3f0f1230ull, 0x3feec32af0d7d3deull, \
    0x3c7690cebb7aafb0ull, 0x3feebfdad5362a27ull, 0x3c931dbdeb54e077ull, 0x3feebcb299fddd0dull, \
    0xbc8f94340071a38eull, 0x3feeb9b2769d2ca7ull, 0xbc87deccdc93a349ull, 0x3feeb6daa2cf6642ull, \
    0xbc78dec6bd0f385full, 0x3feeb42b569d4f82ull, 0xbc861246ec7b5cf6ull, 0x3feeb1a4ca5d920full, \
    0x3c93350518fdd78eull, 0x3feeaf4736b527daull, 0x3c7b98b72f8a9b05ull, 0x3feead12d497c7fdull, \
    0x3c9063e1e21c5409ull, 0x3feeab07dd485429ull, 0x3c34c7855019c6eaull, 0x3feea9268a5946b7ull, \
    0x3c9432e62b64c035ull, 0x3feea76f15ad2148ull, 0xbc8ce44a6199769full, 0x3feea5e1b976dc09ull, \
    0xbc8c33c53bef4da8ull, 0x3feea47eb03a5585ull, 0xbc845378892be9aeull, 0x3feea34634ccc320ull, \
    0xbc93cedd78565858ull, 0x3feea23882552225ull, 0x3c5710aa807e1964ull, 0x3feea155d44ca973ull, \
    0xbc93b3efbf5e2228ull, 0x3feea09e667f3bcdull, 0xbc6a12ad8734b982ull, 0x3feea012750bdabfull, \
    0xbc6367efb86da9eeull, 0x3fee9fb23c651a2full, 0xbc80dc3d54e08851ull, 0x3fee9f7df9519484ull, \
    0xbc781f647e5a3ecfull, 0x3fee9f75e8ec5f74ull, 0xbc86ee4ac08b7db0ull, 0x3fee9f9a48a58174ull, \
    0xbc8619321e55e68aull, 0x3fee9feb564267c9ull, 0x3c909ccb5e09d4d3ull, 0x3feea0694fde5d3full, \
    0xbc7b32dcb94da51dull, 0x3feea11473eb0187ull, 0x3c94ecfd5467c06bull, 0x3feea1ed0130c132ull, \
    0x3c65ebe1abd66c55ull, 0x3feea2f336cf4e62ull, 0xbc88a1c52fb3cf42ull, 0x3feea427543e1a12ull, \
    0xbc9369b6f13b3734ull, 0x3feea589994cce13ull, 0xbc805e843a19ff1eull, 0x3feea71a4623c7adull, \
    0xbc94d450d872576eull, 0x3feea8d99b4492edull, 0x3c90ad675b0e8a00ull, 0x3feeaac7d98a6699ull, \
    0x3c8db72fc1f0eab4ull, 0x3feeace5422aa0dbull, 0xbc65b6609cc5e7ffull, 0x3feeaf3216b5448cull, \
    0x3c7bf68359f35f44ull, 0x3feeb1ae99157736ull, 0xbc93091fa71e3d83ull, 0x3feeb45b0b91ffc6ull, \
    0xbc5da9b88b6c1e29ull, 0x3feeb737b0cdc5e5ull, 0xbc6c23f97c90b959ull, 0x3feeba44cbc8520full, \
    0xbc92434322f4f9aaull, 0x3feebd829fde4e50ull, 0xbc85ca6cd7668e4bull, 0x3feec0f170ca07baull, \
    0x3c71affc2b91ce27ull, 0x3feec49182a3f090ull, 0x3c6dd235e10a73bbull, 0x3feec86319e32323ull, \
    0xbc87c50422622263ull, 0x3feecc667b5de565ull, 0x3c8b1c86e3e231d5ull, 0x3feed09bec4a2d33ull, \
    0xbc91bbd1d3bcbb15ull, 0x3feed503b23e255dull, 0x3c90cc319cee31d2ull, 0x3feed99e1330b358ull, \
    0x3c8469846e735ab3ull, 0x3feede6b5579fdbfull, 0xbc82dfcd978e9db4ull, 0x3feee36bbfd3f37aull, \
    0x3c8c1a7792cb3387ull, 0x3feee89f995ad3adull, 0xbc907b8f4ad1d9faull, 0x3feeee07298db666ull, \
    0xbc55c3d956dcaebaull, 0x3feef3a2b84f15fbull, 0xbc90a40e3da6f640ull, 0x3feef9728de5593aull, \
    0xbc68d6f438ad9334ull, 0x3feeff76f2fb5e47ull, 0xbc91eee26b588a35ull, 0x3fef05b030a1064aull, \
    0x3c74ffd70a5fddcdull, 0x3fef0c1e904bc1d2ull, 0xbc91bdfbfa9298acull, 0x3fef12c25bd71e09ull, \
    0x3c736eae30af0cb3ull, 0x3fef199bdd85529cull, 0x3c8ee3325c9ffd94ull, 0x3fef20ab5fffd07aull, \
    0x3c84e08fd10959acull, 0x3fef27f12e57d14bull, 0x3c63cdaf384e1a67ull, 0x3fef2f6d9406e7b5ull, \
    0x3c676b2c6c921968ull, 0x3fef3720dcef9069ull, 0xbc808a1883ccb5d2ull, 0x3fef3f0b555dc3faull, \
    0xbc8fad5d3ffffa6full, 0x3fef472d4a07897cull, 0xbc900dae3875a949ull, 0x3fef4f87080d89f2ull, \
    0x3c74a385a63d07a7ull, 0x3fef5818dcfba487ull, 0xbc82919e2040220full, 0x3fef60e316c98398ull, \
    0x3c8e5a50d5c192acull, 0x3fef69e603db3285ull, 0x3c843a59ac016b4bull, 0x3fef7321f301b460ull, \
    0xbc82d52107b43e1full, 0x3fef7c97337b9b5full, 0xbc892ab93b470dc9ull, 0x3fef864614f5a129ull, \
    0x3c74b604603a88d3ull, 0x3fef902ee78b3ff6ull, 0x3c83c5ec519d7271ull, 0x3fef9a51fbc74c83ull, \
    0xbc8ff7128fd391f0ull, 0x3fefa4afa2a490daull, 0xbc8dae98e223747dull, 0x3fefaf482d8e67f1ull, \
    0x3c8ec3bc41aa2008ull, 0x3fefba1bee615a27ull, 0x3c842b94c3a9eb32ull, 0x3fefc52b376bba97ull, \
    0x3c8a64a931d185eeull, 0x3fefd0765b6e4540ull, 0xbc8e37bae43be3edull, 0x3fefdbfdad9cbe14ull, \
    0x3c77893b4d91cd9dull, 0x3fefe7c1819e90d8ull, 0x3c5305c14160cc89ull, 0x3feff3c22b8f71f1ull, \
}
#define MPP_LIBM_LOG_TAB {  \
    0x3ff6a00000000000ull, 0xbfd62c82f2b9c800ull, 0x3cfab42428375680ull, 0ull, \
    0x3ff6800000000000ull, 0xbfd5d1bdbf580800ull, 0xbd1ca508d8e0f720ull, 0ull, \
    0x3ff6600000000000ull, 0xbfd5767717455800ull, 0xbd2362a4d5b6506dull, 0ull, \
    0x3ff6400000000000ull, 0xbfd51aad872df800ull, 0xbce684e49eb067d5ull, 0ull, \
    0x3ff6200000000000ull, 0xbfd4be5f95777800ull, 0xbd041b6993293ee0ull, 0ull, \
    0x3ff6000000000000ull, 0xbfd4618bc21c6000ull, 0x3d13d82f484c84ccull, 0ull, \
    0x3ff5e00000000000ull, 0xbfd404308686a800ull, 0x3cdc42f3ed820b3aull, 0ull, \
    0x3ff5c00000000000ull, 0xbfd3a64c55694800ull, 0x3d20b1c686519460ull, 0ull, \
    0x3ff5a00000000000ull, 0xbfd347dd9a988000ull, 0x3d25594dd4c58092ull, 0ull, \
    0x3ff5800000000000ull, 0xbfd2e8e2bae12000ull, 0x3d267b1e99b72bd8ull, 0ull, \
    0x3ff5600000000000ull, 0xbfd2895a13de8800ull, 0x3d15ca14b6cfb03full, 0ull, \
    0x3ff5600000000000ull, 0xbfd2895a13de8800ull, 0x3d15ca14b6cfb03full, 0ull, \
    0x3ff5400000000000ull, 0xbfd22941fbcf7800ull, 0xbd165a242853da76ull, 0ull, \
    0x3ff5200000000000ull, 0xbfd1c898c1699800ull, 0xbd1fafbc68e75404ull, 0ull, \
    0x3ff5000000000000ull, 0xbfd1675cababa800ull, 0x3d1f1fc63382a8f0ull, 0ull, \
    0x3ff4e00000000000ull, 0xbfd1058bf9ae4800ull, 0xbd26a8c4fd055a66ull, 0ull, \
    0x3ff4c00000000000ull, 0xbfd0a324e2739000ull, 0xbd0c6bee7ef4030eull, 0ull, \
    0x3ff4a00000000000ull, 0xbfd0402594b4d000ull, 0xbcf036b89ef42d7full, 0ull, \
    0x3ff4a00000000000ull, 0xbfd0402594b4d000ull, 0xbcf036b89ef42d7full, 0ull, \
    0x3ff4800000000000ull, 0xbfcfb9186d5e4000ull, 0x3d0d572aab993c87ull, 0ull, \
    0x3ff4600000000000ull, 0xbfcef0adcbdc6000ull, 0x3d2b26b79c86af24ull, 0ull, \
    0x3ff4400000000000ull, 0xbfce27076e2af000ull, 0xbd172f4f543fff10ull, 0ull, \
    0x3ff4200000000000ull, 0xbfcd5c216b4fc000ull, 0x3d21ba91bbca681bull, 0ull, \
    0x3ff4000000000000ull, 0xbfcc8ff7c79aa000ull, 0x3d27794f689f8434ull, 0ull, \
    0x3ff4000000000000ull, 0xbfcc8ff7c79aa000ull, 0x3d27794f689f8434ull, 0ull, \
    0x3ff3e00000000000ull, 0xbfcbc286742d9000ull, 0x3d194eb0318bb78full, 0ull, \
    0x3ff3c00000000000ull, 0xbfcaf3c94e80c000ull, 0x3cba4e633fcd9066ull, 0ull, \
    0x3ff3a00000000000ull, 0xbfca23bc1fe2b000ull, 0xbd258c64dc46c1eaull, 0ull, \
    0x3ff3a00000000000ull, 0xbfca23bc1fe2b000ull, 0xbd258c64dc46c1eaull, 0ull, \
    0x3ff3800000000000ull, 0xbfc9525a9cf45000ull, 0xbd2ad1d904c1d4e3ull, 0ull, \
    0x3ff3600000000000ull, 0xbfc87fa06520d000ull, 0x3d2bbdbf7fdbfa09ull, 0ull, \
    0x3ff3400000000000ull, 0xbfc7ab890210e000ull, 0x3d2bdb9072534a58ull, 0ull, \
    0x3ff3400000000000ull, 0xbfc7ab890210e000ull, 0x3d2bdb9072534a58ull, 0ull, \
    0x3ff3200000000000ull, 0xbfc6d60fe719d000ull, 0xbd10e46aa3b2e266ull, 0ull, \
    0x3ff3000000000000ull, 0xbfc5ff3070a79000ull, 0xbd1e9e439f105039ull, 0ull, \
    0x3ff3000000000000ull, 0xbfc5ff3070a79000ull, 0xbd1e9e439f105039ull, 0ull, \
    0x3ff2e00000000000ull, 0xbfc526e5e3a1b000ull, 0xbd20de8b90075b8full, 0ull, \
    0x3ff2c00000000000ull, 0xbfc44d2b6ccb8000ull, 0x3d170cc16135783cull, 0ull, \
    0x3ff2c00000000000ull, 0xbfc44d2b6ccb8000ull, 0x3d170cc16135783cull, 0ull, \
    0x3ff2a00000000000ull, 0xbfc371fc201e9000ull, 0x3cf178864d27543aull, 0ull, \
    0x3ff2800000000000ull, 0xbfc29552f81ff000ull, 0xbd248d301771c408ull, 0ull, \
    0x3ff2600000000000ull, 0xbfc1b72ad52f6000ull, 0xbd2e80a41811a396ull, 0ull, \
    0x3ff2600000000000ull, 0xbfc1b72ad52f6000ull, 0xbd2e80a41811a396ull, 0ull, \
    0x3ff2400000000000ull, 0xbfc0d77e7cd09000ull, 0x3d0a699688e85bf4ull, 0ull, \
    0x3ff2400000000000ull, 0xbfc0d77e7cd09000ull, 0x3d0a699688e85bf4ull, 0ull, \
    0x3ff2200000000000ull, 0xbfbfec9131dbe000ull, 0xbd2575545ca333f2ull, 0ull, \
    0x3ff2000000000000ull, 0xbfbe27076e2b0000ull, 0x3d2a342c2af0003cull, 0ull, \
    0x3ff2000000000000ull, 0xbfbe27076e2b0000ull, 0x3d2a342c2af0003cull, 0ull, \
    0x3ff1e00000000000ull, 0xbfbc5e548f5bc000ull, 0xbd1d0c57585fbe06ull, 0ull, \
    0x3ff1c00000000000ull, 0xbfba926d3a4ae000ull, 0x3d253935e85baac8ull, 0ull, \
    0x3ff1c00000000000ull, 0xbfba926d3a4ae000ull, 0x3d253935e85baac8ull, 0ull, \
    0x3ff1a00000000000ull, 0xbfb8c345d631a000ull, 0x3d137c294d2f5668ull, 0ull, \
    0x3ff1a00000000000ull, 0xbfb8c345d631a000ull, 0x3d137c294d2f5668ull, 0ull, \
    0x3ff1800000000000ull, 0xbfb6f0d28ae56000ull, 0xbd269737c93373daull, 0ull, \
    0x3ff1600000000000ull, 0xbfb51b073f062000ull, 0x3d1f025b61c65e57ull, 0ull, \
    0x3ff1600000000000ull, 0xbfb51b073f062000ull, 0x3d1f025b61c65e57ull, 0ull, \
    0x3ff1400000000000ull, 0xbfb341d7961be000ull, 0x3d2c5edaccf913dfull, 0ull, \
    0x3ff1400000000000ull, 0xbfb341d7961be000ull, 0x3d2c5edaccf913dfull, 0ull, \
    0x3ff1200000000000ull, 0xbfb16536eea38000ull, 0x3d147c5e768fa309ull, 0ull, \
    0x3ff1000000000000ull, 0xbfaf0a30c0118000ull, 0x3d2d599e83368e91ull, 0ull, \
    0x3ff1000000000000ull, 0xbfaf0a30c0118000ull, 0x3d2d599e83368e91ull, 0ull, \
    0x3ff0e00000000000ull, 0xbfab42dd71198000ull, 0x3d1c827ae5d6704cull, 0ull, \
    0x3ff0e00000000000ull, 0xbfab42dd71198000ull, 0x3d1c827ae5d6704cull, 0ull, \
    0x3ff0c00000000000ull, 0xbfa77458f632c000ull, 0xbd2cfc4634f2a1eeull, 0ull, \
    0x3ff0c00000000000ull, 0xbfa77458f632c000ull, 0xbd2cfc4634f2a1eeull, 0ull, \
    0x3ff0a00000000000ull, 0xbfa39e87b9fec000ull, 0x3cf502b7f526feaaull, 0ull, \
    0x3ff0a00000000000ull, 0xbfa39e87b9fec000ull, 0x3cf502b7f526feaaull, 0ull, \
    0x3ff0800000000000ull, 0xbf9f829b0e780000ull, 0xbd2980267c7e09e4ull, 0ull, \
    0x3ff0800000000000ull, 0xbf9f829b0e780000ull, 0xbd2980267c7e09e4ull, 0ull, \
    0x3ff0600000000000ull, 0xbf97b91b07d58000ull, 0xbd288d5493faa639ull, 0ull, \
    0x3ff0400000000000ull, 0xbf8fc0a8b0fc0000ull, 0xbcdf1e7cf6d3a69cull, 0ull, \
    0x3ff0400000000000ull, 0xbf8fc0a8b0fc0000ull, 0xbcdf1e7cf6d3a69cull, 0ull, \
    0x3ff0200000000000ull, 0xbf7fe02a6b100000ull, 0xbd19e23f0dda40e4ull, 0ull, \
    0x3ff0200000000000ull, 0xbf7fe02a6b100000ull, 0xbd19e23f0dda40e4ull, 0ull, \
    0x3ff0000000000000ull, 0x0000000000000000ull, 0x0000000000000000ull, 0ull, \
    0x3ff0000000000000ull, 0x0000000000000000ull, 0x0000000000000000ull, 0ull, \
    0x3fefc00000000000ull, 0x3f80101575890000ull, 0xbd10c76b999d2be8ull, 0ull, \
    0x3fef800000000000ull, 0x3f90205658938000ull, 0xbd23dc5b06e2f7d2ull, 0ull, \
    0x3fef400000000000ull, 0x3f98492528c90000ull, 0xbd2aa0ba325a0c34ull, 0ull, \
    0x3fef000000000000ull, 0x3fa0415d89e74000ull, 0x3d0111c05cf1d753ull, 0ull, \
    0x3feec00000000000ull, 0x3fa466aed42e0000ull, 0xbd2c167375bdfd28ull, 0ull, \
    0x3fee800000000000ull, 0x3fa894aa149fc000ull, 0xbd197995d05a267dull, 0ull, \
    0x3fee400000000000ull, 0x3faccb73cdddc000ull, 0xbd1a68f247d82807ull, 0ull, \
    0x3fee200000000000ull, 0x3faeea31c006c000ull, 0xbd0e113e4fc93b7bull, 0ull, \
    0x3fede00000000000ull, 0x3fb1973bd1466000ull, 0xbd25325d560d9e9bull, 0ull, \
    0x3feda00000000000ull, 0x3fb3bdf5a7d1e000ull, 0x3d2cc85ea5db4ed7ull, 0ull, \
    0x3fed600000000000ull, 0x3fb5e95a4d97a000ull, 0xbd2c69063c5d1d1eull, 0ull, \
    0x3fed400000000000ull, 0x3fb700d30aeac000ull, 0x3cec1e8da99ded32ull, 0ull, \
    0x3fed000000000000ull, 0x3fb9335e5d594000ull, 0x3d23115c3abd47daull, 0ull, \
    0x3fecc00000000000ull, 0x3fbb6ac88dad6000ull, 0xbd1390802bf768e5ull, 0ull, \
    0x3feca00000000000ull, 0x3fbc885801bc4000ull, 0x3d2646d1c65aacd3ull, 0ull, \
    0x3fec600000000000ull, 0x3fbec739830a2000ull, 0xbd2dc068afe645e0ull, 0ull, \
    0x3fec400000000000ull, 0x3fbfe89139dbe000ull, 0xbd2534d64fa10afdull, 0ull, \
    0x3fec000000000000ull, 0x3fc1178e8227e000ull, 0x3d21ef78ce2d07f2ull, 0ull, \
    0x3febe00000000000ull, 0x3fc1aa2b7e23f000ull, 0x3d2ca78e44389934ull, 0ull, \
    0x3feba00000000000ull, 0x3fc2d1610c868000ull, 0x3d039d6ccb81b4a1ull, 0ull, \
    0x3feb800000000000ull, 0x3fc365fcb0159000ull, 0x3cc62fa8234b7289ull, 0ull, \
    0x3feb400000000000ull, 0x3fc4913d8333b000ull, 0x3d25837954fdb678ull, 0ull, \
    0x3feb200000000000ull, 0x3fc527e5e4a1b000ull, 0x3d2633e8e5697dc7ull, 0ull, \
    0x3feae00000000000ull, 0x3fc6574ebe8c1000ull, 0x3d19cf8b2c3c2e78ull, 0ull, \
    0x3feac00000000000ull, 0x3fc6f0128b757000ull, 0xbd25118de59c21e1ull, 0ull, \
    0x3feaa00000000000ull, 0x3fc7898d85445000ull, 0xbd1c661070914305ull, 0ull, \
    0x3fea600000000000ull, 0x3fc8beafeb390000ull, 0xbd073d54aae92cd1ull, 0ull, \
    0x3fea400000000000ull, 0x3fc95a5adcf70000ull, 0x3d07f22858a0ff6full, 0ull, \
    0x3fea000000000000ull, 0x3fca93ed3c8ae000ull, 0xbd28724350562169ull, 0ull, \
    0x3fe9e00000000000ull, 0x3fcb31d8575bd000ull, 0xbd0c358d4eace1aaull, 0ull, \
    0x3fe9c00000000000ull, 0x3fcbd087383be000ull, 0xbd2d4bc4595412b6ull, 0ull, \
    0x3fe9a00000000000ull, 0x3fcc6ffbc6f01000ull, 0xbcf1ec72c5962bd2ull, 0ull, \
    0x3fe9600000000000ull, 0x3fcdb13db0d49000ull, 0xbd2aff2af715b035ull, 0ull, \
    0x3fe9400000000000ull, 0x3fce530effe71000ull, 0x3cc212276041f430ull, 0ull, \
    0x3fe9200000000000ull, 0x3fcef5ade4dd0000ull, 0xbcca211565bb8e11ull, 0ull, \
    0x3fe9000000000000ull, 0x3fcf991c6cb3b000ull, 0x3d1bcbecca0cdf30ull, 0ull, \
    0x3fe8c00000000000ull, 0x3fd07138604d5800ull, 0x3cf89cdb16ed4e91ull, 0ull, \
    0x3fe8a00000000000ull, 0x3fd0c42d67616000ull, 0x3d27188b163ceae9ull, 0ull, \
    0x3fe8800000000000ull, 0x3fd1178e8227e800ull, 0xbd2c210e63a5f01cull, 0ull, \
    0x3fe8600000000000ull, 0x3fd16b5ccbacf800ull, 0x3d2b9acdf7a51681ull, 0ull, \
    0x3fe8400000000000ull, 0x3fd1bf99635a6800ull, 0x3d2ca6ed5147bdb7ull, 0ull, \
    0x3fe8200000000000ull, 0x3fd214456d0eb800ull, 0x3d0a87deba46baeaull, 0ull, \
    0x3fe7e00000000000ull, 0x3fd2bef07cdc9000ull, 0x3d2a9cfa4a5004f4ull, 0ull, \
    0x3fe7c00000000000ull, 0x3fd314f1e1d36000ull, 0xbd28e27ad3213cb8ull, 0ull, \
    0x3fe7a00000000000ull, 0x3fd36b6776be1000ull, 0x3d116ecdb0f177c8ull, 0ull, \
    0x3fe7800000000000ull, 0x3fd3c25277333000ull, 0x3d183b54b606bd5cull, 0ull, \
    0x3fe7600000000000ull, 0x3fd419b423d5e800ull, 0x3d08e436ec90e09dull, 0ull, \
    0x3fe7400000000000ull, 0x3fd4718dc271c800ull, 0xbd2f27ce0967d675ull, 0ull, \
    0x3fe7200000000000ull, 0x3fd4c9e09e173000ull, 0xbd2e20891b0ad8a4ull, 0ull, \
    0x3fe7000000000000ull, 0x3fd522ae0738a000ull, 0x3d2ebe708164c759ull, 0ull, \
    0x3fe6e00000000000ull, 0x3fd57bf753c8d000ull, 0x3d1fadedee5d40efull, 0ull, \
    0x3fe6c00000000000ull, 0x3fd5d5bddf596000ull, 0xbd0a0b2a08a465dcull, 0ull, \
}

// 2^(k/128) as (tail, scale bits) pairs, k = 0..127 (__exp_data.tab)
static const unsigned long long mpp_libm_exp_tab_h[256] = MPP_LIBM_EXP_TAB;
// {1/c, log c, log c tail, 0} for the 128 subintervals of [OFF, 2 OFF) (__pow_log_data.tab)
static const unsigned long long mpp_libm_log_tab_h[512] = MPP_LIBM_LOG_TAB;
#ifdef __CUDACC__
static __device__ const unsigned long long __align__(16) mpp_libm_exp_tab_d[256] = MPP_LIBM_EXP_TAB;
static __device__ const unsigned long long __align__(32) mpp_libm_log_tab_d[512] = MPP_LIBM_LOG_TAB;
#endif

MPP_LIBM_FN uint64_t mpp_libm_bits(double x) {
#ifdef __CUDA_ARCH__
    return (uint64_t)__double_as_longlong(x);
#else
    uint64_t u;
    memcpy(&u, &x, 8);
    return u;
#endif
}
MPP_LIBM_FN double mpp_libm_double(uint64_t u) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)u);
#else
    double x;
    memcpy(&x, &u, 8);
    return x;
#endif
}
// entry i of the exp table / word j of log table entry i
MPP_LIBM_FN uint64_t mpp_libm_exp_tab(unsigned i) {
#ifdef __CUDA_ARCH__
    return __ldg(mpp_libm_exp_tab_d + i);
#else
    return mpp_libm_exp_tab_h[i];
#endif
}
MPP_LIBM_FN double mpp_libm_log_tab(unsigned i, unsigned j) {
#ifdef __CUDA_ARCH__
    return mpp_libm_double(__ldg(mpp_libm_log_tab_d + 4 * i + j));
#else
    return mpp_libm_double(mpp_libm_log_tab_h[4 * i + j]);
#endif
}
// what x86 returns for an arithmetic operation whose NaN operand is v: v with its quiet bit set
MPP_LIBM_FN double mpp_libm_quiet(double v) { return mpp_libm_double(mpp_libm_bits(v) | 0x0008000000000000ull); }

// exp(x + xtail) for the finite x whose top 12 bits are in [0x3c9, 0x409) or whose result over- or underflows
// (`special`); the shared tail of exp (xtail = 0, has_tail false) and pow (e_exp.c / e_pow.c exp_inline).
MPP_LIBM_FN double mpp_libm_exp_core(double x, double xtail, bool has_tail, bool special) {
    const double kd0 = fma(x, 0x1.71547652b82fep+7, 0x1.8p52);        // InvLn2N * x + Shift
    const uint64_t ki = mpp_libm_bits(kd0);
    const double kd = kd0 - 0x1.8p52;
    double r = fma(kd, -0x1.cf79abc9e3b3ap-47, fma(kd, -0x1.62e42fefa0000p-8, x));   // x - kd ln2/128, hi then lo
    if (has_tail) r = xtail + r;
    const unsigned idx = 2 * (unsigned)(ki % 128);
    const double tail = mpp_libm_double(mpp_libm_exp_tab(idx));
    uint64_t sbits = mpp_libm_exp_tab(idx + 1) + (ki << 45);
    const double r2 = r * r;
    const double tmp = fma(r2 * r2, fma(r, 0x1.1111167a4d017p-7, 0x1.55555cf172b91p-5),
                           fma(fma(r, 0x1.555555555543cp-3, 0x1.ffffffffffdbdp-2), r2, r + tail));
    if (!special) {
        const double scale = mpp_libm_double(sbits);
        return fma(scale, tmp, scale);
    }
    // specialcase: the exponent of scale may have over- or underflowed
    if ((ki & 0x80000000u) == 0) {
        sbits -= 1009ull << 52;
        const double scale = mpp_libm_double(sbits);
        return 0x1p1009 * fma(scale, tmp, scale);
    }
    sbits += 1022ull << 52;
    const double scale = mpp_libm_double(sbits);
    const double st = scale * tmp;
    double y = scale + st;
    if (y < 1.0) {
        // round to the subnormal precision once, before the scaling (no double rounding)
        double lo = scale - y + st;
        const double hi = 1.0 + y;
        lo = 1.0 - hi + y + lo;
        y = (hi + lo) - 1.0;
        if (y == 0.0) y = 0.0;
    }
    return 0x1p-1022 * y;
}

// exp(x), bit for bit glibc 2.39 x86-64 __exp_fma, for every double x
MPP_LIBM_FN double mpp_exp(double x) {
    const uint64_t ix = mpp_libm_bits(x);
    const uint32_t abstop = (uint32_t)(ix >> 52) & 0x7ff;
    if (abstop - 0x3c9u >= 0x408u - 0x3c9u) {                         // |x| < 2^-54 or |x| >= 512
        if (abstop < 0x3c9u) return 1.0 + x;
        if (abstop >= 0x409u) {                                        // |x| >= 1024, inf, nan
            if (ix == 0xfff0000000000000ull) return 0.0;
            if (abstop == 0x7ff) return x != x ? mpp_libm_quiet(x) : x;
            return ix >> 63 ? 0.0 : mpp_libm_double(0x7ff0000000000000ull);
        }
        return mpp_libm_exp_core(x, 0.0, false, true);                 // 512 <= |x| < 1024
    }
    return mpp_libm_exp_core(x, 0.0, false, false);
}

// pow(x, y), bit for bit glibc 2.39 x86-64 __pow_fma, for x in [+0, +inf] and every y
MPP_LIBM_FN double mpp_pow(double x, double y) {
    const uint64_t ONE = 0x3ff0000000000000ull, INF = 0x7ff0000000000000ull;
    uint64_t ix = mpp_libm_bits(x);
    const uint64_t iy = mpp_libm_bits(y);
    const uint32_t topx = (uint32_t)(ix >> 52), topy = (uint32_t)(iy >> 52);
    if (topx - 1u >= 0x7feu || (topy & 0x7ff) - 0x3beu >= 0x80u) {
        if (2 * iy - 1 >= 2 * INF - 1) {                               // y is +-0, +-inf or nan
            if (2 * iy == 0) return 1.0;
            if (ix == ONE) return 2 * (iy ^ 0x0008000000000000ull) > 2 * 0x7ff8000000000000ull ? mpp_libm_quiet(y) : 1.0;
            if (2 * iy > 2 * INF) return mpp_libm_quiet(y);
            if ((2 * ix < 2 * ONE) == !(iy >> 63)) return 0.0;         // |x| < 1, y = inf or |x| > 1, y = -inf
            return y * y;
        }
        if (2 * ix - 1 >= 2 * INF - 1) {                               // x is +0 or +inf
            const double x2 = x * x;
            return iy >> 63 ? 1.0 / x2 : x2;
        }
        if ((topy & 0x7ff) - 0x3beu >= 0x80u) {                        // |y| < 2^-65 or |y| >= 2^63
            if (ix == ONE) return 1.0;
            if ((topy & 0x7ff) < 0x3beu) return ix > ONE ? 1.0 + y : 1.0 - y;
            return (ix > ONE) == (topy < 0x800) ? mpp_libm_double(INF) : 0.0;
        }
        if (topx == 0) {                                               // subnormal x: normalise
            ix = mpp_libm_bits(x * 0x1p52) & 0x7fffffffffffffffull;
            ix -= 52ull << 52;
        }
    }
    // log_inline: log(x) = k ln2 + log(c) + log1p(z/c - 1) as hi + tail
    const uint64_t tmp = ix - 0x3fe6955500000000ull;
    const unsigned i = (unsigned)((tmp >> 45) % 128);
    const int k = (int)((int64_t)tmp >> 52);
    const double z = mpp_libm_double(ix - (tmp & 0xfffull << 52)), kd = (double)k;
    const double invc = mpp_libm_log_tab(i, 0), logc = mpp_libm_log_tab(i, 1), logctail = mpp_libm_log_tab(i, 2);
    const double r = fma(z, invc, -1.0);
    const double t1 = fma(kd, 0x1.62e42fefa3800p-1, logc);
    const double t2 = t1 + r;
    const double lo1 = fma(kd, 0x1.ef35793c76730p-45, logctail);
    const double lo2 = t1 - t2 + r;
    const double ar = -0x1p-1 * r;
    const double ar2 = r * ar;
    const double ar3 = r * ar2;
    const double hi = t2 + ar2;
    const double lo3 = fma(ar, r, -ar2);
    const double lo4 = t2 - hi + ar2;
    const double q = fma(ar2, fma(fma(r, 0x1.0002b8b263fc3p+0, -0x1.2495b9b4845e9p+0), ar2,
                                  fma(r, -0x1.555555529a47ap-1, 0x1.999999959554ep-1)),
                         fma(r, 0x1.0000000000006p-1, -0x1.5555555555560p-1));
    const double lo = fma(ar3, q, lo1 + lo2 + lo3 + lo4);
    const double lhi = hi + lo;
    const double ltail = hi - lhi + lo;
    // y log(x) as ehi + elo, then exp_inline
    const double ehi = y * lhi;
    const double elo = fma(y, ltail, fma(y, lhi, -ehi));
    const uint32_t abstop = (uint32_t)(mpp_libm_bits(ehi) >> 52) & 0x7ff;
    if (abstop - 0x3c9u >= 0x408u - 0x3c9u) {                         // |y log x| < 2^-54 or >= 512
        if (abstop < 0x3c9u) return 1.0 + ehi;
        if (abstop >= 0x409u) return mpp_libm_bits(ehi) >> 63 ? 0.0 : mpp_libm_double(INF);
        return mpp_libm_exp_core(ehi, elo, true, true);
    }
    return mpp_libm_exp_core(ehi, elo, true, false);
}
