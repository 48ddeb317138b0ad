// main.cpp -- `kpeg` CLI drop-in (reference main.cpp:8-140).
//
//   kpeg -h              help text
//   kpeg <file.jpg>      decode on the GPU, write <file>.ppm next to the input, log to kpeg.log + stdout
//   kpeg <in.ppm> <out.jpg>   encode on the GPU (kpeg_cuda_encode): binary PPM (P6, maxval 255) as R,G,B or PGM (P5)
//                        as one gray component -> baseline JPEG, Annex K (or, --optimize, per-image) tables, 4:4:4.  The reference's own
//                        encoder is non-functional (reference README.md:23); this one writes byte for byte what
//                        the synthetic reference encoder (host/synth_encoder.cpp) writes for the same pixels.
// Exit status follows the reference: EXIT_SUCCESS for any 2- or 3-argument run, EXIT_FAILURE for
// none or too many (main.cpp:54-79).  Extra, non-reference switches come before the file name:
//   --t81        ITU-T T.81 behaviour instead of bit-exact reference parity (SURVEY F1); when encoding: no DC nudge
//   --device N   CUDA device index
//   --quality N  encoder: IJG quality 1..100 (default 90)
//   --restart N  encoder: restart interval in MCUs (default 0: none)
//   --optimize   encoder: Huffman tables optimised for the image (KPEG_FLAG_OPTIMIZE_HUFFMAN): smaller files
//   kpeg <in.jpg> <out.jpg>   (the first file starts with FF D8) lossless transcode on the GPU (kpeg_cuda_transcode):
//                        the same quantised coefficients, re-coded; --restart N (default: the input's interval),
//                        --optimize, --transform none|flip-h|flip-v|transpose|transverse|rot90|rot180|rot270
//   --devices L  several devices, e.g. 0-7 or 0,2,3: the restart-interval tiles of the image are spread over them
//   --scale 1/N  decode: N = 2, 4 or 8 writes <file>.ppm at 1/N the size (KPEG_FLAG_SCALE_*: libjpeg's reduced IDCTs and
//                integer colour, as djpeg -scale 1/N); 1/1 or no --scale is the full-size decode of the drop-in JPEGDecoder
//   --crop WxH+X+Y  decode: <file>.ppm holds only that rectangle of the output image (after --scale), exactly (djpeg -crop
//                widens it to iMCU boundaries; this does not); kpeg_cuda_decode_file_crop
//   --quiet      log only to kpeg.log
#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <iterator>
#include <string>
#include <vector>

#include "Decoder.hpp"
#include "Logger.hpp"
#include "kpeg_cuda.h"

namespace
{
    void printHelp()
    {
        std::cout << "===========================================" << std::endl;
        std::cout << "   K-PEG - Simple JPEG Encoder & Decoder"    << std::endl;
        std::cout << "===========================================" << std::endl;
        std::cout << "Help\n" << std::endl;
        std::cout << "<filename.jpg>                  : Decompress a JPEG image to a PPM image" << std::endl;
        std::cout << "<filename.ppm> <filename.jpg>   : Encode a PPM (P6) or PGM (P5) image to JPEG on the GPU" << std::endl;
        std::cout << "--quality N                     : Encoder quality 1..100 (default 90)" << std::endl;
        std::cout << "--restart N                     : Encoder restart interval in MCUs (default 0: none)" << std::endl;
        std::cout << "--optimize                      : Encoder Huffman tables optimised for the image (smaller file)" << std::endl;
        std::cout << "<in.jpg> <out.jpg>              : Transcode a baseline JPEG losslessly on the GPU" << std::endl;
        std::cout << "--transform T                   : Transcode: none, flip-h, flip-v, transpose, transverse, rot90, rot180, rot270" << std::endl;
        std::cout << "--scale 1/N                     : Decode at 1/2, 1/4 or 1/8 the size (libjpeg's reduced IDCTs)" << std::endl;
        std::cout << "--crop WxH+X+Y                  : Decode only that rectangle of the (scaled) image" << std::endl;
        std::cout << "-h                              : Print this help message and exit" << std::endl;
    }

    // Utility.hpp:16-38: only names whose first ".jpg" is the suffix are accepted (".jpeg" is not).
    bool isValidFilename( const std::string& filename )
    {
        const std::size_t extPos = filename.find( ".jpg" );
        return extPos != std::string::npos && extPos + 4 == filename.size();
    }

    struct Options
    {
        bool parity = true;
        int device = 0;
        std::vector<int> devices;
        int quality = 90;
        int restart = 0;
        bool restart_given = false;
        bool optimize = false;
        std::string transform = "none";
        std::string scale = "1/1";
        bool crop_given = false;
        kpeg_crop crop = {};
    };

    // "WxH+X+Y" (djpeg's -crop syntax; every part required, decimal) -> crop; false when malformed
    bool parseCrop( const std::string& s, kpeg_crop& c )
    {
        unsigned long v[4];
        const char seps[4] = { 'x', '+', '+', '\0' };
        std::size_t i = 0;
        for ( int k = 0; k < 4; ++k )
        {
            const std::size_t j = i;
            while ( i < s.size() && std::isdigit( (unsigned char)s[i] ) ) ++i;
            if ( i == j || i - j > 10 ) return false;
            v[k] = std::stoul( s.substr( j, i - j ) );
            if ( v[k] > 0xFFFFFFFFul ) return false;
            if ( k < 3 ) { if ( i >= s.size() || s[i] != seps[k] ) return false; ++i; }
        }
        if ( i != s.size() || v[0] == 0 || v[1] == 0 ) return false;
        c.width = (uint32_t)v[0]; c.height = (uint32_t)v[1]; c.x = (uint32_t)v[2]; c.y = (uint32_t)v[3];
        return true;
    }

    // "0-3", "0,2,5", "1": device list of --devices
    std::vector<int> parseDevices( const std::string& s )
    {
        std::vector<int> out;
        std::size_t i = 0;
        while ( i < s.size() )
        {
            std::size_t j = s.find( ',', i );
            if ( j == std::string::npos ) j = s.size();
            const std::string part = s.substr( i, j - i );
            const std::size_t dash = part.find( '-' );
            if ( dash == std::string::npos )
                out.push_back( std::atoi( part.c_str() ) );
            else
                for ( int d = std::atoi( part.substr( 0, dash ).c_str() ); d <= std::atoi( part.substr( dash + 1 ).c_str() ); ++d )
                    out.push_back( d );
            i = j + 1;
        }
        return out;
    }

    // Binary PPM (P6) or PGM (P5), maxval 255; '#' comments and any whitespace between the header fields.
    bool readPNM( const std::string& filename, int& width, int& height, int& ncomp, std::vector<uint8_t>& pixels, std::string& why )
    {
        std::ifstream in( filename, std::ios::binary );
        if ( !in ) { why = "cannot open " + filename; return false; }
        const std::vector<uint8_t> f( ( std::istreambuf_iterator<char>( in ) ), std::istreambuf_iterator<char>() );
        std::size_t pos = 0;
        auto skip = [&]() {
            while ( pos < f.size() )
            {
                if ( f[pos] == '#' ) { while ( pos < f.size() && f[pos] != '\n' ) ++pos; }
                else if ( std::isspace( f[pos] ) ) ++pos;
                else break;
            }
        };
        auto number = [&]( long& v ) {
            skip();
            if ( pos >= f.size() || !std::isdigit( f[pos] ) ) return false;
            v = 0;
            while ( pos < f.size() && std::isdigit( f[pos] ) && v < 1000000 ) v = v * 10 + ( f[pos++] - '0' );
            return v < 1000000;
        };
        if ( f.size() < 2 || f[0] != 'P' || ( f[1] != '6' && f[1] != '5' ) ) { why = "not a binary PPM (P6) or PGM (P5) file"; return false; }
        ncomp = f[1] == '6' ? 3 : 1;
        pos = 2;
        long w = 0, h = 0, maxval = 0;
        if ( !number( w ) || !number( h ) || !number( maxval ) ) { why = "malformed header"; return false; }
        if ( w < 1 || h < 1 || w > 65535 || h > 65535 ) { why = "image size out of range (1..65535)"; return false; }
        if ( maxval != 255 ) { why = "only maxval 255 is supported"; return false; }
        if ( pos >= f.size() || !std::isspace( f[pos] ) ) { why = "malformed header"; return false; }
        ++pos; // exactly one whitespace byte before the samples
        const std::size_t n = (std::size_t)w * h * ncomp;
        if ( f.size() - pos < n ) { why = "truncated pixel data"; return false; }
        pixels.assign( f.begin() + pos, f.begin() + pos + n );
        width = (int)w;
        height = (int)h;
        return true;
    }

    void encodeJPEG( const std::string& in, const std::string& out, const Options& opt )
    {
        if ( !isValidFilename( out ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "Invalid output file name passed.";
            return;
        }
        int width = 0, height = 0, ncomp = 0;
        std::vector<uint8_t> pixels;
        std::string why;
        if ( !readPNM( in, width, height, ncomp, pixels, why ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while encoding: " << in << ": " << why;
            return;
        }
        if ( opt.quality < 1 || opt.quality > 100 || opt.restart < 0 || opt.restart > 65535 )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while encoding: --quality must be 1..100, --restart 0..65535";
            return;
        }
        kpeg_encode_params p = {};
        p.width = (uint16_t)width;
        p.height = (uint16_t)height;
        p.ncomp = (uint8_t)ncomp;
        p.quality = (uint8_t)opt.quality;
        p.restart_interval = (uint16_t)opt.restart;
        p.flags = ( opt.parity ? KPEG_FLAG_REF_PARITY : 0u ) | ( opt.optimize ? KPEG_FLAG_OPTIMIZE_HUFFMAN : 0u );
        kpeg_ctx* ctx = nullptr;
        if ( kpeg_cuda_acquire( opt.device, &ctx ) != KPEG_OK )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while encoding: no usable CUDA device (there is no CPU encode path)";
            return;
        }
        std::vector<uint8_t> jpeg( kpeg_encode_bound( &p ) );
        std::size_t len = 0;
        const int rc = kpeg_cuda_encode( ctx, &p, pixels.data(), jpeg.data(), jpeg.size(), &len, nullptr );
        const std::string err = rc == KPEG_OK ? "" : kpeg_cuda_last_error( ctx );
        kpeg_cuda_release( opt.device, ctx );
        if ( rc != KPEG_OK )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while encoding: " << err;
            return;
        }
        std::ofstream o( out, std::ios::binary );
        o.write( (const char*)jpeg.data(), (std::streamsize)len );
        o.close();
        if ( !o )
        {
            std::remove( out.c_str() );
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while encoding: cannot write " << out;
            return;
        }
        LOG(kpeg::Logger::Level::INFO) << "Encoded " << in << " (" << width << "x" << height << ", " << ncomp
                                       << ( ncomp == 3 ? " components" : " component" ) << ") to " << out << ": " << len << " bytes";
    }

    bool readFile( const std::string& filename, std::vector<uint8_t>& data )
    {
        std::ifstream in( filename, std::ios::binary );
        if ( !in ) return false;
        data.assign( std::istreambuf_iterator<char>( in ), std::istreambuf_iterator<char>() );
        return true;
    }

    bool startsWithSOI( const std::string& filename )
    {
        std::ifstream in( filename, std::ios::binary );
        unsigned char b[2] = { 0, 0 };
        return in.read( (char*)b, 2 ) && b[0] == 0xFF && b[1] == 0xD8;
    }

    void transcodeJPEG( const std::string& in, const std::string& out, const Options& opt )
    {
        static const char* const names[] = { "none", "flip-h", "flip-v", "transpose", "transverse", "rot90", "rot180", "rot270" };
        int xform = -1;
        for ( int t = 0; t < 8; ++t )
            if ( opt.transform == names[t] ) xform = t;
        if ( !isValidFilename( out ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "Invalid output file name passed.";
            return;
        }
        if ( xform < 0 || ( opt.restart_given && ( opt.restart < 0 || opt.restart > 65535 ) ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while transcoding: --transform must be one of none, flip-h, flip-v, "
                                               "transpose, transverse, rot90, rot180, rot270 and --restart 0..65535";
            return;
        }
        std::vector<uint8_t> data;
        if ( !readFile( in, data ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while transcoding: cannot open " << in;
            return;
        }
        kpeg_transcode_params p = {};
        p.restart_interval = opt.restart_given ? opt.restart : KPEG_TRANSCODE_KEEP_RESTART;
        p.transform = (uint32_t)xform;
        p.flags = opt.optimize ? KPEG_FLAG_OPTIMIZE_HUFFMAN : 0u;
        kpeg_ctx* ctx = nullptr;
        if ( kpeg_cuda_acquire( opt.device, &ctx ) != KPEG_OK )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while transcoding: no usable CUDA device (there is no CPU transcode path)";
            return;
        }
        std::vector<uint8_t> jpeg( std::max<std::size_t>( kpeg_transcode_bound( data.data(), data.size(), &p ), 1 ) );
        std::size_t len = 0;
        const int rc = kpeg_cuda_transcode( ctx, data.data(), data.size(), &p, jpeg.data(), jpeg.size(), &len, nullptr );
        const std::string err = rc == KPEG_OK ? "" : kpeg_cuda_last_error( ctx );
        kpeg_cuda_release( opt.device, ctx );
        if ( rc != KPEG_OK )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while transcoding: " << in << ": " << err;
            return;
        }
        std::ofstream o( out, std::ios::binary );
        o.write( (const char*)jpeg.data(), (std::streamsize)len );
        o.close();
        if ( !o )
        {
            std::remove( out.c_str() );
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while transcoding: cannot write " << out;
            return;
        }
        LOG(kpeg::Logger::Level::INFO) << "Transcoded " << in << " (" << data.size() << " bytes) to " << out << " (" << opt.transform
                                       << "): " << len << " bytes";
    }

    // --scale 2, 4, 8 and --crop: the reduced-size or cropped decode through the C ABI (the drop-in JPEGDecoder has the
    // reference's interface, which has neither), written as dumpRawData writes the full-size image: <name up to ".jpg">.ppm,
    // P6, gray as R = G = B
    void decodeScaled( const std::string& filename, const Options& opt, uint32_t scaleFlag )
    {
        std::vector<uint8_t> data;
        if ( !readFile( filename, data ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "Unable to open file: " << filename;
            return;
        }
        kpeg_plan frame;
        kpeg_scan scans[KPEG_MAX_SCANS];
        int nscans = 0;
        if ( kpeg_parse_jfif_scans( data.data(), data.size(), &frame, scans, KPEG_MAX_SCANS, &nscans ) != KPEG_OK )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while decoding: " << filename << ": not a supported baseline JPEG";
            return;
        }
        const uint32_t flags = ( opt.parity ? KPEG_FLAG_REF_PARITY : 0u ) | scaleFlag;
        frame.flags = flags;
        uint32_t w = 0, h = 0;
        size_t bytes = kpeg_output_size( &frame, &w, &h );
        if ( opt.crop_given )
        {
            if ( !opt.devices.empty() )
            {
                LOG(kpeg::Logger::Level::ERROR) << "--crop decodes on one device (no --devices).";
                return;
            }
            w = opt.crop.width;
            h = opt.crop.height;
            bytes = (size_t)w * h * frame.ncomp;
        }
        std::vector<uint8_t> pixels( bytes );
        int rc;
        std::string err;
        if ( !opt.devices.empty() )
        {
            rc = kpeg_cuda_decode_file_tiled( opt.devices.data(), (int)opt.devices.size(), data.data(), data.size(), flags, pixels.data(),
                                              pixels.size(), nullptr, nullptr );
            err = kpeg_tiled_last_error();
        }
        else
        {
            kpeg_ctx* ctx = nullptr;
            rc = kpeg_cuda_acquire( opt.device, &ctx );
            if ( rc == KPEG_OK )
            {
                rc = opt.crop_given ? kpeg_cuda_decode_file_crop( ctx, data.data(), data.size(), flags, &opt.crop, pixels.data(), pixels.size(),
                                                                  nullptr, nullptr )
                                    : kpeg_cuda_decode_file( ctx, data.data(), data.size(), flags, pixels.data(), pixels.size(), nullptr, nullptr );
                err = kpeg_cuda_last_error( ctx );
                kpeg_cuda_release( opt.device, ctx );
            }
            else
                err = "no usable CUDA device (there is no CPU decode path)";
        }
        if ( rc != KPEG_OK )
        {
            LOG(kpeg::Logger::Level::ERROR) << "An error ocurred while decoding: " << filename << ": " << err;
            return;
        }
        const std::string target = filename.substr( 0, filename.find( ".jpg" ) ) + ".ppm";
        std::ofstream out( target, std::ios::out | std::ios::binary );
        char header[160];
        const int hl = kpeg_ppm_header( (int)w, (int)h, header, sizeof header );
        out.write( header, hl );
        if ( frame.ncomp == 3 )
            out.write( (const char*)pixels.data(), (std::streamsize)pixels.size() );
        else
            for ( uint8_t v : pixels )
            {
                const char rgb[3] = { (char)v, (char)v, (char)v };
                out.write( rgb, 3 );
            }
        out.close();
        if ( !out )
        {
            std::remove( target.c_str() );
            LOG(kpeg::Logger::Level::ERROR) << "Unable to create dump file \'" << target << "\'.";
            return;
        }
        LOG(kpeg::Logger::Level::INFO) << "Decoded " << filename << " at " << opt.scale << ( opt.crop_given ? ", cropped" : "" ) << " (" << w << "x" << h
                                       << "): raw image data dumped to file: \'" << target << "\'.";
    }

    void decodeJPEG( const std::string& filename, const Options& opt )
    {
        if ( !isValidFilename( filename ) )
        {
            LOG(kpeg::Logger::Level::ERROR) << "Invalid input file name passed.";
            return;
        }
        static const char* const scales[] = { "1/1", "1/2", "1/4", "1/8" };
        int code = -1;
        for ( int k = 0; k < 4; ++k )
            if ( opt.scale == scales[k] ) code = k;
        if ( code < 0 )
        {
            LOG(kpeg::Logger::Level::ERROR) << "Unknown scale '" << opt.scale << "' (1/1, 1/2, 1/4 or 1/8).";
            return;
        }
        if ( code > 0 || opt.crop_given )
        {
            decodeScaled( filename, opt, (uint32_t)code * KPEG_FLAG_SCALE_1_2 );
            return;
        }
        kpeg::JPEGDecoder decoder;
        decoder.setParity( opt.parity );
        decoder.setDevice( opt.device );
        if ( !opt.devices.empty() )
            decoder.setDevices( opt.devices );
        decoder.open( filename );
        if ( decoder.decodeImageFile() == kpeg::JPEGDecoder::ResultCode::DECODE_DONE )
            decoder.dumpRawData();
    }
}

int main( int argc, char** argv )
{
    try
    {
        kpeg::Logger::get().openLogFile( "kpeg.log" );
        kpeg::Logger::get().setLevel( kpeg::Logger::Level::DEBUG );

        Options opt;
        std::vector<std::string> args;
        for ( int i = 1; i < argc; ++i )
        {
            const std::string a = argv[i];
            if ( a == "--t81" ) opt.parity = false;
            else if ( a == "--quiet" ) kpeg::Logger::get().setQuiet( true );
            else if ( a == "--device" && i + 1 < argc ) opt.device = std::atoi( argv[++i] );
            else if ( a == "--devices" && i + 1 < argc ) opt.devices = parseDevices( argv[++i] );
            else if ( a == "--quality" && i + 1 < argc ) opt.quality = std::atoi( argv[++i] );
            else if ( a == "--restart" && i + 1 < argc ) { opt.restart = std::atoi( argv[++i] ); opt.restart_given = true; }
            else if ( a == "--transform" && i + 1 < argc ) opt.transform = argv[++i];
            else if ( a == "--optimize" ) opt.optimize = true;
            else if ( a == "--scale" && i + 1 < argc ) opt.scale = argv[++i];
            else if ( a == "--crop" )
            {
                if ( i + 1 >= argc || !parseCrop( argv[i + 1], opt.crop ) )
                {
                    std::cout << "Malformed --crop '" << ( i + 1 < argc ? argv[i + 1] : "" ) << "': expected WxH+X+Y, e.g. 224x224+16+8" << std::endl;
                    printHelp();
                    return EXIT_FAILURE;
                }
                opt.crop_given = true;
                ++i;
            }
            else args.push_back( a );
        }

        LOG(kpeg::Logger::Level::INFO) << "KPEG - Simple JPEG Encoder & Decoder";

        if ( args.empty() )
        {
            LOG(kpeg::Logger::Level::ERROR) << "No arguments provided.";
            return EXIT_FAILURE;
        }
        if ( args.size() == 1 && args[0] == "-h" )
        {
            printHelp();
            return EXIT_SUCCESS;
        }
        if ( args.size() == 1 )
        {
            decodeJPEG( args[0], opt );
            return EXIT_SUCCESS;
        }
        if ( args.size() == 2 && startsWithSOI( args[0] ) )
        {
            transcodeJPEG( args[0], args[1], opt );
            return EXIT_SUCCESS;
        }
        if ( args.size() == 2 )
        {
            encodeJPEG( args[0], args[1], opt );
            return EXIT_SUCCESS;
        }
        return EXIT_FAILURE;
    }
    catch ( std::exception& e )
    {
        std::cout << "Exceptions Occurred:-" << std::endl;
        std::cout << "What: " << e.what() << std::endl;
    }
    return EXIT_SUCCESS;
}
