// pose.cpp — host driver of the B200-native reconstruction path.
//
// Keeps the reference's command line (parseCmdArgs, pose_functions.cpp:70-307: same spellings, defaults and
// messages), its dataset layout (data_files/{cam13calib.yml,pose.txt,images.txt}, images/N.png, disparities/N.png,
// segmentlabels/N.png), its cycle structure (pose.cpp:152-458) and its outputs (<folder>/<date>/cloud.ply,
// cloud_uavpos.ply, log.txt), and runs the hot path through the C ABI (include/o3r.h) instead of OpenCV/PCL.
// Feature matching, ICP and visualisation are host-side code of the reference and are not part of this
// driver: frames use the GPS/IMU matrix (the reference's --only_MAVLink path, pose.cpp:236-248) times an
// optional per-frame pose-correction matrix read from --pose_corrections (what T_SVD / tf_icp would provide).
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <map>
#include <sstream>
#include <string>
#include <deque>
#include <vector>

#include "o3r.h"
#include "mapfile.hpp"
#include "ply.hpp"
#include "png.hpp"
#include "tmat.hpp"

using namespace std;
using host::Image;
using host::Mat4;

typedef vector<double> record_t;
typedef vector<record_t> data_t;

struct RawImageData {   // pose.h:54-70
    int img_num = 0;
    Image rgb_image, disparity_image, segment_label;
    double time = 0, tx = 0, ty = 0, tz = 0, qx = 0, qy = 0, qz = 0, qw = 1;
};

struct Pose {
    // defaults: pose.h:92-188
    double minDisparity = 64;
    int boundingBox = 20, rows = 0, cols = 0, cols_start_aft_cutout = 0;
    int jump_pixels = 10, seq_len = -1, blur_kernel = 1, range_width = 30, cutout_ratio = 8;
    double dist_nearby = 2, voxel_size = 0.1;
    unsigned min_points_per_voxel = 1;
    bool downsample = false, only_MAVLink = false, dont_downsample = false, dont_icp = false, log_stuff = true,
         preview = false, use_segment_labels = false, run3d_reconstruction = true, sor = true;
    string read_PLY_filename0, calib_file = "cam13calib.yml";
    string dataFilesPrefix = "data_files/", pose_file = "pose.txt", images_times_file = "images.txt",
           imageNumbersFile = "images/image_numbers.txt";
    string imagePrefix = "images/", disparityPrefix = "disparities/", segmentlblPrefix = "segmentlabels/";
    string folder = "output/", pose_corrections_file;
    bool save_map = false;      // --save_map: <run dir>/map.o3rmap after the last cycle
    bool register_map = false;  // --register_map: from the second cycle on, correct the drift against the map
    bool save_mesh = false;     // --save_mesh: <run dir>/mesh.ply after the last cycle
    double mesh_max_step = HUGE_VAL;   // --mesh_max_step M: drop mesh triangles whose |dz| exceeds M (default: keep all)
    string resume_map_file;     // --resume_map FILE: loaded before the first cycle
    int blur_mode = O3R_BLUR_BILATERAL, device = 0;   // the reference's live filter (pose_functions.cpp:1044)
    double Q[16] = {0};
    vector<RawImageData> rawImageDataVec;
    data_t pose_data, images_times_data;
    vector<double> images_times_seq, pose_times_seq;
    map<int, Mat4> corrections;
    ofstream log_file;
    const int tx_ind = 3, ty_ind = 4, tz_ind = 5, qx_ind = 6, qy_ind = 7, qz_ind = 8, qw_ind = 9;   // pose.h:140

    void printUsage();
    int parseCmdArgs(int argc, char** argv);
    void readCalibFile();
    void readPoseFile();
    void readCorrections();
    int binarySearchImageTime(int l, int r, int imageNumber);
    int binarySearchUsingTime(const vector<double>& seq, int l, int r, double time);
    void populateData();
    int run();
    int runDownsampleTool();
};

void Pose::printUsage() {
    cout << "pose [first_img_num last_img_num] [flags]\n"
            "  reference flags (pose_functions.cpp:70-307): --seq_len N --voxel_size V --jump_pixels J --range_width N\n"
            "      --dist_nearby D --min_points_per_voxel N --blur_kernel K --dont_downsample --use_segment_labels\n"
            "      --only_MAVLink --dont_icp --preview --log 0/1 --downsample <file.ply>\n"
            "  path overrides (the reference hard-codes these, pose.h:129-137): --data_root DIR --image_prefix P\n"
            "      --disparity_prefix P --segmentlbl_prefix P --output DIR --calib FILE\n"
            "  extensions: --blur_mode bilateral|median|box (default bilateral = the reference) --pose_corrections FILE --device N\n"
            "              --no_sor (skip the StatisticalOutlierRemoval the reference applies per frame when jump_pixels > 0)\n"
            "              --save_map (write the resident map to <run dir>/map.o3rmap after the last cycle)\n"
            "              --register_map (from the second cycle on, register the cycle's first, middle and last frame clouds\n"
            "                against the map, gate max(3 voxel_size, 1 m), and premultiply the running correction into every\n"
            "                later frame's matrix)\n"
            "              --resume_map FILE (continue the map of a map.o3rmap saved with the same --voxel_size and --dont_downsample)\n"
            "              --save_mesh (write the map's height field as a triangle mesh to <run dir>/mesh.ply after the last cycle)\n"
            "              --mesh_max_step M (with --save_mesh: drop triangles whose largest |dz| exceeds M metres; default none)\n"
            "  not in this driver (host-side tools of the reference): --visualize --align_point_cloud --smooth_surface\n"
            "      --mesh_surface --segment_cloud --segment_cloud_only --displayUAVPositions\n";
}

int Pose::parseCmdArgs(int argc, char** argv) {
    if (argc == 1) { printUsage(); return -1; }
    int n_imgs = 0, first_img_num = -1, last_img_num = -1;
    string data_root;
    for (int i = 1; i < argc; ++i) {
        const string a = argv[i];
        auto need = [&](const char* what) -> const char* {
            if (i + 1 >= argc) throw "Exception: missing value for a flag!";
            (void)what;
            return argv[++i];
        };
        if (a == "--help" || a == "/?") { printUsage(); return -1; }
        else if (a == "--visualize" || a == "--smooth_surface" || a == "--mesh_surface" || a == "--displayUAVPositions" ||
                 a == "--segment_cloud_only" || a == "--align_point_cloud" || a == "--segment_cloud" ||
                 a == "--test_bad_data_rejection" || a == "--search_radius") {
            cout << a << ": host-side tool of the reference (PCL visualisation / surface / segmentation), not part of the "
                         "B200 hot-path driver." << endl;
            return -2;
        }
        else if (a == "--downsample") { downsample = true; run3d_reconstruction = false; read_PLY_filename0 = need("file"); cout << "Downsample " << read_PLY_filename0 << endl; }
        else if (a == "--voxel_size") { voxel_size = atof(need("v")); cout << "voxel_size " << voxel_size << endl; }
        else if (a == "--min_points_per_voxel") { min_points_per_voxel = atoi(need("n")); cout << "min_points_per_voxel " << min_points_per_voxel << endl; }
        else if (a == "--dist_nearby") { dist_nearby = atof(need("d")); cout << "dist_nearby " << dist_nearby << endl; }
        else if (a == "--blur_kernel") { blur_kernel = atoi(need("k")); cout << "blur_kernel " << blur_kernel << endl; }
        else if (a == "--seq_len") {
            seq_len = atoi(need("n")); cout << "seq_len " << seq_len << endl;
            if (seq_len == 0 || seq_len < -1) throw "Exception: invalid seq_len value!";
        }
        else if (a == "--jump_pixels") { jump_pixels = atoi(need("j")); cout << "jump_pixels " << jump_pixels << endl; }
        else if (a == "--range_width") { range_width = atoi(need("n")); cout << "range_width " << range_width << endl; }
        else if (a == "--log") { log_stuff = atoi(need("0/1")) != 0; cout << "log " << log_stuff << endl; }
        else if (a == "--preview") preview = true;
        else if (a == "--register_map") register_map = true;
        else if (a == "--use_segment_labels") { cout << "use_segment_labels" << endl; use_segment_labels = true; }
        else if (a == "--only_MAVLink") { only_MAVLink = true; cout << "only_MAVLink " << endl; }
        else if (a == "--dont_downsample") { dont_downsample = true; cout << "dont_downsample " << endl; }
        else if (a == "--dont_icp") { dont_icp = true; cout << "dont_icp " << endl; }
        else if (a == "--data_root") data_root = need("dir");
        else if (a == "--image_prefix") imagePrefix = need("p");
        else if (a == "--disparity_prefix") disparityPrefix = need("p");
        else if (a == "--segmentlbl_prefix") segmentlblPrefix = need("p");
        else if (a == "--output") folder = need("dir");
        else if (a == "--calib") calib_file = need("file");
        else if (a == "--pose_corrections") pose_corrections_file = need("file");
        else if (a == "--device") device = atoi(need("n"));
        else if (a == "--no_sor") sor = false;
        else if (a == "--save_map") save_map = true;
        else if (a == "--save_mesh") save_mesh = true;
        else if (a == "--mesh_max_step") {
            mesh_max_step = atof(need("m"));
            if (!(mesh_max_step >= 0)) throw "Exception: --mesh_max_step must be >= 0!";
        }
        else if (a == "--resume_map") resume_map_file = need("file");
        else if (a == "--blur_mode") { const string m = need("mode"); blur_mode = (m == "box") ? O3R_BLUR_BOX : (m == "median") ? O3R_BLUR_MEDIAN : O3R_BLUR_BILATERAL; }
        else {
            cout << atoi(argv[i]) << endl;
            if (first_img_num == -1) first_img_num = atoi(argv[i]); else last_img_num = atoi(argv[i]);
            ++n_imgs;
        }
    }
    if (!data_root.empty()) {
        if (data_root.back() != '/') data_root += '/';
        for (string* s : {&dataFilesPrefix, &imagePrefix, &disparityPrefix, &segmentlblPrefix, &imageNumbersFile})
            if ((*s)[0] != '/') *s = data_root + *s;
    }
    if (!folder.empty() && folder.back() != '/') folder += '/';
    if (run3d_reconstruction && n_imgs == 0) {   // pose_functions.cpp:258-282
        ifstream images_file(imageNumbersFile);
        if (!images_file.is_open()) throw "Exception: Unable to open imageNumbersFile!";
        string line;
        while (getline(images_file, line)) {
            stringstream fs(line);
            int img_num = 0;
            fs >> img_num;
            RawImageData obj; obj.img_num = img_num;
            rawImageDataVec.push_back(obj);
            ++n_imgs;
        }
        cout << "\nRead " << n_imgs << " image numbers from " << imageNumbersFile << endl;
    } else if (run3d_reconstruction) {           // :283-304
        if (last_img_num < first_img_num) last_img_num = first_img_num;
        n_imgs = last_img_num - first_img_num + 1;
        rawImageDataVec = vector<RawImageData>(n_imgs);
        for (int i = 0; i < n_imgs; i++) rawImageDataVec[i].img_num = first_img_num + i;
    }
    return 0;
}

static istream& read_record(istream& ins, record_t& record) {   // pose_functions.cpp:351-379
    record.clear();
    string line;
    getline(ins, line);
    stringstream ss(line);
    string field;
    while (getline(ss, field, ',')) {
        stringstream fs(field);
        double f = 0.0;
        fs >> f;
        record.push_back(f);
    }
    return ins;
}
static void read_data(const string& path, data_t& data, const char* err) {   // :385-397, :478-498
    ifstream f(path);
    if (!f.is_open()) throw err;
    data.clear();
    record_t r;
    while (read_record(f, r)) if (!r.empty()) data.push_back(r);
}

void Pose::readCalibFile() {   // :467-476 — cv::FileStorage["Q"]: rows 4, cols 4, dt d, data [...]
    ifstream f(dataFilesPrefix + calib_file);
    if (!f.is_open()) throw "Exception: could not read Q matrix";
    stringstream ss; ss << f.rdbuf();
    const string s = ss.str();
    size_t at = s.find("\nQ:");
    if (at == string::npos) throw "Exception: could not read Q matrix";
    at = s.find("data:", at);
    const size_t lb = s.find('[', at), rb = s.find(']', lb);
    if (at == string::npos || lb == string::npos || rb == string::npos) throw "Exception: could not read Q matrix";
    string body = s.substr(lb + 1, rb - lb - 1);
    replace(body.begin(), body.end(), ',', ' ');
    stringstream bs(body);
    int n = 0;
    while (n < 16 && (bs >> Q[n])) ++n;
    if (n != 16) throw "Exception: could not read Q matrix";
    cout << "read calib file." << endl;
}

void Pose::readPoseFile() {
    read_data(dataFilesPrefix + pose_file, pose_data, "Exception: Could not open pose_data file!");
    for (auto& r : pose_data) pose_times_seq.push_back(r[2]);
    read_data(dataFilesPrefix + images_times_file, images_times_data, "Exception: Could not open images_times_data file!");
    for (auto& r : images_times_data) images_times_seq.push_back(r[2]);
    cout << "Your images_times file contains " << images_times_data.size() << " records.\n";
    cout << "Your pose_data file contains " << pose_data.size() << " records.\n";
}

void Pose::readCorrections() {   // img_num, 16 row-major floats per line: the matrix T_SVD (* tf_icp) of that frame
    if (pose_corrections_file.empty()) return;
    data_t d;
    read_data(pose_corrections_file, d, "Exception: Could not open pose_corrections file!");
    for (auto& r : d) {
        if (r.size() < 17) continue;
        Mat4 m;
        for (int i = 0; i < 16; ++i) m.m[i] = (float)r[1 + i];
        corrections[(int)r[0]] = m;
    }
    cout << "read " << corrections.size() << " pose corrections." << endl;
}

int Pose::binarySearchImageTime(int l, int r, int imageNumber) {   // :402-424
    while (r >= l) {
        const int mid = l + (r - l) / 2;
        if ((int)images_times_data[mid][0] == imageNumber) return mid;
        if ((int)images_times_data[mid][0] > imageNumber) r = mid - 1; else l = mid + 1;
    }
    throw "Exception: binarySearchImageTime: unsuccessful search!";
}

int Pose::binarySearchUsingTime(const vector<double>& seq, int l, int r, double time) {   // :429-465
    while (r >= l) {
        const int mid = l + (r - l) / 2;
        if (mid > 0 && mid < (int)seq.size() - 1) { if (seq[mid - 1] < time && seq[mid + 1] > time) return mid; }
        else if (mid == 0) return 0;
        else return (int)seq.size() - 1;
        if (seq[mid] > time) r = mid - 1; else l = mid + 1;
    }
    throw "Exception: binarySearchUsingTime: unsuccessful search!";
}

void Pose::populateData() {   // :624-744 (the 7-thread loaders become a plain loop; I/O is off the hot path)
    readCalibFile();
    readPoseFile();
    readCorrections();
    if (log_stuff) log_file.open((folder + "log.txt").c_str(), ios::out);
    for (auto& r : rawImageDataVec) {
        r.rgb_image = host::read_png(imagePrefix + to_string(r.img_num) + ".png", false);
        r.disparity_image = host::read_png(disparityPrefix + to_string(r.img_num) + ".png", true);
        if (use_segment_labels) r.segment_label = host::read_png(segmentlblPrefix + to_string(r.img_num) + ".png", true);
        if (r.rgb_image.empty()) cout << " cannot_read_i" << r.img_num << " " << flush; else cout << " i" << r.img_num << " " << flush;
        if (r.disparity_image.empty()) cout << " cannot_read_d" << r.img_num << " " << flush; else cout << " d" << r.img_num << " " << flush;
        // :568-582 time -> pose
        const int ti = binarySearchImageTime(0, (int)images_times_seq.size() - 1, r.img_num);
        const int pi = binarySearchUsingTime(pose_times_seq, 0, (int)pose_times_seq.size() - 1, images_times_seq[ti]);
        r.time = images_times_seq[ti];
        const record_t& p = pose_data[pi];
        r.tx = p[tx_ind]; r.ty = p[ty_ind]; r.tz = p[tz_ind];
        r.qx = p[qx_ind]; r.qy = p[qy_ind]; r.qz = p[qz_ind]; r.qw = p[qw_ind];
        if (rows == 0 && !r.rgb_image.empty()) { rows = r.rgb_image.rows; cols = r.rgb_image.cols; cols_start_aft_cutout = cols / cutout_ratio; }
    }
    cout << endl;
}


static string currentDateTime() {   // pose_functions.cpp:331-345
    time_t now = time(0);
    char buf[80];
    strftime(buf, sizeof(buf), "%Y-%m-%d.%X", localtime(&now));
    return buf;
}
static double now_s() { return chrono::duration<double>(chrono::steady_clock::now().time_since_epoch()).count(); }

static o3r_ctx* make_ctx(Pose& P, int merge_mode, int max_batch) {
    o3r_params p{};
    p.rows = P.rows; p.cols = P.cols; p.cols_start_aft_cutout = P.cols_start_aft_cutout;
    p.bounding_box = P.boundingBox; p.min_disparity = P.minDisparity;
    for (int i = 0; i < 16; ++i) p.Q[i] = P.Q[i];
    p.jump_pixels = P.jump_pixels; p.blur_kernel = P.blur_kernel; p.blur_mode = P.blur_mode;
    p.voxel_size = P.voxel_size; p.min_points_per_voxel = P.min_points_per_voxel;
    p.dont_downsample = P.dont_downsample; p.use_segment_labels = P.use_segment_labels ? 1 : 0;
    p.sor_mean_k = (P.sor && P.jump_pixels > 0) ? 50 : 0; p.sor_stddev_mul = 1.0;   // pose_functions.cpp:1673-1686
    p.disp_divisor = 200.0; p.merge_mode = merge_mode; p.device = P.device; p.max_batch_frames = max(1, max_batch);
    o3r_ctx* ctx = nullptr;
    if (o3r_create(&p, &ctx) != O3R_OK) { cerr << "o3r_create: " << o3r_last_error(nullptr) << endl; return nullptr; }
    return ctx;
}

int Pose::runDownsampleTool() {   // pose.cpp:71-87
    vector<o3r_point> cloud;
    if (!host::read_ply(read_PLY_filename0, cloud)) { cerr << "cannot read " << read_PLY_filename0 << endl; return 1; }
    cout << "Read PLY file!" << endl;
    rows = 64; cols = 64; cols_start_aft_cutout = 8;   // unused by the cloud entry points
    jump_pixels = 1;
    o3r_ctx* ctx = make_ctx(*this, O3R_MERGE_ACCUMULATE, 1);
    if (!ctx) return 1;
    int rc = o3r_cloud_append(ctx, cloud.data(), cloud.size());
    size_t n = 0;
    if (!rc) rc = o3r_cloud_downsample(ctx, nullptr, 0, &n);
    vector<o3r_point> out(n);
    if (!rc) rc = o3r_cloud_downsample(ctx, out.data(), out.size(), &n);
    if (rc) { cerr << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1; }
    const size_t slash = read_PLY_filename0.find_last_of('/');
    const string dir = slash == string::npos ? "" : read_PLY_filename0.substr(0, slash + 1);
    const string base = slash == string::npos ? read_PLY_filename0 : read_PLY_filename0.substr(slash + 1);
    const string writePath = dir + "downsampled_" + base;
    host::save_ply_binary(writePath, out.data(), n);
    cerr << "Saved Point Cloud with " << n << " data points to " << writePath << endl;
    cout << "Cya!" << endl;
    o3r_destroy(ctx);
    return 0;
}

int Pose::run() {
    const string currentDateTimeStr = currentDateTime();
    cout << "currentDateTime=" << currentDateTimeStr << "\n\n";
    mkdir(folder.c_str(), 0777);
    folder = folder + currentDateTimeStr + "/";
    if (mkdir(folder.c_str(), 0777) == 0) cout << "Created save directory " << folder << endl;
    else { cout << "Could not create save directory!" << folder << endl; return 1; }
    if (downsample) return runDownsampleTool();
    if (!only_MAVLink)
        cout << "note: feature matching / ICP run in the reference's host code; this driver uses the GPS/IMU matrix"
                " (--only_MAVLink path) times --pose_corrections when given." << endl;
    populateData();
    if (rows == 0 || cols == 0 || cols_start_aft_cutout == 0) throw "Exception: some important values not set!";
    const double app_start_time = now_s();
    o3r_ctx* ctx = make_ctx(*this, O3R_MERGE_ACCUMULATE, seq_len);
    if (!ctx) return 1;
    // --preview (pose.cpp:638-674 shows a downsampled copy of cloud_big every cycle): the headless equivalent keeps a
    // key-sorted copy of the combined grid, updated each cycle from the cells that cycle changed, and rewrites preview.ply
    const bool do_preview = preview && !dont_downsample;
    if (preview && dont_downsample)
        cout << "--preview needs the combined grid, which --dont_downsample skips: no preview.ply is written" << endl;
    if (do_preview && o3r_cloud_track_changes(ctx, 1) != O3R_OK) {
        cerr << "o3r_cloud_track_changes: " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1;
    }
    if (!resume_map_file.empty()) {   // after the tracking is on: the first preview.ply already shows the resumed map
        const uint32_t kind = dont_downsample ? host::MAP_KIND_POINTS : host::MAP_KIND_CELLS;
        vector<uint8_t> recs;
        uint64_t n_rec = 0;
        string err;
        if (!host::load_map(resume_map_file, kind, voxel_size, recs, &n_rec, &err)) {
            cerr << "--resume_map: " << err << endl; o3r_destroy(ctx); return 1;
        }
        const int rc = kind == host::MAP_KIND_CELLS ? o3r_cloud_import_cells(ctx, (const o3r_cell*)recs.data(), n_rec)
                                                    : o3r_cloud_append(ctx, (const o3r_point*)recs.data(), n_rec);
        if (rc) { cerr << "--resume_map: " << resume_map_file << ": " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1; }
        for (ostream* o : {(ostream*)&cout, (ostream*)&log_file})
            *o << "Resumed map " << resume_map_file << ": " << n_rec << (kind == host::MAP_KIND_CELLS ? " cells" : " points") << endl;
    }
    std::map<uint64_t, o3r_point> preview_map;
    vector<o3r_point> chg_pts;
    vector<uint64_t> chg_keys;
    vector<o3r_point> hexPos_MAVLink, hexPos_FM;
    vector<int> accepted_nums;
    // --register_map: the running drift correction (what the reference's ICP block multiplies into the later frames,
    // pose.cpp:318-319), and the staging of the clouds it registers
    Mat4 drift = host::mat4_identity();
    vector<o3r_point> reg_pts, frame_pts((size_t)rows * cols);
    if (register_map && dont_downsample)
        cout << "--register_map needs the combined grid, which --dont_downsample skips: no registration" << endl;
    if (save_mesh && dont_downsample)
        cout << "--save_mesh needs the combined grid, which --dont_downsample skips: no mesh.ply is written" << endl;
    int current_idx = 0, cycle = 0;
    const int last_idx = (int)rawImageDataVec.size() - 1;
    size_t accepted = 0;
    cout << "\n\nProgram Start!" << endl;
    while (current_idx <= last_idx) {   // pose.cpp:152
        const double t0 = now_s();
        cout << "\nCycle " << cycle << endl;
        log_file << "\nCycle " << cycle << endl;
        vector<o3r_frame> batch;
        std::deque<vector<double>> plane_coefs;   // per accepted frame, stable addresses for the batch
        int images_in_cycle = 0;
        while (images_in_cycle < seq_len && current_idx <= last_idx) {   // :162-255
            RawImageData& r = rawImageDataVec[current_idx];
            if (r.rgb_image.empty()) { cout << r.img_num << " could not read rgb image. \tRejected!" << endl; log_file << r.img_num << " could not read rgb image. \tRejected!" << endl; current_idx++; continue; }
            if (r.disparity_image.empty()) { cout << r.img_num << " could not read disparity image. \tRejected!" << endl; log_file << r.img_num << " could not read disparity image. \tRejected!" << endl; current_idx++; continue; }
            double disp_img_var = 0;   // getVariance (pose_functions.cpp:1007) on the GPU
            if (o3r_disp_variance(ctx, r.disparity_image.data.data(), r.disparity_image.step(), &disp_img_var) != O3R_OK)
                throw "Exception: o3r_disp_variance failed";
            cout << r.img_num << " " << flush;
            log_file << r.img_num << " disp_img_var " << disp_img_var << "\t";
            if (disp_img_var > 5) { cout << " disp_img_var = " << disp_img_var << " > 5.\tRejected!" << endl; log_file << " disp_img_var = " << disp_img_var << " > 5.\tRejected!" << endl; current_idx++; continue; }
            Mat4 t = host::generate_tmat(r.tx, r.ty, r.tz, r.qx, r.qy, r.qz, r.qw);   // :198
            auto c = corrections.find(r.img_num);
            if (c != corrections.end()) t = host::mat4_mul(c->second, t);               // :232
            if (register_map) t = host::mat4_mul(drift, t);                             // :318-319
            o3r_frame f{};
            if (use_segment_labels) {   // createPlaneFittedDisparityImages (pose_functions.cpp:900-985) on the GPU
                if (r.segment_label.empty()) { cout << r.img_num << " could not read segment labels. \tRejected!" << endl; log_file << r.img_num << " could not read segment labels. \tRejected!" << endl; current_idx++; continue; }
                plane_coefs.emplace_back(255 * 3, 0.0);
                int n_planes = 0;
                double pf_var = 0;
                if (o3r_plane_fit(ctx, r.segment_label.data.data(), r.segment_label.step(), r.disparity_image.data.data(),
                                  r.disparity_image.step(), plane_coefs.back().data(), 255, &n_planes, &pf_var) != O3R_OK)
                    throw "Exception: o3r_plane_fit failed";
                log_file << " plane_fitted_disp_img_var " << pf_var << "\t";
                if (pf_var > 3) {   // :975-982
                    cout << "Exception: plane_fitted_disp_img_var " << current_idx << " > 3. Unacceptable disparity image." << endl;
                    throw "Error";
                }
                f.labels = r.segment_label.data.data(); f.labels_step = r.segment_label.step();
                f.plane_coef = plane_coefs.back().data(); f.n_planes = n_planes;
            }
            f.disp = r.disparity_image.data.data(); f.disp_step = r.disparity_image.step();
            f.bgr = r.rgb_image.data.data(); f.bgr_step = r.rgb_image.step();
            memcpy(f.T, t.m, sizeof(f.T));
            batch.push_back(f);
            o3r_point hp{(float)r.tx, (float)r.ty, (float)r.tz, 255u << 16};           // generateUAVpos :1815 (red)
            hexPos_MAVLink.push_back(hp);
            o3r_point hf = hp;
            if (c != corrections.end()) {                                              // transformPoint :1827
                const float* m = c->second.m;
                hf.x = m[0] * hp.x + m[1] * hp.y + m[2] * hp.z + m[3];
                hf.y = m[4] * hp.x + m[5] * hp.y + m[6] * hp.z + m[7];
                hf.z = m[8] * hp.x + m[9] * hp.y + m[10] * hp.z + m[11];
            }
            hf.rgb = 255u << 8;                                                        // green, :244
            hexPos_FM.push_back(hf);
            accepted_nums.push_back(r.img_num);
            cout << "\tAccepted!" << endl;
            current_idx++; images_in_cycle++;
        }
        if (register_map && !dont_downsample && cycle > 0 && !batch.empty()) {
            // the cycle's first, middle and last frames as the library makes their clouds, registered against the map
            const int disp_type = use_segment_labels ? O3R_DISP_F64 : O3R_DISP_U8;
            const size_t nb = batch.size();
            reg_pts.clear();
            vector<size_t> pick{0};
            if (nb / 2 != pick.back()) pick.push_back(nb / 2);
            if (nb - 1 != pick.back()) pick.push_back(nb - 1);
            for (size_t i : pick) {
                size_t m = 0;
                if (o3r_frame_cloud(ctx, &batch[i], disp_type, frame_pts.data(), frame_pts.size(), &m) != O3R_OK) {
                    cerr << "o3r_frame_cloud: " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1;
                }
                reg_pts.insert(reg_pts.end(), frame_pts.begin(), frame_pts.begin() + m);
            }
            const Mat4 I = host::mat4_identity();
            Mat4 T;
            o3r_register_stats st{};
            o3r_register_params rp{20, std::max(3.0 * voxel_size, 1.0), 1e-5, 1e-4, 1e-3};   // a cycle may drift more than 3 voxels
            if (o3r_cloud_register(ctx, reg_pts.data(), reg_pts.size(), I.m, &rp, T.m, &st) != O3R_OK) {
                cerr << "o3r_cloud_register: " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1;
            }
            drift = host::mat4_mul(T, drift);
            for (auto& f : batch) {
                Mat4 ft;
                memcpy(ft.m, f.T, sizeof(ft.m));
                ft = host::mat4_mul(T, ft);
                memcpy(f.T, ft.m, sizeof(f.T));
            }
            char line[256];
            snprintf(line, sizeof(line), "Map registration: %u/%zu, rms %.4f -> %.4f, rank %u, t = (%.4f, %.4f, %.4f)", st.n_inliers,
                     reg_pts.size(), st.rms_initial, st.rms_final, st.rank, T.m[3], T.m[7], T.m[11]);
            for (ostream* o : {(ostream*)&cout, (ostream*)&log_file}) *o << line << endl;
        }
        const double t2 = now_s();
        cout << "\nMatching features and finding transformations time: " << (t2 - t0) << " sec" << endl;
        log_file << "Matching features n transformations time:\t" << (t2 - t0) << " sec" << endl;
        cout << "Adding Point Cloud number/points ";
        log_file << "Adding Point Cloud number/points ";
        vector<uint32_t> counts(batch.size());
        if (!batch.empty()) {
            const int rc = o3r_frames_cloud(ctx, batch.data(), (int)batch.size(), use_segment_labels ? O3R_DISP_F64 : O3R_DISP_U8,
                                            counts.data());
            if (rc != O3R_OK) cout << "Exception caught in cycle " << cycle << ": " << o3r_last_error(ctx) << endl;   // pose.cpp:620-635
            for (size_t i = 0; i < batch.size(); ++i) {
                cout << " " << accepted_nums[accepted + i] << flush;
                log_file << " " << accepted_nums[accepted + i] << "/" << counts[i] << flush;
            }
            accepted += batch.size();
        }
        const double t4 = now_s();
        cout << "\n\nPoint Cloud Creation time: " << (t4 - t2) << " sec" << endl;
        log_file << "\nPoint Cloud Creation time:\t\t\t" << (t4 - t2) << " sec" << endl;
        if (do_preview) {
            size_t m = 0;
            int rc = o3r_cloud_changes(ctx, nullptr, nullptr, nullptr, 0, &m);
            chg_pts.resize(std::max<size_t>(m, 1)); chg_keys.resize(std::max<size_t>(m, 1));
            if (!rc) rc = o3r_cloud_changes(ctx, chg_pts.data(), chg_keys.data(), nullptr, chg_pts.size(), &m);
            if (rc) { cerr << "o3r_cloud_changes: " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1; }
            for (size_t i = 0; i < m; ++i) preview_map[chg_keys[i]] = chg_pts[i];
            vector<o3r_point> view;
            view.reserve(preview_map.size());
            for (const auto& kv : preview_map) view.push_back(kv.second);
            host::save_ply_binary(folder + "preview.ply", view.data(), view.size());
            for (ostream* o : {(ostream*)&cout, (ostream*)&log_file})
                *o << "Preview cells changed/total: " << m << "/" << preview_map.size() << endl;
        }
        cycle++;
        cout << "\nCycle time: " << (now_s() - t0) << " sec" << endl;
        log_file << "Cycle time:\t\t\t\t\t" << (now_s() - t0) << " sec" << endl;
    }
    const double tend = now_s();
    for (ostream* o : {(ostream*)&cout, (ostream*)&log_file})
        *o << "\nFinished Pose Estimation, total time: " << (tend - app_start_time) << " sec at "
           << 1.0 * accepted / (tend - app_start_time) << " fps"
           << "\nraw_images " << rawImageDataVec.size() << "\naccepted_images " << accepted
           << "\njump_pixels " << jump_pixels << "\nseq_len " << seq_len << "\nrange_width " << range_width
           << "\nblur_kernel " << blur_kernel << "\nvoxel_size " << voxel_size
           << "\nmin_points_per_voxel " << min_points_per_voxel << "\ndist_nearby " << dist_nearby << endl;
    if (save_map) {   // the resident state itself (cells with their sums and counts, or cloud_big), before the final downsample
        const uint32_t kind = dont_downsample ? host::MAP_KIND_POINTS : host::MAP_KIND_CELLS;
        size_t m = 0;
        int rc = kind == host::MAP_KIND_CELLS ? o3r_cloud_export_cells(ctx, nullptr, 0, &m) : o3r_cloud_export_points(ctx, nullptr, 0, &m);
        vector<uint8_t> recs(std::max<size_t>(m, 1) * host::map_record_bytes(kind));
        if (!rc) rc = kind == host::MAP_KIND_CELLS ? o3r_cloud_export_cells(ctx, (o3r_cell*)recs.data(), m, &m)
                                                   : o3r_cloud_export_points(ctx, (o3r_point*)recs.data(), m, &m);
        if (rc) { cerr << "--save_map: " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1; }
        const string path = folder + "map.o3rmap";
        if (!host::save_map(path, kind, recs.data(), m, voxel_size)) { cerr << "--save_map: cannot write " << path << endl; o3r_destroy(ctx); return 1; }
        cerr << "Saved map with " << m << (kind == host::MAP_KIND_CELLS ? " cells" : " points") << " to " << path << endl;
    }
    size_t n = 0;
    if (!dont_downsample) cout << "downsample before saving..." << endl;
    int rc = o3r_cloud_downsample(ctx, nullptr, 0, &n);       // pose.cpp:527-536
    vector<o3r_point> cloud_small(n);
    if (!rc) rc = o3r_cloud_downsample(ctx, cloud_small.data(), cloud_small.size(), &n);
    if (rc) { cerr << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1; }
    if (!dont_downsample) cout << "downsampled." << endl;
    cout << "Saving point clouds..." << endl;
    string path = folder + "cloud.ply";
    host::save_ply_binary(path, cloud_small.data(), n);
    cerr << "Saved Point Cloud with " << n << " data points to " << path << endl;
    if (save_mesh && !dont_downsample) {   // the map's height field; its vertices are cloud.ply's points, in the same order
        size_t nv = 0, nt = 0;
        rc = o3r_cloud_mesh(ctx, mesh_max_step, nullptr, nullptr, 0, &nv, nullptr, 0, &nt);
        vector<o3r_point> verts(nv);
        vector<float> normals(nv * 3);
        vector<uint32_t> tris(nt * 3);
        if (!rc) rc = o3r_cloud_mesh(ctx, mesh_max_step, verts.data(), normals.data(), nv, &nv, tris.data(), nt, &nt);
        if (rc) { cerr << "--save_mesh: " << o3r_last_error(ctx) << endl; o3r_destroy(ctx); return 1; }
        path = folder + "mesh.ply";
        if (!host::save_mesh_ply(path, verts.data(), normals.data(), nv, tris.data(), nt)) {
            cerr << "--save_mesh: cannot write " << path << endl; o3r_destroy(ctx); return 1;
        }
        cerr << "Saved mesh with " << nv << " vertices and " << nt << " triangles to " << path << endl;
    }
    hexPos_FM.insert(hexPos_FM.end(), hexPos_MAVLink.begin(), hexPos_MAVLink.end());   // pose.cpp:553
    path = folder + "cloud_uavpos.ply";
    host::save_ply_binary(path, hexPos_FM.data(), hexPos_FM.size());
    cerr << "Saved Point Cloud with " << hexPos_FM.size() << " data points to " << path << endl;
    o3r_destroy(ctx);
    return 0;
}

int main(int argc, char* argv[]) {   // pose.cpp:727-767
    try {
        Pose pose;
        const int rc = pose.parseCmdArgs(argc, argv);
        if (rc != 0) return rc == -1 ? 0 : 2;
        if (pose.run3d_reconstruction && pose.seq_len == -1) throw "Exception: --seq_len must be given (the reference never terminates without it, pose.h:97)";
        return pose.run();
    } catch (const exception& e) {
        cout << "std::exception caught: " << e.what() << endl;
        return 1;
    } catch (const char* msg) {
        cout << msg << endl;
        return 1;
    }
}
