// host/ggp_data.hpp — input side of the gfp_gaussian command line: csv_config, the MOMA csv reader, segment
// slicing, genealogy and the hand-over to the C ABI (ggp_forest_desc).
//
// Replaces, from the reference (src/): CSVconfig.h:13-98, moma_input.h:327-352 (cell ids), :401-527 (read_data),
// :538-578 (segment indices), :580-620 (get_segment), :125-151 (build_cell_genealogy), :663-735 (init_cells).
// The reference keeps an AoS std::vector<MOMAdata> of heap Eigen vectors grown one element at a time (O(T^2) per
// cell) and resolves parents by an O(N^2) string scan; here the table is SoA from the start (the layout the C ABI
// takes) and parents are resolved through a hash map, with the same outcome: a cell's parent is the cell whose id
// equals its parent id, daughter1/daughter2 are the first/second child in file order.
#pragma once
#include <algorithm>
#include <cstdint>
#include <unordered_map>

#include "../include/ggp_b200.h"
#include "ggp_util.hpp"

namespace ggp {

struct CsvConfig {
    std::string time_col = "time", length_col = "length", fp_col = "gfp", delm = ",", segment_col, filter_col;
    double rescale_time = 1., fp_auto = 0;
    bool length_islog = false;
    std::vector<std::string> cell_tags{"cell_id"}, parent_tags{"parent_id"};

    explicit CsvConfig(const std::string& filename, std::ostream* log = nullptr) {
        std::ifstream fin(filename);
        std::string line;
        while (std::getline(fin, line)) {
            if (line.empty() || line[0] == '#') continue;
            auto parts = split(line, "=");
            if (parts.size() < 2) continue;
            const std::string key = trim(parts[0]), val = trim(parts[1]);
            auto number = [&](const char* what) {
                try { return std::stod(val); }
                catch (std::exception& e) {
                    if (log) *log << "(CSVconfig) ERROR: " << what << " in 'csv_file' cannnot be processed (" << e.what() << ")" << std::endl;
                    throw;
                }
            };
            auto list = [&]() {
                std::vector<std::string> v;
                for (const auto& s : split(val, ",")) v.push_back(trim(s));
                return v;
            };
            if (key == "time_col") time_col = val;
            else if (key == "rescale_time") rescale_time = number("rescale_time");
            else if (key == "length_col") length_col = val;
            else if (key == "length_islog") length_islog = to_bool(val);
            else if (key == "fp_col") fp_col = val;
            else if (key == "fp_auto") fp_auto = number("fp_auto");
            else if (key == "delm") delm = val;
            else if (key == "cell_tags") cell_tags = list();
            else if (key == "parent_tags") parent_tags = list();
            else if (key == "segment_col") segment_col = val;
            else if (key == "filter_col") filter_col = val;
        }
    }
};

inline std::ostream& operator<<(std::ostream& os, const CsvConfig& c) {
    const int w = 15;
    os << "Configuration used for reading the input file\n_____________________________________________\n"
       << pad("time_col:", w) << c.time_col << "\n" << pad("rescale_time:", w) << c.rescale_time << "\n"
       << pad("length_col:", w) << c.length_col << "\n" << pad("length_islog:", w) << c.length_islog << "\n"
       << pad("fp_col:", w) << c.fp_col << "\n" << pad("fp_auto:", w) << c.fp_auto << "\n" << pad("delm:", w) << c.delm << "\n";
    if (!c.segment_col.empty()) os << pad("segment_col:", w) << c.segment_col << "\n";
    if (!c.filter_col.empty()) os << pad("filter_col:", w) << c.filter_col << "\n";
    os << pad("cell_tags:", w);
    for (const auto& t : c.cell_tags) os << t << ' ';
    os << "\n" << pad("parent_tags:", w);
    for (const auto& t : c.parent_tags) os << t << ' ';
    return os << "\n";
}

// the data set: cells in file order, their points concatenated
struct LineageTable {
    std::vector<std::string> cell_id, parent_id;
    std::vector<int64_t> offset{0};            // [n_cells + 1]
    std::vector<double> time, log_length, fp;  // [n_ctp]
    std::vector<int32_t> segment;              // [n_ctp]
    std::vector<int32_t> parent, daughter1, daughter2;   // [n_cells], set by build_genealogy
    std::string noise_model, division_model;
    double fp_auto = 0;

    int64_t n_cells() const { return (int64_t)cell_id.size(); }
    int64_t n_ctp() const { return (int64_t)time.size(); }
    int64_t n_points(int64_t c) const { return offset[c + 1] - offset[c]; }
};

// "7.0" -> "7" for purely numeric tags (moma_input.h:327-338)
inline std::string remove_last_decimal(const std::string& s) {
    for (char ch : s) if (!isdigit((unsigned char)ch) && ch != '.') return s;
    const auto parts = split(s, ".");
    for (char ch : parts.back()) if (ch != '0') return s;
    return std::to_string(std::stoi(s));
}

inline LineageTable read_data(const std::string& filename, const CsvConfig& cfg, const std::string& noise_model,
                              const std::string& division_model, std::ostream& log) {
    std::ifstream file(filename);
    LineageTable T;
    T.noise_model = noise_model; T.division_model = division_model; T.fp_auto = cfg.fp_auto;
    std::string line;
    std::getline(file, line);
    std::unordered_map<std::string, int> col;
    {
        const auto head = split(line, cfg.delm);
        for (size_t i = 0; i < head.size(); ++i) col.emplace(trim_all(head[i]), (int)i);
    }
    auto need = [&](const std::string& name, const char* what) {
        if (!col.count(name)) {
            log << "(read_data) ERROR: (" << what << ") is not an column in input file: " << name << "\n";
            throw std::invalid_argument("Invalid argument");
        }
        return col[name];
    };
    const int c_time = need(cfg.time_col, "time_col"), c_len = need(cfg.length_col, "length_col"), c_fp = need(cfg.fp_col, "fp_col");
    const int c_seg = cfg.segment_col.empty() ? -1 : need(cfg.segment_col, "segment_col");
    const int c_filter = cfg.filter_col.empty() ? -1 : need(cfg.filter_col, "filter_col");
    std::vector<int> c_cell, c_parent;
    for (const auto& t : cfg.cell_tags) c_cell.push_back(need(t, "at least one of (cell_tags)"));
    for (const auto& t : cfg.parent_tags) c_parent.push_back(need(t, "at least one of (parent_tags)"));
    auto compose = [](const std::vector<std::string>& parts, const std::vector<int>& cols) {
        std::string id;
        for (size_t i = 0; i < cols.size(); ++i) {
            if (i) id += ".";
            id += remove_last_decimal(parts.at(cols[i]));
        }
        return id;
    };
    std::string last_cell, curr_cell;
    long line_count = 1;
    std::vector<std::string> parts;
    while (std::getline(file, line)) {
        ++line_count;
        try {
            parts = split(line, cfg.delm);
            if (c_filter >= 0 && !to_bool(parts.at(c_filter))) continue;
            curr_cell = compose(parts, c_cell);
            if (curr_cell != last_cell) {
                if (!T.cell_id.empty()) T.offset.push_back((int64_t)T.time.size());
                T.cell_id.push_back(curr_cell);
                T.parent_id.push_back(compose(parts, c_parent));
            }
            const double t = to_double_no_nan(parts.at(c_time)) / cfg.rescale_time;
            const double len = to_double_no_nan(parts.at(c_len));
            const double fp = to_double_no_nan(parts.at(c_fp));
            const int seg = c_seg < 0 ? 0 : std::stoi(parts.at(c_seg));
            T.time.push_back(t);
            T.log_length.push_back(cfg.length_islog ? len : std::log(len));
            T.fp.push_back(fp);
            T.segment.push_back(seg);
            last_cell = curr_cell;
        } catch (std::exception& e) {
            log << "(read_data) ERROR: Line no." << line_count << " [" << curr_cell << "] cannnot be processed (" << e.what() << ")" << std::endl;
            throw;
        }
    }
    if (!T.cell_id.empty()) T.offset.push_back((int64_t)T.time.size());
    log << T.n_cells() << " cells and " << line_count << " data points found in file " << filename << std::endl;
    return T;
}

// ---- binary forest file (SURVEY.md 8f row 1): the table as it is handed to the C ABI, for data sets that are too large to be
// worth parsing as text (a 12.6 M-row csv is 600 MB of digits) and for synthetic forests.  Little endian:
//   char magic[8] = "GGPFORE1"; int64 n_cells, n_ctp; int64 cell_offset[n_cells + 1]; double time[n_ctp], log_length[n_ctp],
//   fp[n_ctp]; int32 segment[n_ctp]; then per cell: uint32 length + bytes of its cell id, uint32 length + bytes of its parent id.
// Times are final (no rescale_time), lengths are logarithms, there is no filter column; fp_auto still comes from the csv_config.
// Written by gfp_gaussian_process_b200/io.py::write_forest_binary.
inline bool is_binary_forest(const std::string& filename) {
    std::ifstream f(filename, std::ios::binary);
    char magic[8] = {};
    f.read(magic, 8);
    return f.gcount() == 8 && std::string(magic, 8) == "GGPFORE1";
}

inline LineageTable read_binary_forest(const std::string& filename, const CsvConfig& cfg, const std::string& noise_model,
                                       const std::string& division_model, std::ostream& log) {
    std::ifstream f(filename, std::ios::binary);
    LineageTable T;
    T.noise_model = noise_model; T.division_model = division_model; T.fp_auto = cfg.fp_auto;
    auto fail = [&](const char* what) {
        log << "(read_binary_forest) ERROR: " << what << " in " << filename << "\n";
        throw std::invalid_argument("Invalid argument");
    };
    char magic[8];
    int64_t n_cells = 0, n_ctp = 0;
    f.read(magic, 8);
    f.read(reinterpret_cast<char*>(&n_cells), 8);
    f.read(reinterpret_cast<char*>(&n_ctp), 8);
    if (!f || std::string(magic, 8) != "GGPFORE1" || n_cells <= 0 || n_ctp < n_cells) fail("bad header");
    auto read_array = [&](auto& v, int64_t n) {
        v.resize((size_t)n);
        f.read(reinterpret_cast<char*>(v.data()), (std::streamsize)(n * (int64_t)sizeof(v[0])));
        if (!f) fail("file ends inside an array");
    };
    read_array(T.offset, n_cells + 1);
    read_array(T.time, n_ctp);
    read_array(T.log_length, n_ctp);
    read_array(T.fp, n_ctp);
    read_array(T.segment, n_ctp);
    if (T.offset.front() != 0 || T.offset.back() != n_ctp) fail("cell offsets do not cover the time points");
    for (int64_t c = 0; c < n_cells; ++c) if (T.offset[c + 1] <= T.offset[c]) fail("a cell without a time point");
    auto read_string = [&]() {
        uint32_t len = 0;
        f.read(reinterpret_cast<char*>(&len), 4);
        if (!f || len > (1u << 20)) fail("bad id string");
        std::string s(len, '\0');
        f.read(&s[0], len);
        if (!f) fail("file ends inside an id");
        return s;
    };
    T.cell_id.reserve((size_t)n_cells); T.parent_id.reserve((size_t)n_cells);
    for (int64_t c = 0; c < n_cells; ++c) {
        T.cell_id.push_back(read_string());
        T.parent_id.push_back(read_string());
    }
    log << T.n_cells() << " cells and " << n_ctp << " data points found in binary file " << filename << std::endl;
    return T;
}

// the table as a binary forest file (the layout above, ids included): what io.write_forest_binary writes
inline void write_binary_forest(const std::string& filename, const LineageTable& T) {
    std::ofstream f(filename, std::ios::binary);
    const int64_t n_cells = T.n_cells(), n_ctp = T.n_ctp();
    f.write("GGPFORE1", 8);
    f.write(reinterpret_cast<const char*>(&n_cells), 8);
    f.write(reinterpret_cast<const char*>(&n_ctp), 8);
    auto write_array = [&](const auto& v) { f.write(reinterpret_cast<const char*>(v.data()), (std::streamsize)(v.size() * sizeof(v[0]))); };
    write_array(T.offset);
    write_array(T.time);
    write_array(T.log_length);
    write_array(T.fp);
    write_array(T.segment);
    for (int64_t c = 0; c < n_cells; ++c)
        for (const std::string* s : {&T.cell_id[c], &T.parent_id[c]}) {
            const uint32_t len = (uint32_t)s->size();
            f.write(reinterpret_cast<const char*>(&len), 4);
            f.write(s->data(), len);
        }
    if (!f) throw std::runtime_error("cannot write " + filename);
}

// segment indices in order of first occurrence; must be 0..n-1 (moma_input.h:538-570)
inline std::vector<int> segment_indices(const LineageTable& T, std::ostream& log) {
    std::vector<int> segs;
    for (int s : T.segment) if (std::find(segs.begin(), segs.end(), s) == segs.end()) segs.push_back(s);
    auto fail = [&](const char* what) {
        log << "(get_segment_indices) ERROR: The segment indices " << what << ":";
        for (int s : segs) log << " " << s;
        log << "\n";
        throw std::invalid_argument("Invalid argument");
    };
    if (segs.empty() || *std::min_element(segs.begin(), segs.end()) != 0) fail("do not start at 0");
    if ((int)segs.size() - 1 != *std::max_element(segs.begin(), segs.end())) fail("are not consecutive");
    return segs;
}

// the points of one segment; cells without a point in it vanish, so their daughters become roots (moma_input.h:580-620)
inline LineageTable get_segment(const LineageTable& T, int segment) {
    LineageTable S;
    S.noise_model = T.noise_model; S.division_model = T.division_model; S.fp_auto = T.fp_auto;
    for (int64_t c = 0; c < T.n_cells(); ++c) {
        const size_t before = S.time.size();
        for (int64_t k = T.offset[c]; k < T.offset[c + 1]; ++k)
            if (T.segment[k] == segment) {
                S.time.push_back(T.time[k]); S.log_length.push_back(T.log_length[k]); S.fp.push_back(T.fp[k]);
                S.segment.push_back(T.segment[k]);
            }
        if (S.time.size() > before) {
            S.cell_id.push_back(T.cell_id[c]);
            S.parent_id.push_back(T.parent_id[c]);
            S.offset.push_back((int64_t)S.time.size());
        }
    }
    return S;
}

// parent / daughter1 / daughter2 of every cell (moma_input.h:125-151) through a hash map
inline void build_genealogy(LineageTable& T, std::ostream& log) {
    const int64_t N = T.n_cells();
    std::unordered_map<std::string, int32_t> index;
    index.reserve((size_t)N * 2);
    for (int64_t c = 0; c < N; ++c)
        if (!index.emplace(T.cell_id[c], (int32_t)c).second) {
            log << "(build_cell_genealogy) ERROR: cell id appears in two separate blocks of rows: " << T.cell_id[c] << "\n";
            throw std::invalid_argument("Invalid argument");
        }
    T.parent.assign(N, -1); T.daughter1.assign(N, -1); T.daughter2.assign(N, -1);
    for (int64_t k = 0; k < N; ++k) {
        const auto it = index.find(T.parent_id[k]);
        if (it == index.end()) continue;
        const int32_t j = it->second;
        T.parent[k] = j;
        if (T.daughter1[j] < 0) T.daughter1[j] = (int32_t)k;
        else if (T.daughter2[j] < 0) T.daughter2[j] = (int32_t)k;
        else {
            log << "(build_cell_genealogy) ERROR: Both daughter pointers are set, cell_id: " << T.cell_id[j] << "\n"
                << "-> daughter1 " << T.cell_id[T.daughter1[j]] << "\n-> daughter2 " << T.cell_id[T.daughter2[j]] << "\n";
            throw std::invalid_argument("Invalid argument");
        }
    }
}

// descriptor of the C ABI over the table's arrays (the table must outlive the call that takes the descriptor);
// compute_init = 1: the init_cells statistics are those of this table, as init_cells(cells) computes them
inline ggp_forest_desc make_desc(const LineageTable& T, int device) {
    ggp_forest_desc d{};
    d.n_cells = T.n_cells(); d.n_ctp = T.n_ctp();
    d.cell_offset = T.offset.data(); d.parent = T.parent.data(); d.daughter1 = T.daughter1.data(); d.daughter2 = T.daughter2.data();
    d.time = T.time.data(); d.log_length = T.log_length.data(); d.fp = T.fp.data(); d.segment = T.segment.data();
    d.noise_model = T.noise_model == "scaled" ? GGP_NOISE_SCALED : GGP_NOISE_CONST;
    d.division_model = T.division_model == "binomial" ? GGP_DIVISION_BINOMIAL : GGP_DIVISION_GAUSS;
    d.fp_auto = T.fp_auto;
    d.compute_init = 1;
    d.device = device;
    return d;
}

}  // namespace ggp
